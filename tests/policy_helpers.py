"""Float64 NumPy reference of policy sampling (gcb_env_sample_policy / BatchedChessEnv.sample_policy) and the comparison
rule, shared by tests/test_policy_host.py (host emulation) and tests/test_policy_gpu.py (CUDA library).

L of an env is the oracle's legal list of the env's exported position re-sorted by action code; Philox words come from
oracle.draw_u32 with purpose 3 + (side to move is black).  u * Z and the prefix sums are float64.  The device action must
equal the reference action, except where the reference's u * Z lies within 2^-13 * Z of a prefix-sum boundary AND the two
actions are neighbours in L order (the fp32 sums of the device may round across the boundary): those are counted and must
stay rare.  logp must be within 1e-4 of the float64 log-softmax of the action the device chose.
"""
import numpy as np

from oracle import oracle as orc

RESIGN = 4100
NEAR = 2.0 ** -13


def policy_u(words):
    """u of the random words exactly as the library computes it: (word >> 8) * 2^-24 + 2^-25 in fp32"""
    w = np.asarray(words).astype(np.uint32)
    return (w >> 8).astype(np.float32) * np.float32(2.0 ** -24) + np.float32(2.0 ** -25)


def bf16_bits(x):
    """float32 array -> bf16 bit patterns (uint16), round to nearest even"""
    import torch

    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def bf16_values(bits):
    """bf16 bit patterns -> the float32 values they stand for"""
    return (np.asarray(bits).astype(np.uint32) << 16).view(np.float32)


def legal_codes(boards, info):
    """the legal set of every exported env, sorted by action code: (codes int64 [N, K] padded with -1, counts [N])"""
    out, cnt = orc.movegen_batch(boards, info[:, 0].astype(np.int8), info[:, 1:5].astype(np.uint8), stride=512)
    K = max(1, int(cnt.max()))
    codes = np.where(np.arange(512)[None, :] < cnt[:, None], out.astype(np.int64), 1 << 20)[:, :K]
    codes = np.sort(codes, axis=1)
    codes[codes == 1 << 20] = -1
    return codes, cnt


def philox_words(seed, env_id_offset, info):
    """the default words: Philox, counter (global env id, episode, step in episode, 3 + side to move is black)"""
    return np.array([orc.draw_u32(seed, env_id_offset + e, int(info[e, 10]), int(info[e, 11]), 3 + int(info[e, 0] < 0))
                     for e in range(len(info))], np.uint32)


def reference(x, codes, cnt, temperature, words):
    """x float32 [N, >= 4101] (the values the device reads: bf16 already widened).  -> (action [N], z - m - log Z of every
    entry of L [N, K] (float64), near [N] bool, index of the reference action in L [N], -1 for RESIGN)"""
    N, K = codes.shape
    valid = codes >= 0
    xv = np.where(valid, np.take_along_axis(x, np.maximum(codes, 0), 1).astype(np.float64), -np.inf)
    if temperature == 0:
        idx = np.argmax(xv, 1)  # first maximum = lowest code
        ok = xv[np.arange(N), idx] > -np.inf
        logsm = np.zeros((N, K))
        near = np.zeros(N, bool)
    else:
        z = xv / temperature
        m = z.max(1)
        ok = m > -np.inf
        m = np.where(ok, m, 0.0)
        w = np.where(valid, np.exp(z - m[:, None]), 0.0)
        cum = np.cumsum(w, 1)
        Z = cum[:, -1]
        target = policy_u(words).astype(np.float64) * Z
        above = cum > target[:, None]
        idx = np.where(above.any(1), np.argmax(above, 1), K - 1 - np.argmax((w > 0)[:, ::-1], 1))
        with np.errstate(divide="ignore"):
            logsm = z - m[:, None] - np.log(np.where(ok, Z, 1.0))[:, None]
        near = (np.abs(cum - target[:, None]) < NEAR * Z[:, None]).any(1)
    ok &= cnt > 0
    act = np.where(ok, codes[np.arange(N), idx], RESIGN)
    return act, logsm, near, np.where(ok, idx, -1)


def compare(act, logp, x, codes, cnt, temperature, words, tag=""):
    """the comparison rule of the module docstring; returns the number of boundary exceptions"""
    act, logp = np.asarray(act).astype(np.int64), np.asarray(logp, np.float64)
    N = len(act)
    ref, logsm, near, ridx = reference(x, codes, cnt, temperature, words)
    # every sampled action is legal (or RESIGN where the reference resigns)
    didx = np.argmax(codes == act[:, None], 1)
    legal = (codes[np.arange(N), didx] == act) & (act != RESIGN)
    assert ((ref == RESIGN) == (act == RESIGN)).all(), "%sRESIGN mismatch at %s" % (tag, np.nonzero((ref == RESIGN) != (act == RESIGN))[0][:10])
    assert (legal | (act == RESIGN)).all(), "%sillegal action at %s" % (tag, np.nonzero(~legal & (act != RESIGN))[0][:10])
    diff = act != ref
    exc = diff & near & (np.abs(didx - ridx) == 1)
    bad = diff & ~exc
    assert not bad.any(), "%s%d actions differ from the reference, e.g. env %s: %s vs %s" % (
        tag, bad.sum(), np.nonzero(bad)[0][:5], act[bad][:5], ref[bad][:5])
    if temperature == 0:
        assert (logp == 0).all(), tag
    else:
        exp = np.where(legal, logsm[np.arange(N), didx], 0.0)
        err = np.abs(logp - exp)
        assert (err <= 1e-4).all(), "%slogp off by %g at env %d" % (tag, err.max(), int(np.argmax(err)))
    assert exc.sum() <= max(1, N // 1000), "%s%d boundary exceptions in %d draws" % (tag, exc.sum(), N)
    return int(exc.sum())


def check_env(E, seed, env_id_offset, rng, temperatures=(0.5, 1.0, 2.0), tag="", randn=None):
    """E: an env with export() and sample_policy(logits, T, u32) (numpy in / out; uint16 logits = bf16 bits).  Checks fp32
    and bf16 logits from N(0, 3^2), with caller words and with Philox words, at every temperature and at T = 0.
    randn(N): float32 [N, 4101] standard normals (default: from rng)."""
    boards, info, _ = E.export()
    codes, cnt = legal_codes(boards, info)
    N = len(info)
    pwords = philox_words(seed, env_id_offset, info)
    exceptions = 0
    for dt in ("f32", "bf16"):
        x = (rng.standard_normal((N, 4101)).astype(np.float32) if randn is None else randn(N)) * np.float32(3)
        inp = x if dt == "f32" else bf16_bits(x)
        xv = x if dt == "f32" else bf16_values(inp)
        for T in tuple(temperatures) + (0.0,):
            for src in ("caller", "philox"):
                if T == 0 and src == "philox":
                    continue
                cw = rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32)
                act, logp = E.sample_policy(inp, T, cw if src == "caller" else None)
                exceptions += compare(act, logp, xv, codes, cnt, T, cw if src == "caller" else pwords,
                                      "%s%s T=%g %s: " % (tag, dt, T, src))
    return exceptions
