"""Shared checks of the per-env clone (gcb_env_clone / BatchedChessEnv.clone_from), run against the host emulation
(tests/test_clone_host.py) and the CUDA library (tests/test_clone_gpu.py).

The oracle side of a clone is a deep copy of the oracle's plain C struct (`oracle_clone`): every field of the source env,
its saved_boards history included, except what the destination keeps -- env_id, seed, initial_board, the forced bot move --
and the episode counter, which becomes the destination's own + 1.
"""
import ctypes as C

import numpy as np

from oracle import oracle as orc
from tests import parity_helpers as ph

EPISODE_COL = 10


class _GcoEnv(C.Structure):
    """layout of gco_env (oracle/gc_oracle.h)"""
    _fields_ = [("st", orc._State), ("initial_board", C.c_int8 * 64), ("agent_black", C.c_int), ("opponent", C.c_int),
                ("done", C.c_int), ("move_count", C.c_int), ("moves_max", C.c_int), ("n_legal", C.c_int),
                ("legal", C.c_uint16 * orc.MAX_MOVES), ("wedged_bot", C.c_int), ("hist_n", C.c_int), ("hist_cap", C.c_int),
                ("hist", C.c_void_p), ("seed", C.c_uint64), ("env_id", C.c_uint32), ("episode", C.c_uint32),
                ("step_in_episode", C.c_uint32), ("last_bot_action", C.c_int), ("forced_bot_action", C.c_int)]


_KEEP = ("initial_board", "hist", "hist_cap", "seed", "env_id", "episode", "forced_bot_action")
_libc = C.CDLL(None)
_libc.realloc.restype = C.c_void_p
_libc.realloc.argtypes = [C.c_void_p, C.c_size_t]


def _raw(o):
    e = _GcoEnv.from_address(o._h)
    v = o.view()  # the layout above must match the C struct
    assert (e.episode, e.step_in_episode, e.hist_n, e.n_legal, e.move_count, e.done) == (
        v["episode"], v["step_in_episode"], v["hist_n"], v["n_legal"], v["move_count"], v["done"]), "gco_env layout"
    return e


def oracle_clone(dst, src):
    """OracleEnv `dst` continues as `src` would (see the module docstring)"""
    a, b = _raw(dst), _raw(src)
    if a is b or dst._h == src._h:
        return
    if a.hist_cap < b.hist_n:
        p = _libc.realloc(a.hist, b.hist_cap * 64)
        assert p
        a.hist, a.hist_cap = p, b.hist_cap
    if b.hist_n:
        C.memmove(a.hist, b.hist, b.hist_n * 64)
    for name, _ in _GcoEnv._fields_:
        if name not in _KEEP:
            setattr(a, name, getattr(b, name))
    a.episode = (a.episode + 1) & 0xFFFFFFFF


def mixed_index(rng, n_dst, n_src):
    """-1 entries, fan-out (repeated rows) and a permutation block"""
    idx = rng.permutation(n_src)[:n_dst] if n_src >= n_dst else rng.randint(0, n_src, size=n_dst)
    idx = idx.astype(np.int32)
    k = n_dst // 4
    idx[:k] = -1
    idx[k:2 * k] = rng.randint(0, max(1, n_src // 8), size=k)  # a few roots, many children
    return idx


def run_actions(env, O, steps, rng, tot, auto_reset=True, tag=""):
    """step(actions): mostly a random legal action of the oracle, sometimes garbage -- against the oracle envs O"""
    N = env.N
    for t in range(steps):
        acts = np.zeros(N, np.int32)
        for i, o in enumerate(O):
            v = o.view()
            if v["n_legal"] > 0 and rng.rand() < 0.8:
                acts[i] = int(v["legal"][rng.randint(v["n_legal"])])
            else:
                acts[i] = int(rng.choice([rng.randint(0, 4101), 4100, 4096, 4099, 0]))
        r, d, f = env.step(acts)[:3]
        for i, o in enumerate(O):
            rr, dd, _ = o.step(int(acts[i]))
            v2 = o.view()
            assert (rr, dd) == (int(r[i]), bool(d[i])), (tag, t, i, int(acts[i]), (rr, dd), (int(r[i]), int(d[i])), int(f[i]))
            terminal = dd or v2["n_legal"] == 0
            assert bool(f[i] & 32) == (terminal and auto_reset), (tag, t, i, int(f[i]), terminal)
            tot["steps"] += 1
            tot["reward_sum"] += rr
            tot["episodes"] += int(terminal)
            if terminal and auto_reset:
                o.reset(v2["episode"] + 1)
    ph._cmp_export(env, O, tag + "after actions")


def stats_delta(after, before):
    a, b = np.asarray(after, np.uint64), np.asarray(before, np.uint64)
    d = (a - b).view(np.int64)
    return dict(steps=int(d[0]), reward_sum=int(d[8]), episodes=int(d[2]))


def check_clone_vs_oracle(make_env, opponent, color, n, rng, seed_src=11, seed_dst=29, offset_dst=100003, index=None):
    """Phase-spread a source batch (sampled steps with staggered masked resets) and a destination batch of another seed, id
    offset and auto_reset; clone with `index` (default: -1 entries, fan-out and a permutation); the destination's export
    must equal the oracle copies row by row (episode = the old destination episode + 1 on cloned rows); then >= 200
    further steps (caller words, external actions, sampled) against the oracle, and the statistics."""
    auto_dst = opponent != "none"
    S = make_env(n, opponent=opponent, player_color=color, seed=seed_src, auto_reset=True)
    OS = [orc.OracleEnv(None, color, opponent, seed_src, i) for i in range(n)]
    tot = dict(steps=0, reward_sum=0, episodes=0)
    for rnd in range(3):
        ph._run_sampled(S, OS, seed_src, 23 + 17 * rnd, tot, compare_every=1000, tag="source %d " % rnd)
        mask = (rng.rand(n) < 0.3).astype(np.uint8)
        S.reset(mask)
        for i, o in enumerate(OS):
            if mask[i]:
                o.reset(o.view()["episode"] + 1)
    D = make_env(n, opponent=opponent, player_color=color, seed=seed_dst, auto_reset=auto_dst, env_id_offset=offset_dst)
    OD = [orc.OracleEnv(None, color, opponent, seed_dst, offset_dst + j) for j in range(n)]
    tot_d = dict(steps=0, reward_sum=0, episodes=0)
    ph._run_sampled(D, OD, seed_dst, 9, tot_d, auto_reset=auto_dst, env_id_offset=offset_dst, compare_every=1000, tag="dest ")
    idx = mixed_index(rng, n, n) if index is None else np.asarray(index, np.int32)
    ep_before = D.export()[1][:, EPISODE_COL].copy()
    st_before = D.stats()
    D.clone_from(S, idx)
    for j, o in enumerate(OD):
        if 0 <= idx[j] < n:
            oracle_clone(o, OS[idx[j]])
    assert (np.asarray(D.stats()) == np.asarray(st_before)).all(), "a clone moves no statistics counter"
    info = D.export()[1]
    sel = (idx >= 0) & (idx < n)
    assert (info[sel, EPISODE_COL] == ep_before[sel] + 1).all() and (info[~sel, EPISODE_COL] == ep_before[~sel]).all()
    ph._cmp_export(D, OD, "after clone")
    tot = dict(steps=0, reward_sum=0, episodes=0)
    ph._run_sampled(D, OD, seed_dst, 90, tot, auto_reset=auto_dst, env_id_offset=offset_dst, mode="index", rng=rng,
                    compare_every=30, tag="clone index ")
    run_actions(D, OD, 40, rng, tot, auto_reset=auto_dst, tag="clone ")
    ph._run_sampled(D, OD, seed_dst, 90, tot, auto_reset=auto_dst, env_id_offset=offset_dst, compare_every=30, tag="clone sampled ")
    assert stats_delta(D.stats(), st_before) == tot, (stats_delta(D.stats(), st_before), tot)
    return S, D, idx


def assert_same_rows(src_exp, dst_exp, idx, tag=""):
    """export of every cloned row j equals that of source row idx[j], apart from the episode column"""
    sel = np.nonzero(idx >= 0)[0]
    if len(sel) == 0:
        return
    for a, b, name in zip(src_exp, dst_exp, ("boards", "info", "legal")):
        x, y = np.asarray(a)[idx[sel]], np.asarray(b)[sel]
        if name == "info":
            x, y = np.delete(x, EPISODE_COL, 1), np.delete(y, EPISODE_COL, 1)
        bad = np.nonzero((x != y).reshape(len(sel), -1).any(1))[0]
        assert len(bad) == 0, "%s%s differ at rows %s" % (tag, name, sel[bad[:10]])


def drive_pair(S, D, idx, steps, rng, external=False, check_every=25, tag=""):
    """Step S and D with the same inputs, gathered by idx (row j of D gets what row idx[j] of S gets; rows of D with
    idx < 0 get their own random inputs); every output of the cloned rows must equal that of their source rows.  Caller
    words (step_index) and, for the external opponent, the same bot plies.  D may be S (an in-object clone whose source
    rows are not themselves cloned rows): then one call steps both."""
    sel = idx >= 0
    same = D is S

    def both(call, x_s, x_d):
        if same:
            x_s = x_s.copy()
            x_s[sel] = x_s[idx[sel]]
            out = [np.array(v) for v in call(S)(x_s)[:3]]
            return out, out
        return [np.array(v) for v in call(S)(x_s)[:3]], [np.array(v) for v in call(D)(x_d)[:3]]

    def cmp(out_s, out_d, names, rows, t):
        for a, b, name in zip(out_s, out_d, names):
            assert (a[idx[rows]] == b[rows]).all(), "%sstep %d: %s differ at rows %s" % (tag, t, name, rows[np.nonzero(a[idx[rows]] != b[rows])[0][:10]])

    rows = np.nonzero(sel)[0]
    for t in range(steps):
        w = rng.randint(0, 2 ** 32, size=S.N, dtype=np.uint64).astype(np.uint32)
        wd = rng.randint(0, 2 ** 32, size=D.N, dtype=np.uint64).astype(np.uint32)
        wd[sel] = w[idx[sel]]
        out_s, out_d = both(lambda e: e.step_index, w, wd)
        cmp(out_s, out_d, ("reward", "done", "flags"), rows, t)
        if external:
            def bots(e):
                _, info, legal = e.export()
                n = np.maximum(info[:, 9], 1)
                return legal[np.arange(e.N), rng.randint(0, 1 << 30, size=e.N) % n].astype(np.int32), info
            b_s, info_s = bots(S)
            b_d = bots(D)[0]
            b_d[sel] = b_s[idx[sel]]
            out_s, out_d = both(lambda e: e.bot_ply, b_s, b_d)
            cmp(out_s, out_d, ("bot reward", "bot done", "bot flags"), rows[info_s[idx[rows], 14] == 1], t)
        if t % check_every == 0 or t == steps - 1:
            assert_same_rows(S.export(), D.export(), idx, "%sstep %d: " % (tag, t))
