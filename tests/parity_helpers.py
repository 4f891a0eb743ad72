"""Shared parity checks: the same comparisons run against
   * the oracle itself (pins the oracle to the fixtures made from the real chess_v2.py),
   * tests/host_emul (the device rules compiled with g++; logic check without a GPU),
   * the CUDA library through its C ABI (the parity tests proper, -m gpu).
An "env adapter" offers: N, step(actions), step_index(u32), step_sampled(), reset(mask), export(), stats();
step* return (reward, done, flags, agent_action, bot_action) as numpy arrays.
"""
import gzip
import json
import os

import numpy as np

from oracle import oracle as orc

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def load_golden():
    def gz(name):
        with gzip.open(os.path.join(GOLD, name)) as f:
            return json.loads(f.read())

    with open(os.path.join(GOLD, "reference_v2_tests.json")) as f:
        ref = json.load(f)
    return dict(reference_tests=ref, trajectories=gz("trajectories.json.gz"), positions=gz("positions.json.gz"),
                v1_move_sets=gz("v1_move_sets.json.gz"), render_info=gz("render_info.json.gz"),
                v1_next_states=gz("v1_next_states.json.gz"))


# ------------------------------------------------------------------ engine level
def check_positions(movegen_fn, update_fn, positions):
    """movegen_fn(boards, player(+1/-1), rights, attack) -> (actions[n,stride], counts[n], ...)"""
    boards = np.array([p["board"] for p in positions], np.int8)
    rights = np.array([p["rights"] for p in positions], np.uint8)
    for player, pname in ((1, "WHITE"), (-1, "BLACK")):
        for attack in (0, 1):
            res = movegen_fn(boards, player, rights, bool(attack))
            out, cnt = res[0], res[1]
            for i, p in enumerate(positions):
                exp = p["lists"]["%s_%d" % (pname, attack)]
                got = [int(x) for x in out[i, : cnt[i]]]
                assert got == exp, "position %d %s attack=%d\nboard=%s\nexp=%s\ngot=%s" % (
                    i, pname, attack, np.array(p["board"]).reshape(8, 8), exp, got)
    orr, oc = update_fn(boards, rights)
    exp = np.array([p["update_state"] for p in positions], np.uint8)
    assert (np.concatenate([orr, oc], 1) == exp).all()


def check_reference_test_calls(engine, report):
    """Replay every engine-visible call the reference's own v2 tests made (logged by make_golden.py)."""
    ncalls = 0
    for rec in report:
        if rec["module"] == "test_benchmark":
            continue
        assert rec["passed"], rec
        for c in rec["calls"]:
            st = c["state"]
            state = dict(board=np.array(st["board"], np.int8).reshape(8, 8).tolist(), current_player=st["player"],
                         white_king_castle_is_possible=bool(st["rights"][0]), white_queen_castle_is_possible=bool(st["rights"][1]),
                         black_king_castle_is_possible=bool(st["rights"][2]), black_queen_castle_is_possible=bool(st["rights"][3]))
            if c["kind"] == "get_possible_moves":
                got = [orc.str_to_action(m) for m in engine.get_possible_moves(state, c["player"], c["attack"])]
                assert got == c["actions"], (rec["test"], c)
            elif c["kind"] == "get_castle_moves":
                got = [orc.str_to_action(m) for m in engine.get_castle_moves(state, c["player"])]
                assert got == c["actions"], (rec["test"], c)
            else:  # a step of test_run_moves: the engine part is next_state
                ns, _ = engine.next_state(state, st["player"], orc.action_to_str(c["action"]))
                assert [v for row in ns["board"] for v in row] == c["board_after"], (rec["test"], c)
            ncalls += 1
    return ncalls


def harvest_positions(n_envs=64, steps=400, seed=1, every=3):
    """positions from oracle random self-play (uniform over the game), both sides to move"""
    boards, players, rights = [], [], []
    for i in range(n_envs):
        e = orc.OracleEnv(seed=seed, env_id=i)
        for t in range(steps):
            v = e.view()
            if t % every == i % every:
                boards.append(v["board"].copy())
                players.append(v["current_player"])
                rights.append([v["wk"], v["wq"], v["bk"], v["bq"]])
            u = orc.draw_u32(seed, i, v["episode"], v["step_in_episode"], 0)
            r, d, _ = e.step(e.pick(u))
            if d or e.view()["n_legal"] == 0:
                e.reset(v["episode"] + 1)
    return np.array(boards, np.int8), np.array(players, np.int8), np.array(rights, np.uint8)


def crafted_positions(rng, n=2000):
    """random piece soups: kingless, multi-king, many queens, pawns on last ranks, random rights"""
    boards = np.zeros((n, 64), np.int8)
    for i in range(n):
        k = rng.randint(1, 24)
        sq = rng.choice(64, size=k, replace=False)
        kind = rng.randint(4)
        if kind == 0:    # anything goes
            boards[i, sq] = rng.choice([-6, -5, -4, -3, -2, -1, 1, 2, 3, 4, 5, 6], size=k)
        elif kind == 1:  # exactly one king each + soup
            boards[i, sq] = rng.choice([-6, -5, -4, -3, -2, 2, 3, 4, 5, 6], size=k)
            boards[i, sq[0]] = 1
            if k > 1:
                boards[i, sq[1]] = -1
        elif kind == 2:  # castle shapes
            boards[i, sq] = rng.choice([-6, -5, -4, -3, 3, 4, 5, 6], size=k)
            boards[i, 56:64] = 0
            boards[i, 0:8] = 0
            boards[i, 60], boards[i, 56], boards[i, 63] = 1, 3, 3
            boards[i, 4], boards[i, 0], boards[i, 7] = rng.choice([-1, 1]), rng.choice([-3, 3]), rng.choice([-3, 3])
            if rng.rand() < 0.5:
                boards[i, rng.randint(56, 64)] = rng.choice([0, 0, 5, -5, 4])
        else:            # sliders heavy
            boards[i, sq] = rng.choice([-4, -3, -2, 2, 3, 4, 1, -1], size=k)
    players = rng.choice([-1, 1], size=n).astype(np.int8)
    rights = rng.randint(0, 2, size=(n, 4)).astype(np.uint8)
    return boards, players, rights


def check_movegen_vs_oracle(movegen_fn, boards, players, rights, attack=False, stride=256):
    res = movegen_fn(boards, players, rights, attack)
    out, cnt = res[0], res[1]
    exp, ecnt = orc.movegen_batch(boards, players, rights, attack, stride=stride, threads=os.cpu_count() or 1)
    assert (np.asarray(cnt) == ecnt).all(), "count mismatch at %s" % np.nonzero(np.asarray(cnt) != ecnt)[0][:10]
    mask = np.arange(stride)[None, :] < ecnt[:, None]
    bad = ((np.asarray(out)[:, :stride] != exp) & mask).any(1)
    assert not bad.any(), "list mismatch at %s" % np.nonzero(bad)[0][:10]
    return int(ecnt.sum())


def check_next_state_vs_oracle(next_state_fn, movegen_out, counts, boards, players, rights, rng):
    """play one random legal move (and some illegal / empty-square ones) from every position"""
    n = len(boards)
    idx = (rng.rand(n) * np.maximum(counts, 1)).astype(np.int64)
    actions = np.where(counts > 0, movegen_out[np.arange(n), idx], 4100).astype(np.int32)
    weird = rng.rand(n) < 0.15
    actions[weird] = rng.randint(0, 4100, size=int(weird.sum()))
    got = next_state_fn(boards, players, rights, actions)
    exp = orc.next_state_batch(boards, players, rights, actions)
    names = ("boards", "rights", "checks", "reward", "status")
    for g, e_, nm in zip(got, exp, names):
        assert (np.asarray(g).reshape(np.asarray(e_).shape) == e_).all(), nm


# ------------------------------------------------------------------ env level
def _cmp_export(env, oracles, tag):
    b, info, legal = env.export()
    for i, o in enumerate(oracles):
        v = o.view()
        mine = dict(board=[int(x) for x in b[i]], cp=int(info[i, 0]), fl=[int(x) for x in info[i, 1:7]], done=int(info[i, 7]),
                    mc=int(info[i, 8]), n=int(info[i, 9]), ep=int(info[i, 10]), st=int(info[i, 11]),
                    legal=[int(x) for x in legal[i, : info[i, 9]]])
        ref = dict(board=[int(x) for x in v["board"]], cp=v["current_player"], fl=[v[k] for k in "wk wq bk bq wchk bchk".split()],
                   done=v["done"], mc=v["move_count"], n=v["n_legal"], ep=v["episode"], st=v["step_in_episode"],
                   legal=[int(x) for x in v["legal"]])
        assert mine == ref, "%s env %d: %s" % (tag, i, {k: (mine[k], ref[k]) for k in mine if mine[k] != ref[k]})


def oracle_sampled_step(o, seed, env_id, tot, auto_reset=True, u=None):
    """One sampled step of oracle env `o` (global id env_id): the device's Philox draw (or the caller's word u), the step,
    and the device's auto-reset rule (a new episode when the step ended one or left no legal move).  Accumulates steps /
    reward_sum / episodes in `tot`.  -> (action, reward, done, view after the step and before any reset, terminal)"""
    v = o.view()
    if u is None:
        u = orc.draw_u32(seed, env_id, v["episode"], v["step_in_episode"], 0)
    act = o.pick(u)
    rr, dd, _ = o.step(act)
    v2 = o.view()
    terminal = dd or v2["n_legal"] == 0
    tot["steps"] += 1
    tot["reward_sum"] += rr
    tot["episodes"] += int(terminal)
    if terminal and auto_reset:
        o.reset(v2["episode"] + 1)
    return act, rr, dd, v2, terminal


def _run_sampled(env, O, seed, steps, tot, auto_reset=True, env_id_offset=0, compare_every=25, mode="sampled", rng=None, tag=""):
    """`steps` steps on the device env and the SAME draws through the oracle envs O; compares every output of every
    step and the full state every `compare_every` steps; accumulates steps / reward_sum / episodes in `tot`."""
    N = env.N
    for t in range(steps):
        words = None
        if mode == "sampled":
            r, d, f, a, bot = env.step_sampled()
        else:
            words = rng.randint(0, 2 ** 32, size=N, dtype=np.uint64).astype(np.uint32)
            r, d, f, a, bot = env.step_index(words)
        for i, o in enumerate(O):
            act, rr, dd, v2, terminal = oracle_sampled_step(o, seed, env_id_offset + i, tot, auto_reset,
                                                            None if words is None else int(words[i]))
            assert (rr, dd) == (int(r[i]), bool(d[i])), "%sstep %d env %d: oracle %s device %s flags %d" % (tag, t, i, (rr, dd), (r[i], d[i]), f[i])
            if a is not None:
                assert act == int(a[i]) and v2["last_bot_action"] == int(bot[i]), (tag, t, i, act, a[i], v2["last_bot_action"], bot[i])
            assert bool(f[i] & 32) == (terminal and auto_reset), (tag, t, i, int(f[i]), terminal)
            assert bool(f[i] & 16) == ((not dd) and v2["n_legal"] == 0), (tag, t, i, int(f[i]))
        if t % compare_every == 0 or t == steps - 1:
            _cmp_export(env, O, "%sstep %d" % (tag, t))


# the info columns a device export (BatchedChessEnv.INFO_NAMES) and an oracle view (OracleEnv.view / SelfplayPool.export)
# share, in this order; column 12 differs on purpose (the device's repetition window hist_len vs the oracle's hist_n)
EXPORT_FIELDS = ("current_player", "wk", "wq", "bk", "bq", "wchk", "bchk", "done", "move_count", "n_legal", "episode",
                 "step_in_episode")


def oracle_views(O, stride=256):
    """OracleEnv.view() of every env of O as the arrays of SelfplayPool.export(stride)"""
    n = len(O)
    boards, info, legal = np.zeros((n, 64), np.int8), np.zeros((n, 16), np.int32), np.zeros((n, stride), np.uint16)
    for i, o in enumerate(O):
        v = o.view()
        boards[i] = v["board"]
        info[i, : len(EXPORT_FIELDS)] = [v[k] for k in EXPORT_FIELDS]
        k = min(v["n_legal"], stride)
        legal[i, :k] = v["legal"][:k]
    return boards, info, legal


def check_export_arrays(got, ref, env_id_offset=0, tag="", show=8):
    """got / ref: (boards [n,64], info [n,>=12], legal [n,stride]) with info columns EXPORT_FIELDS.  Board, every shared
    info column and the legal list in order (its first min(n_legal, stride) entries) must agree for every env; on a
    mismatch the message names the first `show` global env ids and, for each, the fields that differ."""
    (b, info, legal), (rb, rinfo, rlegal) = got, ref
    nf = len(EXPORT_FIELDS)
    stride = min(legal.shape[1], rlegal.shape[1])
    valid = np.arange(stride)[None, :] < np.minimum(rinfo[:, 9], stride)[:, None]
    bad_board = (np.asarray(b) != rb).any(1)
    bad_info = np.asarray(info)[:, :nf] != rinfo[:, :nf]
    bad_legal = ((np.asarray(legal)[:, :stride] != rlegal[:, :stride]) & valid).any(1)
    bad = bad_board | bad_info.any(1) | bad_legal
    if not bad.any():
        return
    lines = []
    for i in np.nonzero(bad)[0][:show]:
        diff = {EXPORT_FIELDS[k]: (int(info[i, k]), int(rinfo[i, k])) for k in np.nonzero(bad_info[i])[0]}
        if bad_board[i]:
            diff["board"] = "squares %s" % np.nonzero(b[i] != rb[i])[0].tolist()
        if bad_legal[i]:
            diff["legal"] = "first difference at index %d" % int(np.argmax((legal[i, :stride] != rlegal[i, :stride]) & valid[i]))
        lines.append("  env id %d (row %d): %s" % (env_id_offset + i, i, diff))
    raise AssertionError("%s%d of %d envs differ (values: got, reference)\n%s" % (tag, int(bad.sum()), len(bad), "\n".join(lines)))


def _check_totals(env, tot):
    st = env.stats()
    assert int(st[0]) == tot["steps"] and int(np.array(st[8:9], np.uint64).view(np.int64)[0]) == tot["reward_sum"] and int(st[2]) == tot["episodes"], (st, tot)
    return st


def check_sampled_vs_oracle(env, opponent, color, seed, steps, auto_reset=True, boards=None, env_id_offset=0,
                            compare_every=25, mode="sampled", rng=None, moves_max=149):
    """Run `steps` steps on the device env and replay the SAME draws through N oracle envs; compare every output of
    every step, the full state every `compare_every` steps, and the statistics at the end."""
    N = env.N
    nt = 1 if boards is None else len(boards)
    O = [orc.OracleEnv(None if boards is None else boards[(env_id_offset + i) % nt], color, opponent, seed, env_id_offset + i,
                       moves_max=moves_max)
         for i in range(N)]
    _cmp_export(env, O, "reset")
    tot = dict(steps=0, reward_sum=0, episodes=0)
    _run_sampled(env, O, seed, steps, tot, auto_reset, env_id_offset, compare_every, mode, rng)
    return _check_totals(env, tot)


def check_external_actions_vs_oracle(env, opponent, color, seed, steps, rng, auto_reset):
    """step(actions) with caller-chosen actions: mostly a random entry of the oracle's legal list, sometimes garbage
    (illegal squares, castles, RESIGN, repeats after done) -- the invalid / done / cap early exits of chess_v2.py:240-258
    in every opponent mode, with and without auto-reset."""
    N = env.N
    O = [orc.OracleEnv(None, color, opponent, seed, i) for i in range(N)]
    tot = dict(steps=0, reward_sum=0, episodes=0)
    for t in range(steps):
        acts = np.zeros(N, np.int32)
        for i, o in enumerate(O):
            v = o.view()
            if v["n_legal"] > 0 and rng.rand() < 0.8:
                acts[i] = int(v["legal"][rng.randint(v["n_legal"])])
            else:
                acts[i] = int(rng.choice([rng.randint(0, 4101), 4100, 4096, 4097, 4098, 4099, 0, 4095]))
        r, d, f, _, _ = env.step(acts)
        for i, o in enumerate(O):
            rr, dd, raised = o.step(int(acts[i]))
            v2 = o.view()
            assert (rr, dd) == (int(r[i]), bool(d[i])), (t, i, int(acts[i]), (rr, dd), (int(r[i]), int(d[i])), int(f[i]))
            terminal = dd or v2["n_legal"] == 0
            assert bool(f[i] & 32) == (terminal and auto_reset), (t, i, int(f[i]), terminal)
            tot["steps"] += 1
            tot["reward_sum"] += rr
            tot["episodes"] += int(terminal)
            if terminal and auto_reset:
                o.reset(v2["episode"] + 1)
        if t % 20 == 0 or t == steps - 1:
            _cmp_export(env, O, "step %d" % t)
    return _check_totals(env, tot)


def check_state_import_vs_oracle(env, opponent, color, seed, rng):
    """State import (the `state` setter for many envs): play, import harvested positions (random side to move, rights,
    move counters incl. values next to the 150-move cap) into a masked half of the envs, keep playing -- all against the
    oracle doing the same."""
    N = env.N
    O = [orc.OracleEnv(None, color, opponent, seed, i) for i in range(N)]
    tot = dict(steps=0, reward_sum=0, episodes=0)
    _run_sampled(env, O, seed, 40, tot, tag="before import ")
    hb, hp, hr = harvest_positions(n_envs=24, steps=300, seed=9)
    for rnd in range(3):
        pick = rng.randint(0, len(hb), size=N)
        boards, players, rights = hb[pick], hp[pick] * rng.choice([-1, 1], size=N).astype(np.int8), rng.randint(0, 2, size=(N, 4)).astype(np.uint8)
        move_count = rng.choice([0, 7, 148, 149, 150], size=N).astype(np.int32)
        mask = (rng.rand(N) < 0.5).astype(np.uint8)
        env.set_state(boards, players, rights, move_count, mask)
        for i, o in enumerate(O):
            if mask[i]:
                o.import_state(boards[i], int(players[i]), rights[i], int(move_count[i]), episode=o.view()["episode"] + 1)
        _cmp_export(env, O, "import %d" % rnd)
        _run_sampled(env, O, seed, 60, tot, tag="after import %d " % rnd)
        # a masked reset in mid-game (ChessEnvV2.reset of some envs), the others keep their repetition windows
        mask = (rng.rand(N) < 0.3).astype(np.uint8)
        env.reset(mask)
        for i, o in enumerate(O):
            if mask[i]:
                o.reset(o.view()["episode"] + 1)
        _cmp_export(env, O, "masked reset %d" % rnd)
        _run_sampled(env, O, seed, 30, tot, tag="after masked reset %d " % rnd)
    return _check_totals(env, tot)


def check_trajectory_replay(make_env, traj):
    """Replay a recorded self-play game (opponent none) of the REAL chess_v2.py through a 1-env device env."""
    assert traj["opponent"] == "none"
    env = make_env(np.array(traj["initial_board"], np.int8))

    def cmp(s, where):
        b, info, legal = env.export()
        assert [int(x) for x in b[0]] == s["board"], where
        assert [int(x) for x in info[0, 1:7]] == s["flags"], where
        assert int(info[0, 8]) == s["move_count"], where
        assert int(info[0, 0]) == (1 if s["current_player"] == "WHITE" else -1), where
        assert [int(x) for x in legal[0, : info[0, 9]]] == s["legal"], where

    cmp(traj["reset"], (traj["name"], "reset"))
    for i, s in enumerate(traj["steps"]):
        r, d, f, _, _ = env.step(np.array([s["action"]], np.int32))
        assert (int(r[0]), bool(d[0])) == (int(s["reward"]), bool(s["done"])), (traj["name"], traj["seed"], i, r, d, s["reward"], s["done"])
        cmp(s, (traj["name"], traj["seed"], i))
    return len(traj["steps"])


def check_external_bot_replay(make_env, traj):
    """Replay a recorded game of the REAL chess_v2.py against its (callable) bot through a 1-env device env created with
    opponent="external": every step stops where the bot would move (F_BOT_PENDING) and the recorded bot move is supplied
    with bot_ply() -- WHITE and BLACK agents (the BLACK agent's reset owes White's opening ply, chess_v2.py:208-216)."""
    assert traj["opponent"] == "random"
    env = make_env(np.array(traj["initial_board"], np.int8), traj["player_color"])

    def cmp(s, where):
        b, info, legal = env.export()
        assert [int(x) for x in b[0]] == s["board"], where
        assert [int(x) for x in info[0, 1:7]] == s["flags"], where
        assert int(info[0, 8]) == s["move_count"], where
        assert int(info[0, 0]) == (1 if s["current_player"] == "WHITE" else -1), where
        assert [int(x) for x in legal[0, : info[0, 9]]] == s["legal"], where
        assert int(info[0, 14]) == 0, where  # nothing owed between steps

    if traj["player_color"] == "BLACK":
        assert int(env.export()[1][0, 14]) == 1  # the opening ply is owed
        env.bot_ply(np.array([traj["reset"]["bot_action"]], np.int32))
    cmp(traj["reset"], (traj["name"], "reset"))
    n = 0
    for i, s in enumerate(traj["steps"]):
        if s["raised"]:  # the bot had no move: the reference raises TypeError (Q9); here the ply stays owed
            r, d, f = env.step(np.array([s["action"]], np.int32))[:3]
            assert int(f[0]) & 64 and s["bot_action"] < 0
            break
        r, d, f = env.step(np.array([s["action"]], np.int32))[:3]
        reward, done = int(r[0]), bool(d[0])
        if int(f[0]) & 64:
            assert s["bot_action"] >= 0, (traj["name"], i)
            r2, d2, f2 = env.bot_ply(np.array([s["bot_action"]], np.int32))[:3]
            reward, done = reward + int(r2[0]), bool(d2[0])
        else:
            assert s["bot_action"] < 0, (traj["name"], i)
        assert (reward, done) == (int(s["reward"]), bool(s["done"])), (traj["name"], traj["seed"], i, reward, done, s["reward"], s["done"])
        cmp(s, (traj["name"], traj["seed"], i))
        n += 1
    return n


def check_v1_next_states(next_state_fn, records):
    """`next_state` of the reference's own pure-Python env (chess_v1.py:366-450, unmodified; tests/golden/
    make_golden_v1_next.py): board after the move, reward (capture value, K = 0; the dead promotion of Q1 by direct call)
    and both check flags (v1.py:1008-1026) for plain moves, castles and pawn moves onto the wrong last rank.  Rights are
    not compared (v1 tracks them differently, SURVEY.md 9.4)."""
    boards = np.array([r["board"] for r in records], np.int8)
    players = np.array([r["player"] for r in records], np.int8)
    actions = np.array([r["action"] for r in records], np.int32)
    ob, orr, oc, rew, st = next_state_fn(boards, players, np.ones((len(records), 4), np.uint8), actions)
    ob, oc, rew, st = np.asarray(ob).reshape(-1, 64), np.asarray(oc).reshape(-1, 2), np.asarray(rew), np.asarray(st)
    exp_b = np.array([r["board_after"] for r in records], np.int8)
    assert (ob == exp_b).all(), np.nonzero((ob != exp_b).any(1))[0][:10]
    assert (rew == np.array([r["reward"] for r in records])).all()
    assert (st >= 0).all()
    for i, r in enumerate(records):
        if r["checks"] is not None:
            assert [int(x) for x in oc[i]] == r["checks"], (i, r)
    return len(records)


def check_v1_castle_through_attack_vector(castle_moves_fn):
    """gym_chess/test/v1/test_castle_moves.py:54-74 (commented out in the v2 twin, same rule in lib.rs:966-1012): white pawns
    on rank 2 except c2, Ra1, Ke1, black Rc8 -> c1 is attacked, no queen-side castle; with the c-pawn back it is offered.
    castle_moves_fn(board int8[64], player) -> list of action codes."""
    b = np.zeros(64, np.int8)
    b[48:56] = 6
    b[50] = 0
    b[2], b[56], b[60] = -3, 3, 1
    assert castle_moves_fn(b, 1) == []
    b[50] = 6
    assert castle_moves_fn(b, 1) == [4097]
    b[63] = 3                                             # and with Rh1 both, queen side first (lib.rs:992, 1011)
    assert castle_moves_fn(b, 1) == [4097, 4096]


def queen_heavy_boards():
    """initial boards on which White has more than 255 legal moves (found by hill climbing; 266 and 271 moves).  Sixteen
    pieces cannot get there (best found: 243), so these have 24 and 28 white pieces -> more than 16 piece slots."""
    a = [-1, 0, 2, 0, 2, 2, 2, -3, 2, 2, 0, 0, 0, 0, 0, 2, 0, 0, 0, 2, 0, 0, 0, 2, 2, 0, 0, 0, 0, 0, 0, 2, 2, 0, 0, 0, 0, 0, 0, 2,
         1, 0, 2, 0, 0, 0, 0, 2, 2, 0, 0, 0, 0, 0, 0, 2, 0, 2, 2, 2, 2, 2, 2, 0]
    b = [-1, 2, 2, 2, 2, 2, 2, -3, 2, 2, 0, 0, 0, 0, 0, 2, 2, 0, 0, 0, 0, 2, 0, 2, 2, 0, 0, 0, 0, 0, 0, 2, 2, 0, 0, 0, 0, 0, 0, 1,
         2, 0, 0, 0, 0, 0, 0, 2, 2, 0, 0, 0, 0, 0, 0, 2, 2, 2, 2, 2, 2, 2, 2, 2]
    return np.array([a, b], np.int8)


def endgame_boards():
    """BASELINE.json configs[4]: repetition-heavy endgames (the presets live in the package: gym_chess_b200/boards.py)"""
    from gym_chess_b200.boards import endgame_boards as eb
    return eb()


def check_v1_move_sets(movegen_fn, records):
    """Move lists of the reference's own pure-Python env (chess_v1.py, unmodified; tests/golden/make_golden_v1.py): an
    implementation that shares no code with lib.rs or with the oracle.  v1 never captures a king with a non-pawn piece
    and castles under other conditions (SURVEY.md 9.4): castles and moves onto the enemy king square are dropped from
    both sides, everything else must agree exactly -- as SETS and in ORDER, for both colours.  The one documented order
    difference is normalised: v1 lists a black pawn's captures as (col-1, col+1), v2 as (col+1, col-1) for both colours
    (v1.py:761-764 vs lib.rs:921-924)."""
    boards = np.array([r["board"] for r in records], np.int8)
    players = np.array([r["player"] for r in records], np.int8)
    res = movegen_fn(boards, players, np.zeros((len(records), 4), np.uint8), False)
    out, cnt = res[0], res[1]
    n = 0
    for i, r in enumerate(records):
        eking = int(np.nonzero(boards[i] == -r["player"])[0][0])
        mine = [(int(a) >> 6, int(a) & 63) for a in out[i, : cnt[i]] if a < 4096 and (int(a) & 63) != eking]
        theirs = [tuple(m) for m in r["moves"] if not isinstance(m, str) and m[1] != eking]
        assert set(mine) == set(theirs), (i, np.array(r["board"]).reshape(8, 8), r["player"], sorted(set(mine) ^ set(theirs)))
        if r["player"] < 0:
            k = 0
            while k + 1 < len(theirs):
                (f0, t0), (f1, t1) = theirs[k], theirs[k + 1]
                if f0 == f1 and boards[i][f0] == -6 and t0 == f0 + 7 and t1 == f0 + 9:
                    theirs[k], theirs[k + 1] = theirs[k + 1], theirs[k]
                    k += 2
                else:
                    k += 1
        assert mine == theirs, ("order", i, np.array(r["board"]).reshape(8, 8), r["player"], mine, theirs)
        n += len(theirs)
    # attack=True lists (v1's get_possible_moves(attack=True)): the whole ordered list, same black-pawn normalisation
    if records and "attack" in records[0]:
        res = movegen_fn(boards, players, np.zeros((len(records), 4), np.uint8), True)
        out, cnt = res[0], res[1]
        for i, r in enumerate(records):
            mine = [(int(a) >> 6, int(a) & 63) for a in out[i, : cnt[i]]]
            theirs = [tuple(m) for m in r["attack"]]
            if r["player"] < 0:
                k = 0
                while k + 1 < len(theirs):
                    (f0, t0), (f1, t1) = theirs[k], theirs[k + 1]
                    if f0 == f1 and boards[i][f0] == -6 and t0 == f0 + 7 and t1 == f0 + 9:
                        theirs[k], theirs[k + 1] = theirs[k + 1], theirs[k]
                        k += 2
                    else:
                        k += 1
            assert mine == theirs, ("attack", i, np.array(r["board"]).reshape(8, 8), r["player"], mine, theirs)
            n += len(theirs)
    return n
