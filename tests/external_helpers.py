"""Reference model of envs with an external opponent (opponent="external": the caller supplies the bot's plies with
bot_ply), shared by the host-emulation test and the GPU test.

Each env pairs with one oracle env of the "random" kind whose bot moves are forced to the plies the driver supplies
(OracleEnv.step(action, bot_action=b); for White's opening of a BLACK-agent episode, gco_env_force_bot + gco_env_reset).
The oracle plays the agent's ply and the bot's reply in one call, so the model adds what the device exposes in between:
  * the owed ply: None, "reply" (the agent's ply is played, the bot's reply is owed) or "opening" (a BLACK-agent episode
    has begun, White's opening is owed); the position the env shows while a reply is owed comes from the oracle's engine
    (next_state + the bot's move list);
  * refused steps (a step while a ply is owed: -10, F_INVALID | F_BOT_PENDING, nothing else changes);
  * the per-step flags, F_BOT_PENDING = "a ply is owed when the call returns";
  * the statistics counters except hist_scanned (which counts probes of the device's hash table): the pre-move boards of
    the episode give F_REPETITION independently of F_MATE, the reversible window (plies since the last pawn move or
    capture, chess_core.cuh apply_action) gives hist_len and hist_window.
Counters are classified like gco_selfplay does (n_legal == 0 before the step -> none; done before -> none; cap; mate or
repetition; wedged) and counted where the device ends the step: a step that leaves a reply owed ends nothing.

An env adapter offers call(form, inputs) (a step; see run_external), bot_ply(actions), reset(mask), export(), stats(); a
step returns (reward, done, flags, the reported actions or None), bot_ply returns (reward, done, flags) over output rows
that it filled with SENTINEL first, so that rows that owed nothing must still hold it.
"""
import numpy as np

from oracle import oracle as orc

F_INVALID, F_MATE, F_REPETITION, F_CAP, F_WEDGED, F_RESET, F_BOT_PENDING = 1, 2, 4, 8, 16, 32, 64
ACT_RESIGN = 4100
SENTINEL = (77, 7, 199)  # reward, done, flags a bot_ply must not write for rows that owe nothing
(ST_STEPS, ST_PLIES, ST_EPISODES, ST_MATES, ST_REPS, ST_CAPS, ST_WEDGED, ST_INVALID, ST_REWARD, ST_LEGAL, ST_INCHECK,
 ST_HISTOVF, ST_SLOTOVF, ST_HISTSCAN, ST_WINDOW) = range(15)


def _castle_bits(legal):
    """info[13]: bit 0 a queen-side castle is legal, bit 1 a king-side castle"""
    s = set(int(a) for a in legal)
    return (1 if s & {4097, 4099} else 0) | (2 if s & {4096, 4098} else 0)


def _irreversible(board, action):
    """apply_action's test: a pawn moves or the target square is occupied (castles are reversible)"""
    if action >= 4096:
        return False
    return abs(int(board[action >> 6])) == 6 or int(board[action & 63]) != 0


def _pick(legal, u32):
    n = len(legal)
    return int(legal[(int(u32) * n) >> 32]) if n else ACT_RESIGN


class ExternalModel:
    """one env with an external opponent (see the module docstring)"""

    def __init__(self, initial_board, color, seed, env_id, auto_reset, moves_max):
        self.ib = np.asarray(orc.default_board() if initial_board is None else initial_board, np.int8).reshape(64)
        self.black, self.auto_reset, self.moves_max = color == "BLACK", bool(auto_reset), int(moves_max)
        self.o = orc.OracleEnv(self.ib, color, "random", seed, env_id, moves_max=moves_max)
        v = orc.OracleEnv(self.ib, "WHITE", "none").view()  # the position of a fresh episode before any ply
        self.start = dict(board=v["board"].copy(), cp=1, fl=[v[k] for k in "wk wq bk bq wchk bchk".split()], done=0, mc=0,
                          n=v["n_legal"], legal=[int(x) for x in v["legal"]], st=0)
        assert self.start["n"] > 0  # White can open on every board the tests use
        self.stats = np.zeros(15, np.int64)
        self.ep = 0
        self.needs_reset = False  # the agent's ply left the bot without a move (the reference raises, Q9): reset both sides
        self._new_episode(first=True)

    # ------------------------------------------------------------------ state
    def _new_episode(self, first=False):
        if not first:
            self.ep += 1
        self.hist, self.hist_len = [], 0  # pre-move boards of the episode; plies since the last irreversible one
        self.needs_reset = False
        self.reply = None
        if self.black:
            self.owed = "opening"
        else:
            self.owed = None
            if not first:
                self.o.reset(self.ep)

    def reset(self):
        """a masked reset of this env (no statistics)"""
        self._new_episode()

    def _ply(self, pre_board, action):
        """bookkeeping of one applied ply from pre_board: -> the pre-move board's 3rd occurrence (F_REPETITION)"""
        rep = sum(1 for h in self.hist if (h == pre_board).all()) + 1 >= 3
        self.hist.append(pre_board.copy())
        self.stats[ST_PLIES] += 1
        self.stats[ST_WINDOW] += self.hist_len
        self.hist_len = 0 if _irreversible(pre_board, action) else min(self.hist_len + 1, 511)
        return rep

    def view(self):
        """the env as export() must show it: dict(board, info int[16], legal)"""
        if self.owed == "opening":
            s = dict(self.start, ep=self.ep)
        elif self.owed == "reply":
            s = self.reply["view"]
        else:
            v = self.o.view()
            s = dict(board=v["board"], cp=v["current_player"], fl=[v[k] for k in "wk wq bk bq wchk bchk".split()], done=v["done"],
                     mc=v["move_count"], n=v["n_legal"], ep=v["episode"], st=v["step_in_episode"], legal=[int(x) for x in v["legal"]])
        info = [s["cp"]] + list(s["fl"]) + [s["done"], s["mc"], s["n"], s["ep"], s["st"], self.hist_len, _castle_bits(s["legal"]),
                                            int(self.owed is not None), 0]
        return dict(board=np.asarray(s["board"], np.int8), info=np.array(info, np.int64), legal=list(s["legal"]))

    def _stm_checked(self, view):
        return int(view["info"][5] if view["info"][0] > 0 else view["info"][6])

    # ------------------------------------------------------------------ calls
    def _finish(self, R, d_out, fl, n0, was_done, capped, owe_bot, n_after):
        """the end of a step or bot ply: F_WEDGED / F_RESET / F_BOT_PENDING, the episode classification, auto-reset"""
        terminal = not owe_bot and (d_out or n_after == 0)
        if not owe_bot and not d_out and n_after == 0:
            fl |= F_WEDGED
        if n0 == 0 or was_done or owe_bot or fl & F_INVALID:
            pass
        elif capped:
            self.stats[ST_CAPS] += 1
        elif d_out:
            self.stats[ST_MATES if fl & F_MATE else ST_REPS] += 1
        elif n_after == 0:
            self.stats[ST_WEDGED] += 1
        self.stats[ST_EPISODES] += int(terminal)
        self.stats[ST_REWARD] += R
        if self.auto_reset and terminal:
            fl |= F_RESET
            self._new_episode()
        if self.owed is not None:
            fl |= F_BOT_PENDING
        return R, int(d_out), fl

    def step(self, action=None, word=None, choose_bot=None):
        """one step with `action`, or with the index word `word` (step_index: the agent plays legal[(word * n) >> 32]);
        choose_bot(bot_legal, board, side) -> the bot's reply the driver will supply if this step leaves one owed.
        -> (reward, done, flags, the action the device reports)"""
        v = self.view()
        n0, chk = int(v["info"][9]), self._stm_checked(v)
        if word is not None:
            action = _pick(v["legal"], word)
        self.stats[ST_STEPS] += 1
        self.stats[ST_LEGAL] += n0
        self.stats[ST_INCHECK] += chk
        if self.owed is not None:  # refused: the env keeps its state
            self.stats[ST_INVALID] += 1
            return self._finish(-10, False, F_INVALID, n0, False, False, False, n0) + (action,)
        ov = self.o.view()
        was_done, capped = bool(ov["done"]), ov["move_count"] > self.moves_max
        if action not in v["legal"]:  # chess_v2.py:240-242, before the done test
            rr, dd, _ = self.o.step(action)
            assert (rr, dd) == (-10, was_done)
            self.stats[ST_INVALID] += 1
            return self._finish(-10, was_done, F_INVALID, n0, was_done, capped, False, n0) + (action,)
        if was_done or capped:
            rr, dd, _ = self.o.step(action)
            assert (rr, dd) == (0, True)
            return self._finish(0, True, 0 if was_done else F_CAP, n0, was_done, capped, False, n0) + (action,)
        # the agent's ply, and what the position is when the step ends
        pre, cp = ov["board"].copy(), ov["current_player"]
        rights = np.array([[ov["wk"], ov["wq"], ov["bk"], ov["bq"]]], np.uint8)
        ob, orr, oc, rew, status = orc.next_state_batch(pre[None], cp, rights, [action])
        assert status[0] >= 0
        rep = self._ply(pre, action)
        bl, bn = orc.movegen_batch(ob, -cp, orr, stride=512)
        bot_legal = [int(x) for x in bl[0, : bn[0]]]
        bot_checked = int(oc[0, 0] if -cp > 0 else oc[0, 1])
        mate = not bot_legal and bot_checked
        R = -10 + int(rew[0]) + (100 if mate else 0)
        fl = (F_REPETITION if rep else 0) | (F_MATE if mate else 0)
        done = bool(rep or mate)
        if done:
            rr, dd, _ = self.o.step(action)
            assert (rr, dd) == (R, True), (rr, dd, R)
            return self._finish(R, True, fl, n0, False, False, False, int(self.o.view()["n_legal"])) + (action,)
        view = dict(board=ob[0].copy(), cp=-cp, fl=[int(x) for x in orr[0]] + [int(x) for x in oc[0]], done=0, mc=ov["move_count"],
                    n=len(bot_legal), ep=ov["episode"], st=ov["step_in_episode"] + 1, legal=bot_legal)
        if not bot_legal:  # the bot has no move and is not mated: the reference raises (Q9); the driver resets this env
            _, _, raised = self.o.step(action)
            assert raised
            self.needs_reset = True
            self.owed, self.reply = "reply", dict(view=view)
            return self._finish(R, False, fl, n0, False, False, True, 0) + (action,)
        b = int(choose_bot(bot_legal, ob[0], -cp))
        rr, dd, raised = self.o.step(action, bot_action=b)
        assert not raised
        self.owed = "reply"
        self.reply = dict(view=view, action=b, R=rr - R, done=bool(dd), capped=ov["move_count"] > self.moves_max)
        return self._finish(R, False, fl, n0, False, False, True, len(bot_legal)) + (action,)

    def bot_action(self, choose_bot):
        """the action the driver passes to bot_ply for this env (-> None if nothing is owed: any value will do)"""
        if self.owed == "reply":
            return self.reply["action"]
        if self.owed == "opening":
            self.opening = int(choose_bot(self.start["legal"], self.start["board"], 1))
            return self.opening
        return None

    def bot_ply(self):
        """-> (reward, done, flags, act_out) of the bot's ply, or None if nothing is owed (the row must stay untouched)"""
        if self.owed is None:
            return None
        if self.owed == "opening":
            b = self.opening
            self._ply(self.start["board"], b)
            L = orc.lib()
            L.gco_env_force_bot(self.o._h, b)
            self.o.reset(self.ep)
            L.gco_env_force_bot(self.o._h, -1)
            self.owed = None
            return 0, 0, 0, b
        rp = self.reply
        pre = rp["view"]["board"]
        rep = self._ply(pre, rp["action"])
        self.owed, self.reply = None, None
        v2 = self.o.view()
        agent_checked = v2["wchk"] if v2["current_player"] > 0 else v2["bchk"]
        mate = v2["n_legal"] == 0 and bool(agent_checked)
        assert rp["done"] == bool(rep or mate), (rp["done"], rep, mate)
        fl = (F_REPETITION if rep else 0) | (F_MATE if mate else 0)
        return self._finish(rp["R"], rp["done"], fl, rp["view"]["n"], False, rp["capped"], False, v2["n_legal"]) + (rp["action"],)


def cmp_export(env, models, tag):
    """the full export (board, all 16 info fields, the legal list) of every env against its model"""
    b, info, legal = env.export()
    for i, m in enumerate(models):
        v = m.view()
        mine = dict(board=[int(x) for x in b[i]], info=[int(x) for x in info[i]], legal=[int(x) for x in legal[i, : info[i, 9]]])
        ref = dict(board=[int(x) for x in v["board"]], info=[int(x) for x in v["info"]], legal=v["legal"])
        assert mine == ref, "%s env %d (owed %s): %s" % (tag, i, m.owed, {k: (mine[k], ref[k]) for k in mine if mine[k] != ref[k]})


def make_models(N, color, seed, auto_reset, moves_max, boards=None):
    nt = 1 if boards is None else len(boards)
    return [ExternalModel(None if boards is None else boards[i % nt], color, seed, i, auto_reset, moves_max) for i in range(N)]


WORD_FORMS = {"index": 32, "index_host": 32, "index_packed": 16}  # the other forms take action codes


def run_external(env, models, rng, calls, forms=("step",), compare_every=6, p_bot=0.4, p_garbage_bot=0.1, p_reset=0.02):
    """`calls` random calls on the env and the models: a step through env.call(form, inputs) -- forms "step", "host",
    "packed" take action codes (mostly legal, sometimes not), forms in WORD_FORMS random words of that width -- or a bot_ply
    with mostly legal and sometimes unlisted bot moves; now and then a masked reset.  Every output is compared every call,
    the export every `compare_every` calls and after each reset.  -> the models' statistics summed (int64[15])"""
    N = len(models)

    def choose_bot(legal, board, side):
        if legal and rng.rand() >= p_garbage_bot:
            return legal[rng.randint(len(legal))]
        # a move that is not in the list, by one of the bot's own pieces (moving an enemy pawn onto the wrong last rank
        # would turn it into a queen of the mover's colour, Q1: a 17th piece, beyond the env's piece slots; from == to would
        # "capture" the mover itself)
        f = int(rng.choice(np.nonzero(np.asarray(board) * side > 0)[0]))
        t = int(rng.choice([s for s in range(64) if s != f]))
        return f * 64 + t

    for c in range(calls):
        if rng.rand() < p_bot:
            kind = "bot_ply"
            acts = np.zeros(N, np.int32)
            for i, m in enumerate(models):
                a = m.bot_action(choose_bot)
                acts[i] = rng.randint(0, 4100) if a is None else a
            r, d, f = env.bot_ply(acts)[:3]
            for i, m in enumerate(models):
                exp = m.bot_ply()
                got = (int(r[i]), int(d[i]), int(f[i]))
                if exp is None:
                    assert got == SENTINEL, ("call %d bot_ply env %d owed nothing but its outputs were written" % (c, i), got)
                else:
                    assert got == exp[:3], ("call %d bot_ply env %d" % (c, i), int(acts[i]), got, exp)
        else:
            kind = forms[rng.randint(len(forms))]
            bits = WORD_FORMS.get(kind)
            if bits is None:
                inp = np.zeros(N, np.int32)
                for i, m in enumerate(models):
                    legal = m.view()["legal"]
                    if legal and rng.rand() < 0.85:
                        inp[i] = legal[rng.randint(len(legal))]
                    else:
                        inp[i] = int(rng.choice([rng.randint(0, 4101), ACT_RESIGN, 4096, 4099, 0]))
            else:
                inp = rng.randint(0, 2 ** bits, size=N, dtype=np.uint64).astype(np.uint32 if bits == 32 else np.uint16)
            r, d, f, a_out = env.call(kind, inp)
            for i, m in enumerate(models):
                kw = dict(action=int(inp[i])) if bits is None else dict(word=int(inp[i]) << (32 - bits))
                e = m.step(choose_bot=choose_bot, **kw)
                got = (int(r[i]), int(d[i]), int(f[i]))
                assert got == e[:3], ("call %d %s env %d" % (c, kind, i), int(inp[i]), got, e[:3])
                if a_out is not None:
                    assert int(a_out[i]) == e[3], ("call %d %s env %d action" % (c, kind, i), int(a_out[i]), e[3])
            need = np.array([m.needs_reset for m in models], np.uint8)
            if need.any():  # bots without a move: reset both sides of those envs
                env.reset(need)
                for i in np.nonzero(need)[0]:
                    models[i].reset()
        mask = (rng.rand(N) < p_reset).astype(np.uint8)
        if mask.any():
            env.reset(mask)
            for i in np.nonzero(mask)[0]:
                models[i].reset()
        if c % compare_every == 0 or c == calls - 1 or mask.any():
            cmp_export(env, models, "call %d (%s)" % (c, kind))
    return sum(m.stats for m in models)


def check_totals(env, models_sum):
    """the first 15 statistics counters except hist_scanned, exactly"""
    st = np.asarray(env.stats()[:15]).astype(np.uint64).view(np.int64)
    for k in range(15):
        if k != ST_HISTSCAN:
            assert int(st[k]) == int(models_sum[k]), ("counter %d" % k, int(st[k]), int(models_sum[k]), st.tolist(), models_sum.tolist())
    return st
