/*
 * gymchess_b200.h -- C ABI of libgymchess_b200.so, the B200 (sm_100a) drop-in for the
 * gym-chess v2 env's step / legal-move-generation path.
 *
 * Plain pointers and sizes only (no torch / CUDA types): `stream` arguments are a
 * cudaStream_t passed as void* (NULL = default stream).  Every entry point returns
 * GCB_OK (0) or a negative GCB_E_* code; gcb_last_error() gives the text.
 *
 * What each entry point replaces in the reference (bobu36000/gym-chess):
 *   engine level  = the 4 methods of the PyO3 class `ChessEngine`, src/lib.rs:1412-1512,
 *                   batched: one call handles n independent positions;
 *   env level     = `ChessEnvV2.reset/step` and the random opponent,
 *                   gym_chess/envs/chess_v2.py:116-127, 183-294, 393-412, batched over N envs
 *                   held in device memory.
 * The reference-side bindings a maintainer would add are shown in INTEGRATION.md.
 *
 * Wire format (host or device, as stated per function):
 *   board   int8[64]  row-major, row 0 = rank 8; K1 Q2 R3 B4 N5 P6, black negative
 *                     (lib.rs:11-17, 41-50)
 *   player  int8      +1 = "WHITE", -1 = "BLACK"
 *   rights  uint8[4]  (white_king, white_queen, black_king, black_queen)_castle_is_possible
 *   action  int32     from*64+to | 4096 KSW | 4097 QSW | 4098 KSB | 4099 QSB | 4100 resign
 *                     (chess_v2.py:492-506)
 *   checks  uint8     bit0 white_king_is_checked, bit1 black_king_is_checked
 */
#ifndef GYMCHESS_B200_H
#define GYMCHESS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GCB_OK 0
#define GCB_E_CUDA (-1)    /* a CUDA runtime call failed */
#define GCB_E_ARG (-2)     /* bad argument */
#define GCB_E_NOGPU (-3)   /* no CUDA device: there is NO CPU fallback */
#define GCB_E_NOMEM (-4)

#define GCB_ACT_CASTLE_KS_WHITE 4096
#define GCB_ACT_CASTLE_QS_WHITE 4097
#define GCB_ACT_CASTLE_KS_BLACK 4098
#define GCB_ACT_CASTLE_QS_BLACK 4099
#define GCB_ACT_RESIGN 4100

/* per-env flags written by the step entry points */
#define GCB_F_INVALID 1u     /* action not in the legal list: reward -10, done unchanged (chess_v2.py:240-242) */
#define GCB_F_MATE 2u        /* side to move has no legal move and is in check (chess_v2.py:270-272, 286-288) */
#define GCB_F_REPETITION 4u  /* pre-move board seen for the 3rd time (chess_v2.py:404-407) */
#define GCB_F_CAP 8u         /* move_count > 149 early exit (chess_v2.py:252-258) */
#define GCB_F_WEDGED 16u     /* side to move has no legal move and is NOT in check: the reference never
                                terminates here (stalemate is not a terminal state; with the random bot it raises
                                TypeError).  Reported so that callers / auto-reset can act on it. */
#define GCB_F_RESET 32u      /* the env was auto-reset after this step */
#define GCB_F_BOT_PENDING 64u /* opponent 2 (external): the env owes the bot a ply when the call returns (gcb_env_bot_ply):
                                 the reply to the agent's ply of this step, a ply still owed (the step was refused), or the
                                 opening of the BLACK-agent episode an auto-reset started */

const char *gcb_last_error(void);
int gcb_version(void);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
uint64_t gcb_launch_count(void);
int gcb_device_count(void);

/* ------------------------------------------------------------------------------------------
 * Packed device-side position set (structure of arrays; 34 B per position)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    uint64_t *bb01;  /* [n][2]  piece-code bit-planes t0, t1                (16 B, 16-B aligned) */
    uint64_t *bb23;  /* [n][2]  piece-code bit-plane t2, colour plane white (16 B, 16-B aligned) */
    uint8_t *player; /* [n]     0 = white to move, 1 = black to move */
    uint8_t *rights; /* [n]     bit0 wk, bit1 wq, bit2 bk, bit3 bq */
} gcb_positions;

/* wire format (device pointers) -> packed; replaces convert_py_state, lib.rs:1246-1276 */
int gcb_pack(int n, const int8_t *d_boards, const int8_t *d_players, const uint8_t *d_rights4, gcb_positions out,
             void *stream);
/* packed -> wire format; replaces State::to_py_object, lib.rs:355-395 */
int gcb_unpack(int n, gcb_positions in, int8_t *d_boards, int8_t *d_players, uint8_t *d_rights4, void *stream);

/* ------------------------------------------------------------------------------------------
 * Engine level, device pointers
 * ------------------------------------------------------------------------------------------ */
/* ChessEngine.get_possible_moves(state, player, attack), lib.rs:1454-1480.
 * d_actions uint16[n][stride] receives the ORDERED move list (normal moves in generation order,
 * then castles); d_counts int32[n] the true count (entries beyond `stride` are dropped, so
 * count > stride signals overflow); d_incheck uint8[n] (may be NULL) whether the mover's king square is in
 * the opponent's attack map.  castles_only != 0 gives ChessEngine.get_castle_moves, lib.rs:1482-1500.
 * `stride` must be even. */
int gcb_get_possible_moves(int n, gcb_positions pos, int attack, int castles_only, uint16_t *d_actions, int stride,
                           int32_t *d_counts, uint8_t *d_incheck, void *stream);

/* ChessEngine.next_state(state, player, move), lib.rs:1422-1452: mask rights by king presence on the input
 * board, apply, recompute both check flags.  `pos.player` is the mover.  d_status int8[n]: 0 ok, 1 ok but BOTH kings
 * are in check afterwards (the reference sets a Python exception and still returns the state, lib.rs:1442-1446), -1 the from
 * square is empty (the reference panics, lib.rs:693-695), -2 bad action code; on an error (< 0) the position is copied. */
int gcb_next_state(int n, gcb_positions pos, const int32_t *d_actions, gcb_positions out, uint8_t *d_checks,
                   int32_t *d_reward, int8_t *d_status, void *stream);

/* ChessEngine.update_state(state), lib.rs:1502-1511: masked rights + both check flags */
int gcb_update_state(int n, gcb_positions pos, uint8_t *d_rights_out, uint8_t *d_checks, void *stream);

/* ------------------------------------------------------------------------------------------
 * Engine level, HOST buffers in the reference's wire format (copies + pack inside the call).
 * These are what a binding of the reference's `ChessEngine` would call.
 * ------------------------------------------------------------------------------------------ */
int gcb_host_get_possible_moves(int n, const int8_t *boards, const int8_t *players, const uint8_t *rights4, int attack,
                                int castles_only, uint16_t *actions, int stride, int32_t *counts, uint8_t *incheck);
int gcb_host_next_state(int n, const int8_t *boards, const int8_t *players, const uint8_t *rights4,
                        const int32_t *actions, int8_t *out_boards, uint8_t *out_rights4, uint8_t *out_checks,
                        int32_t *out_reward, int8_t *out_status);
int gcb_host_update_state(int n, const int8_t *boards, const uint8_t *rights4, uint8_t *out_rights4,
                          uint8_t *out_checks);

/* ------------------------------------------------------------------------------------------
 * Env level: N envs resident in device memory (ChessEnvV2, chess_v2.py:132-294)
 * ------------------------------------------------------------------------------------------ */
typedef struct gcb_env gcb_env;

typedef struct {
    int32_t num_envs;       /* N on this device */
    uint32_t env_id_offset; /* global id of local env 0 (multi-GPU shards; enters the Philox counter) */
    uint64_t seed;          /* Philox key */
    int32_t opponent;       /* 0 = "none" (self-play, one ply per step), 1 = "random" (bot replies inside step, drawn on
                               the device), 2 = "external": a callable opponent (chess_v2.py:171-179) -- the step stops
                               where the bot would move, reports GCB_F_BOT_PENDING and the reward so far, and the caller
                               supplies the bot's ply with gcb_env_bot_ply */
    int32_t agent_black;    /* player_color == "BLACK": the bot opens at reset (chess_v2.py:208-216) */
    int32_t auto_reset;     /* reset an env in the same step in which it terminates (done | cap | wedged) */
    int32_t piece_slots;    /* slots of the per-env legal set (one 64-bit target set per own piece of the side to
                               move); 0 = auto = max(16, most pieces of one colour on any initial board) */
    int32_t history_cap;    /* longest repetition window (plies since the last pawn move / capture) that is
                               tracked exactly (power of two in [8, 1024]; default 512 when 0); the per-env hash
                               table has twice as many 16-byte slots */
    int32_t moves_max;      /* 149 in the reference (chess_v2.py:141); <0 selects 149 */
    int32_t n_templates;    /* number of initial boards (0 = the default start position) */
    const int8_t *template_boards; /* HOST int8[n_templates][64]; env i starts from template (global id % n) */
    int32_t device;         /* CUDA device ordinal */
} gcb_env_config;

int gcb_env_create(const gcb_env_config *cfg, gcb_env **out);
int gcb_env_destroy(gcb_env *env);

/* ChessEnvV2.reset, chess_v2.py:183-217.  d_mask uint8[N] selects envs (NULL = all).  A reset starts a new
 * episode (episode counter + 1, enters the Philox counter). */
int gcb_env_reset(gcb_env *env, const uint8_t *d_mask, void *stream);

/* State import: a new episode of the selected envs (d_mask uint8[N], NULL = all) from arbitrary positions in the
 * reference's wire format -- what assigning `env.state = s` (the setter of chess_v2.py:315-323) and the bookkeeping of
 * reset() amount to: rights masked by king presence and both check flags (engine.update_state), the legal set of the side
 * to move, empty repetition window, done = False, step_in_episode = 0, episode counter + 1.  d_boards int8[N][64],
 * d_players int8[N] (+1/-1), d_rights4 uint8[N][4], d_move_count int32[N] (NULL = 0).  More own pieces than the env has
 * piece slots (gcb_env_config.piece_slots) are reported through the slot_overflow statistic of later steps. */
int gcb_env_import(gcb_env *env, const int8_t *d_boards, const int8_t *d_players, const uint8_t *d_rights4,
                   const int32_t *d_move_count, const uint8_t *d_mask, void *stream);

/* Per-env clone: branch games mid-episode (search rollouts, lookahead, duplicating games of a batch).  d_src_index int32[N of
 * dst] (device): for every destination row j of `dst` with 0 <= d_src_index[j] < src's N, env j of `dst` becomes env
 * i = d_src_index[j] of `src`.  Rows with a negative index are left untouched (this takes the place of a mask; fan-out is
 * repeated indices).  Unlike gcb_env_import, the clone continues the source's EPISODE, repetition window included:
 *   copied from the source: board planes, Zobrist key, meta (side to move, rights, check flags, done, castle bits, n_legal,
 *     move_count, step_in_episode, hist_len, bot_pending), count bytes, all piece slots, and the live entries of the
 *     repetition table;
 *   kept from the destination: global env id and seed (the Philox draws of a clone differ from its source's), templates
 *     (used by a later auto-reset), statistics rows (a clone is not a step: no counter moves);
 *   episode counter: the destination's own + 1, like gcb_env_import (re-cloning a root into the same row does not replay the
 *     same random words);
 *   repetition table: new generation G = the destination's generation + 1; every live source entry is written to the SAME
 *     slot of the destination's table, retagged to G, and nothing else is written (the destination's older entries are dead
 *     under G; a source with an empty window needs no table read).
 * src and dst must live on the same device and agree in the resolved piece_slots, history_cap, opponent, agent_black and
 * moves_max (GCB_E_ARG otherwise); num_envs, seed, env_id_offset, auto_reset and templates may differ.  src == dst is
 * allowed, but no selected destination row may also be the source row of a selected destination (the result is then
 * unspecified).  An index >= src's N leaves its row untouched; the CHECKED build additionally records it (and the aliasing
 * case) through gcb_debug_violations.  Enqueued on `stream`: ordering against work on `src` on other streams is the
 * caller's.  A mask output registered on dst (gcb_env_step_mask_output) is current afterwards. */
int gcb_env_clone(gcb_env *dst, const gcb_env *src, const int32_t *d_src_index, void *stream);

/* ChessEnvV2.step(action), chess_v2.py:219-294, for all N envs.  Outputs (device, any may be NULL):
 * d_reward int32[N] (the two float 0.0 literals are 0), d_done uint8[N], d_flags uint8[N] (GCB_F_*).
 * Opponent 2 (external): the step of an env that owes a bot ply is refused -- reward -10, done unchanged, GCB_F_INVALID |
 * GCB_F_BOT_PENDING, and the env's state is left as it was (step_in_episode included; only an env whose bot has no legal
 * move is reported GCB_F_WEDGED and auto-reset); the statistics count a step and an invalid action.  GCB_F_BOT_PENDING is
 * set on every output of an env that owes a ply when the call returns. */
int gcb_env_step(gcb_env *env, const int32_t *d_actions, int32_t *d_reward, uint8_t *d_done, uint8_t *d_flags,
                 void *stream);
/* The bot's ply of an env created with opponent 2 (external), for every env that owes one (after an output that reported
 * GCB_F_BOT_PENDING, or after gcb_env_reset with agent_black): d_bot_actions int32[N] is applied the way the reference applies
 * opponent_policy(env) -- player_move without a membership test (chess_v2.py:277-288, 208-216).  Outputs like gcb_env_step,
 * written only for envs that owed a ply:
 *   the reply to the agent's ply: d_reward = -(the bot's capture value) - 100 if the agent is mated (to be ADDED to the
 *     reward of the agent's half), d_done, d_flags (GCB_F_BOT_PENDING when an auto-reset started a BLACK-agent episode);
 *   White's opening of a BLACK-agent episode (owed from the reset until this call, however many steps were refused
 *     meanwhile): reward 0, done 0, flags 0 -- the reference's reset discards the opening's reward and clears done.
 * Envs that owe nothing are left alone: no state change, their output rows are not written. */
int gcb_env_bot_ply(gcb_env *env, const int32_t *d_bot_actions, int32_t *d_reward, uint8_t *d_done, uint8_t *d_flags,
                    void *stream);
/* same, but env i plays possible_actions[i][(u32[i] * n_legal[i]) >> 32] (RESIGN when it has no legal move): the uniform
 * draw of make_random_policy (chess_v2.py:116-127) with caller-provided random words */
int gcb_env_step_index(gcb_env *env, const uint32_t *d_u32, int32_t *d_reward, uint8_t *d_done, uint8_t *d_flags,
                       void *stream);
/* same, the word is drawn on the device: Philox4x32-10, counter (global env id, episode, step in episode, 0),
 * key = seed.  Runs `nsteps` consecutive steps -- up to 64 of them per kernel launch: envs are independent, so a thread
 * keeps stepping its env with the state in registers (no launch gap, no grid-wide sync); outputs are those of the LAST
 * step.  d_actions_out int32[nsteps][N] (may be NULL) records the action each env played, d_bot_out likewise the bot's
 * reply (-1 = none). */
int gcb_env_step_sampled(gcb_env *env, int nsteps, int32_t *d_reward, uint8_t *d_done, uint8_t *d_flags,
                         int32_t *d_actions_out, int32_t *d_bot_out, void *stream);

/* HOST-buffer forms (synchronous; what a binding of the reference env calls).  Page-locked buffers (cudaHostAlloc /
 * cudaHostRegister / torch pin_memory) are read and written IN PLACE by the step kernel through their device aliases --
 * one launch, no staging copy; pageable buffers are staged in up to 4 pipelined chunks.  The step is ordered after the work
 * already enqueued on `stream` (NULL = the default stream) and has finished when the call returns. */
int gcb_env_step_host(gcb_env *env, const int32_t *actions, int32_t *reward, uint8_t *done, uint8_t *flags, void *stream);
int gcb_env_step_index_host(gcb_env *env, const uint32_t *u32, int32_t *reward, uint8_t *done, uint8_t *flags,
                            void *stream);

/* Asynchronous HOST-buffer forms: page-locked buffers ONLY (GCB_E_ARG otherwise -- nothing is staged); the step is
 * enqueued on `stream` and the call returns; the outputs are valid once gcb_env_wait(env, stream) (or any other
 * synchronisation of that stream) has returned, and the input buffer may be rewritten from then on.  This is how a caller
 * keeps two or more env objects (shards of one device, gcb_env_config.env_id_offset) in flight: the device steps one
 * shard while the host consumes the other's results and prepares its actions, so the launch / completion latency of a
 * synchronous step() call is hidden. */
int gcb_env_step_host_async(gcb_env *env, const int32_t *actions, int32_t *reward, uint8_t *done, uint8_t *flags,
                            void *stream);
int gcb_env_step_index_host_async(gcb_env *env, const uint32_t *u32, int32_t *reward, uint8_t *done, uint8_t *flags,
                                  void *stream);
int gcb_env_wait(gcb_env *env, void *stream);

/* Packed 16-bit records (asynchronous, enqueued on `stream` like the device-pointer forms): 2 bytes in and 2 bytes out
 * per env instead of 4 + 6 -- host-buffer steps are bound by the bytes that cross PCIe, and with 8 GPUs by the host's
 * memory fabric.  actions16 uint16[N] (an action code is < 4101); u16 uint16[N]: word w draws like the 32-bit word
 * w << 16 of gcb_env_step_index, i.e. possible_actions[(w * n_legal) >> 16]; result16 uint16[N]: bits 0-7 the reward as
 * int8 (a step's reward is always within [-120, 100]: -10, a capture <= 10, +-100 for a mate, minus the bot's capture),
 * bits 8-14 the GCB_F_* flags (GCB_F_INVALID .. GCB_F_BOT_PENDING: flag f sits at bit 8 + log2 f), bit 15 done.  An
 * external-opponent env is stepped like with gcb_env_step, and bit 14 tells which envs owe gcb_env_bot_ply.  Each pointer may be device memory or page-locked host memory (read / written
 * in place through its device alias); results are valid after gcb_env_wait / a synchronisation of the stream. */
int gcb_env_step_packed(gcb_env *env, const uint16_t *actions16, uint16_t *result16, void *stream);
int gcb_env_step_index_packed(gcb_env *env, const uint16_t *u16, uint16_t *result16, void *stream);

/* observation / state export (device pointers, any may be NULL):
 *   d_boards int8[N][64]   -- `state["board"]`, the Box(-6,6,(8,8)) observation
 *   d_info   int32[N][16]  -- current_player(+1/-1), wk, wq, bk, bq, wchk, bchk, done, move_count, n_legal,
 *                             episode, step_in_episode, hist_len, castle bits (1 queen side | 2 king side),
 *                             bot_pending (opponent 2: a gcb_env_bot_ply is owed), 0 */
int gcb_env_export(gcb_env *env, int8_t *d_boards, int32_t *d_info, void *stream);
/* legal action mask uint8[N][4101] (possible_actions as a mask) */
int gcb_env_legal_mask(gcb_env *env, uint8_t *d_mask, void *stream);
/* the same mask as BITS: d_bits uint64[N][stride_words], stride_words >= 65; bit (a & 63) of word (a >> 6) is set iff
 * action a is in possible_actions -- word `from` (0..63) is the legal-target set of the piece standing on that square,
 * word 64 holds the castle actions 4096..4099 in bits 0..3.  520 B per env instead of 4101: the form a learner should
 * read every step (one streaming kernel, HBM-bound). */
int gcb_env_legal_bitmask(gcb_env *env, uint64_t *d_bits, int stride_words, void *stream);
/* The bit mask as an OUTPUT OF EVERY STEP CALL (what a learner reads next to the reward: possible_actions of the state the
 * step leaves behind, chess_v2.py:333-335): once a buffer is registered here, gcb_env_step / _step_index / _step_sampled /
 * the host-buffer and packed forms fill d_bits (uint64[N][stride_words], device memory, layout of gcb_env_legal_bitmask)
 * on the stream of the step: the step kernel writes the mask itself, right where it leaves the env's legal set (no second
 * kernel, no second pass over the state) -- the rows of a warp's envs are zero-filled with coalesced stores and each
 * thread scatters the at most 17 non-zero words of its env.
 * gcb_env_reset and gcb_env_import keep a registered buffer current too (the mask kernel runs behind them; gcb_env_restore does
 * not).  d_bits = NULL switches the output off.  An even stride_words (e.g. 66) lets the rows be written as 16-byte stores. */
int gcb_env_step_mask_output(gcb_env *env, uint64_t *d_bits, int stride_words);
/* ChessEnvV2.possible_actions (chess_v2.py:333-335) of every env: d_actions uint16[N][stride] receives the list in
 * the reference's order (normal moves in generation order, then castles), d_counts int32[N] (may be NULL) the true
 * count.  Like the reference's property, the list is DERIVED on access: the resident form of possible_moves is one
 * 64-bit legal-target set per own piece (gcb_env_piece_slots) and the list is a pure decode of (board, slots). */
int gcb_env_legal_actions(gcb_env *env, uint16_t *d_actions, int stride, int32_t *d_counts, void *stream);
/* zero-copy views of the resident state: slots uint64[n_slots][N] (slot r of env e at [r][e] = legal targets of the
 * r-th piece, in ascending square order, of the side to move); positions (player/rights are NULL: they live in meta) */
int gcb_env_piece_slots(gcb_env *env, uint64_t **d_slots, int32_t *n_slots);
int gcb_env_positions(gcb_env *env, gcb_positions *out);

/* Checkpoint / resume (the reference has none: its whole env state is the `state` dict + saved_boards + counters).  A
 * snapshot is the concatenation of the resident arrays (positions, meta, keys, generations, legal set, repetition
 * tables, statistics rows) in ONE device buffer of gcb_env_snapshot_bytes() bytes plus the launch counter `tick`; restoring it into an env
 * created with the same configuration resumes bit-identically (same Philox counters). */
int gcb_env_snapshot_bytes(gcb_env *env, uint64_t *bytes);
int gcb_env_snapshot(gcb_env *env, void *d_buf, uint64_t *tick, void *stream);
int gcb_env_restore(gcb_env *env, const void *d_buf, uint64_t tick, void *stream);

/* episode statistics accumulated on the device since the last gcb_env_stats_reset:
 * out uint64[16] = steps, plies, episodes, mates, repetitions, caps, wedged, invalid, reward_sum (two's complement
 * int64), legal_sum, in_check, hist_overflow, slot_overflow, hist_scanned (repetition-table probes beyond
 * the first one of a ply), hist_window (sum over plies of the repetition window length), 0.   Synchronises the stream. */
int gcb_env_stats(gcb_env *env, uint64_t *out16, void *stream);
int gcb_env_stats_reset(gcb_env *env, void *stream);
/* device pointer to the 16 counters (for an NCCL reduce by the caller); the totals are brought up to date by a small
 * reduction kernel enqueued on `stream` */
int gcb_env_stats_ptr(gcb_env *env, uint64_t **d_stats, void *stream);

/* ------------------------------------------------------------------------------------------
 * Memory-safety net (test support; compute-sanitizer is not available on the GPU pool this was built on).
 * (1) Guard regions: with GCB_GUARD_BYTES=<n> in the environment when gcb_env_create runs, every device array of the
 *     env sits between two regions of n (rounded up to 256) bytes filled with 0xA5; gcb_env_check_guards counts the guard
 *     bytes that no longer hold the pattern (0 = no kernel wrote outside an array).  GCB_E_ARG for an env without guards.
 * (2) The CHECKED build of the library (libgymchess_b200_checked.so, -DGCB_CHECKED) verifies the index of every indexed
 *     global access of the env kernels against the extent of its array; gcb_debug_violations returns the bit set of
 *     violated checks (always 0 in the product build, gcb_build_is_checked() == 0) and optionally clears it.
 * ------------------------------------------------------------------------------------------ */
int gcb_env_check_guards(gcb_env *env, uint64_t *n_bad_bytes);
int gcb_debug_violations(uint64_t *out, int reset);
int gcb_build_is_checked(void);

#ifdef __cplusplus
}
#endif
#endif
