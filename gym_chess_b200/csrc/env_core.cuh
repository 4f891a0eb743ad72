// env_core.cuh -- per-env step / reset logic of the batched env (ChessEnvV2, chess_v2.py:183-294,
// 393-412) over the resident structure-of-arrays state.  One call of env_step_one() advances ONE
// env by one `step()`; the kernels in gcb_kernels.cu run it with one thread per env.
//
// Layout in HBM (structure of arrays):
//   bb01[N]  ulonglong2 {t0,t1}       16 B   piece-code bit-planes
//   bb23[N]  ulonglong2 {t2,white}    16 B
//   meta[N]  u64                       8 B   stm | rights | check flags | done | castle bits | n_legal |
//                                            move_count | step_in_episode | hist_len
//   zkey[N]  u64                       8 B   Zobrist key of the current board (board only)
//   gen[N]   u32                       4 B   generation of the repetition window (bumped by every irreversible ply and
//                                            every new episode): table entries of older generations are dead
//   episode[N] u32                     4 B
//   cnt[N]   ulonglong2               16 B   byte r = number of legal targets of the r-th own piece (r < 16): the
//                                            uniform draw over the ordered list finds its piece from this one record
//                                            and then reads a single slot
//   tgt[S][N] u64                            the cached legal set = ChessEnvV2.possible_moves: slot r = legal
//                                            targets of the r-th own piece of the side to move (ascending square
//                                            order = the reference's scan order); castles are two bits of meta.
//                                            The ordered action list is a pure decode of (board, slots).
//   rep[N][2H] ulonglong2                    the Zobrist-hash history of the repetition window as an open-addressing
//                                            table: {key, generation << 2 | count}; slot = key bits, linear probing;
//                                            one 16-byte entry read and written per ply
#pragma once
#include <math.h>

#include "chess_core.cuh"

#if !defined(__CUDACC__)
struct ulonglong2 {
    u64 x, y;
};
static inline ulonglong2 make_ulonglong2(u64 x, u64 y) {
    ulonglong2 r = {x, y};
    return r;
}
#endif

// Memory-safety net for a pool without compute-sanitizer (DESIGN.md section 3.8): the CHECKED build (-DGCB_CHECKED,
// libgymchess_b200_checked.so) verifies the index of every indexed global access of the env kernels against the extent of
// its array and records violations here; gcb_debug_violations() reads the word.  The product build compiles the checks out.
#if defined(__CUDACC__)
__device__ unsigned long long g_violations = 0ULL;
#endif
#if defined(GCB_CHECKED) && defined(__CUDA_ARCH__)
#define GCB_CHK(cond, code)                                                   \
    do {                                                                      \
        if (!(cond)) atomicOr(&g_violations, 1ULL << (code));                 \
    } while (0)
#else
#define GCB_CHK(cond, code) \
    do {                    \
    } while (0)
#endif
// CHK_CLONE_INDEX: a clone index >= the source's env count (the row is left alone in both builds); CHK_CLONE_ALIAS: a clone
// destination row that is also the source row of some destination of the same call
// CHK_POLICY_INDEX: a policy sample (gcb_env_sample_policy) that would read a logit column >= 4101 or an env row >= N
// CHK_ENCODE_INDEX: an encode (gcb_env_encode) that would read an env row >= N or write a plane element beyond [N][19][64]
enum { CHK_STAT_ROW = 0, CHK_ENV_INDEX = 1, CHK_SLOT_INDEX = 2, CHK_REP_INDEX = 3, CHK_IO_INDEX = 4, CHK_LIST_INDEX = 5,
       CHK_CLONE_INDEX = 6, CHK_CLONE_ALIAS = 7, CHK_POLICY_INDEX = 8, CHK_ENCODE_INDEX = 9 };

// The resident state is touched once per step: stream it past L1 (ld.global.cs / st.global.cs, evict-first) so that
// the geometry tables the generation hammers stay L1-resident.
#if defined(__CUDA_ARCH__)
#define GCB_LDS(p) __ldcs(p)
#define GCB_STS(p, v) __stcs((p), (v))
#else
#define GCB_LDS(p) (*(p))
#define GCB_STS(p, v) (*(p) = (v))
#endif

// per-env flags (mirrors include/gymchess_b200.h GCB_F_*)
#define EF_INVALID 1u
#define EF_MATE 2u
#define EF_REPETITION 4u
#define EF_CAP 8u
#define EF_WEDGED 16u
#define EF_RESET 32u
#define EF_BOT_PENDING 64u

// ordered move list -> global memory, two 16-bit entries per 32-bit store
struct ListWriter {
    uint16_t* out;
    int n, cap;
    u32 pend;
    GCB_HD ListWriter(uint16_t* o, int c) : out(o), n(0), cap(c), pend(0) {}
    GCB_HD void push(int action) {
        if (n & 1) {
            if (n < cap) *reinterpret_cast<u32*>(out + n - 1) = pend | ((u32)action << 16);
        } else {
            pend = (u32)action;
        }
        n++;
    }
    GCB_HD void flush() {
        if ((n & 1) && n <= cap) out[n - 1] = (uint16_t)pend;
    }
};

// meta word: bit 0 stm, 1-4 rights, 5-6 check flags, 7 done, 8-9 castle (queen side, king side), 10-21 n_legal,
// 22-37 move_count, 38-53 step_in_episode, 54-62 hist_len (saturates at 511; only its being zero matters, the rest is
// statistics), 63 bot_pending (opponent "external": the caller owes this env the bot's ply, gcb_env_bot_ply)
#define M_RIGHTS_SHIFT 1
#define M_CASTLE_SHIFT 8
#define M_NLEGAL_SHIFT 10
#define M_MOVECOUNT_SHIFT 22
#define M_STEP_SHIFT 38
#define M_HIST_SHIFT 54

enum { ST_STEPS = 0, ST_PLIES, ST_EPISODES, ST_MATES, ST_REPS, ST_CAPS, ST_WEDGED, ST_INVALID, ST_REWARD, ST_LEGAL,
       ST_INCHECK, ST_HISTOVF, ST_SLOTOVF, ST_HISTSCAN, ST_WINDOW, ST_USED, ST_COUNT = 16 };

struct EnvView {
    ulonglong2* bb01;
    ulonglong2* bb23;
    u64* meta;
    u64* zkey;
    u32* gen;         // [N] generation of the current repetition window
    ulonglong2* rep;  // [N][2H] {key, generation << 2 | count}: the window's keys, open addressing (H = history_cap; hist_mask = 2H - 1)
    u32* episode;
    ulonglong2* cnt;
    u64* tgt;
    const ulonglong2* t_bb01;
    const ulonglong2* t_bb23;
    const u64* t_meta;
    const u64* t_zkey;
    const u64* t_tgt;
    const ulonglong2* t_cnt;
    const u64* zob;
    u64* stats;      // [ST_COUNT] totals (written by the reduction of stat_rows)
    u64* stat_rows;  // [ceil(N/32)][ST_COUNT] per-warp accumulators: no atomics, no block barrier in the step kernel
    u64 seed;
    int N, slots, hist_mask, n_templates, stat_nrows;
    u32 env_offset;
    int moves_max, opponent, agent_black, auto_reset, pps;
};

struct EnvRegs {
    Board b;
    u64 zk, cnt_lo, cnt_hi;
    u32 rights, chk, castle;  // chk bit0 white checked, bit1 black checked; castle bit0 queen side, bit1 king side
    int stm_black, done, n_legal, move_count, step, hist_len, pending;
    u32 gen;
};

GCB_HD void unpack_meta(u64 m, EnvRegs& s) {
    s.stm_black = (int)(m & 1);
    s.rights = (u32)(m >> M_RIGHTS_SHIFT) & 15u;
    s.chk = (u32)(m >> 5) & 3u;
    s.done = (int)(m >> 7) & 1;
    s.castle = (u32)(m >> M_CASTLE_SHIFT) & 3u;
    s.n_legal = (int)(m >> M_NLEGAL_SHIFT) & 0xFFF;
    s.move_count = (int)(m >> M_MOVECOUNT_SHIFT) & 0xFFFF;
    s.step = (int)(m >> M_STEP_SHIFT) & 0xFFFF;
    s.hist_len = (int)(m >> M_HIST_SHIFT) & 0x1FF;
    s.pending = (int)(m >> 63);
}
GCB_HD u64 pack_meta(const EnvRegs& s) {
    return (u64)(s.stm_black & 1) | ((u64)(s.rights & 15u) << M_RIGHTS_SHIFT) | ((u64)(s.chk & 3u) << 5) |
           ((u64)(s.done & 1) << 7) | ((u64)(s.castle & 3u) << M_CASTLE_SHIFT) | ((u64)(s.n_legal & 0xFFF) << M_NLEGAL_SHIFT) |
           ((u64)(s.move_count & 0xFFFF) << M_MOVECOUNT_SHIFT) | ((u64)(s.step & 0xFFFF) << M_STEP_SHIFT) |
           ((u64)(s.hist_len & 0x1FF) << M_HIST_SHIFT) | ((u64)(s.pending & 1) << 63);
}

GCB_HD bool stm_checked(const EnvRegs& s) { return (s.chk >> s.stm_black) & 1u; }
GCB_HD u64 stm_pieces(const EnvRegs& s) { return s.stm_black ? (bb_occ(s.b) & ~s.b.w) : s.b.w; }
GCB_HD u32 castle_word(const EnvRegs& s) {  // castle bits of meta -> bit (action - 4096)
    u32 c = 0;
    if (s.castle & 1u) c |= 1u << (castle_action(!s.stm_black, 0) - 4096);
    if (s.castle & 2u) c |= 1u << (castle_action(!s.stm_black, 1) - 4096);
    return c;
}

// piece slots of env e in the resident array (slot r of env e at tgt[r*N + e]: coalesced when a warp reads slot r).
// The per-piece target counts of the first 16 slots go to 16 bytes of scratch (shared memory in the kernel: one
// byte store per piece instead of a 128-bit shift-and-add; read back as one 16-byte record).
struct alignas(16) CountBytes {
    uint8_t c[16];
};
// where the piece slots of one env live: slot r at base[r * stride].  Resident form: base = tgt + e, stride = N
// (streamed past L1); inside a multi-step launch: the thread's column of a shared-memory tile (plain accesses).
struct SlotRef {
    u64* base;
    unsigned stride;  // slots * stride < 2^31 (checked at create): 32-bit index arithmetic
    int slots;
    bool plain;
};
GCB_HD SlotRef resident_slots(const EnvView& v, int e) {
    SlotRef r = {v.tgt + e, (unsigned)v.N, v.slots, false};
    return r;
}
struct TgtSink {
    u64* base;
    unsigned N;
    int slots, dropped, extra;  // extra = targets of pieces beyond the 16 counted slots
    bool plain;
    uint8_t* cb;
    GCB_HD TgtSink(const SlotRef& sr, CountBytes* scratch)
        : base(sr.base), N(sr.stride), slots(sr.slots), dropped(0), extra(0), plain(sr.plain), cb(scratch ? scratch->c : nullptr) {
        if (scratch) {
            u64* z = reinterpret_cast<u64*>(scratch);
            z[0] = 0, z[1] = 0;
        }
    }
    GCB_HD void put(int r, u64 t) {
        if (r < slots) st(r, t);
        else dropped++;
        const int c = gcb_popc(t);
        if (r < 16) cb[r] = (uint8_t)c;
        else extra += c;
    }
    GCB_HD void st(int r, u64 t) {
        GCB_CHK((unsigned)r < (unsigned)slots, CHK_SLOT_INDEX);
        if (plain) base[(unsigned)r * N] = t;
        else GCB_STS(&base[(unsigned)r * N], t);
    }
    GCB_HD u64 get(int r) const {
        if (r >= slots) return 0ULL;
        return plain ? base[(unsigned)r * N] : GCB_LDS(&base[(unsigned)r * N]);
    }
    GCB_HD void replace(int r, u64 told, u64 tnew) {  // tnew is a subset of told
        if (r < slots) st(r, tnew);
        const int c = gcb_popc(tnew);
        if (r < 16) cb[r] = (uint8_t)c;
        else extra -= gcb_popc(told) - c;
    }
    GCB_HD u64 count_lo() const { return reinterpret_cast<const u64*>(cb)[0]; }
    GCB_HD u64 count_hi() const { return reinterpret_cast<const u64*>(cb)[1]; }
    GCB_HD int total() const {  // sum of the 16 bytes + extra
        u64 a = count_lo(), b = count_hi();
        a = (a & 0x00FF00FF00FF00FFULL) + ((a >> 8) & 0x00FF00FF00FF00FFULL);
        b = (b & 0x00FF00FF00FF00FFULL) + ((b >> 8) & 0x00FF00FF00FF00FFULL);
        a += b;
        a += a >> 32;
        a += a >> 16;
        return (int)(a & 0xFFFF) + extra;
    }
};

// The same sink for a thread that KNOWS its env has at most 16 pieces of either colour and 16 plain (shared-memory)
// slots: no bounds tests, no overflow bookkeeping (multi-step launches check this once per launch).
struct TgtSinkFast {
    u64* base;
    unsigned N;
    int dropped;
    uint8_t* cb;
    GCB_HD TgtSinkFast(const SlotRef& sr, CountBytes* scratch) : base(sr.base), N(sr.stride), dropped(0), cb(scratch->c) {
        u64* z = reinterpret_cast<u64*>(scratch);
        z[0] = 0, z[1] = 0;
    }
    GCB_HD void put(int r, u64 t) {
        GCB_CHK((unsigned)r < 16u, CHK_SLOT_INDEX);
        base[(unsigned)r * N] = t;
        cb[r] = (uint8_t)gcb_popc(t);
    }
    GCB_HD u64 get(int r) const { return base[(unsigned)r * N]; }
    GCB_HD void replace(int r, u64, u64 tnew) {
        GCB_CHK((unsigned)r < 16u, CHK_SLOT_INDEX);
        base[(unsigned)r * N] = tnew;
        cb[r] = (uint8_t)gcb_popc(tnew);
    }
    GCB_HD u64 count_lo() const { return reinterpret_cast<const u64*>(cb)[0]; }
    GCB_HD u64 count_hi() const { return reinterpret_cast<const u64*>(cb)[1]; }
    GCB_HD int total() const {
        u64 a = count_lo(), b = count_hi();
        a = (a & 0x00FF00FF00FF00FFULL) + ((a >> 8) & 0x00FF00FF00FF00FFULL);
        b = (b & 0x00FF00FF00FF00FFULL) + ((b >> 8) & 0x00FF00FF00FF00FFULL);
        a += b;
        a += a >> 32;
        a += a >> 16;
        return (int)(a & 0xFFFF);
    }
};

// per-thread statistics of one step: the small counters live as bit fields of ONE register (fewer live registers in
// the step kernel), the wide ones in four ints
struct StepStats {
    // f: the three counters EVERY step touches as 7/8-bit fields (bits 0-6 steps, 7-14 plies, 15-21 in_check: their sum
    // over the 32 lanes of a warp fits the field, so one warp reduction of the masked word adds all three), then the rare
    // events: bit 22 episodes, 23 mates, 24 repetitions, 25 caps, 26 wedged, 27 invalid, 28-29 hist_overflow, 30-31
    // slot_overflow (the kernel looks at them only when some lane of the warp has one)
    u32 f;
    int reward, legal, scan, window;
    bool wrote_slots;  // (not a statistic) the step rewrote the env's piece slots: a ply was generated or a reset copied its template
    GCB_HD void clear() { f = 0, reward = 0, legal = 0, scan = 0, window = 0, wrote_slots = false; }
    GCB_HD int get(int k) const {
        switch (k) {
        case ST_STEPS: return (int)(f & 127u);
        case ST_PLIES: return (int)((f >> 7) & 255u);
        case ST_EPISODES: return (int)((f >> 22) & 1u);
        case ST_MATES: return (int)((f >> 23) & 1u);
        case ST_REPS: return (int)((f >> 24) & 1u);
        case ST_CAPS: return (int)((f >> 25) & 1u);
        case ST_WEDGED: return (int)((f >> 26) & 1u);
        case ST_INVALID: return (int)((f >> 27) & 1u);
        case ST_REWARD: return reward;
        case ST_LEGAL: return legal;
        case ST_INCHECK: return (int)((f >> 15) & 127u);
        case ST_HISTOVF: return (int)((f >> 28) & 3u);
        case ST_SLOTOVF: return (int)((f >> 30) & 3u);
        case ST_HISTSCAN: return scan;
        default: return window;
        }
    }
};
#define SF_STEPS 1u
#define SF_PLIES (1u << 7)
#define SF_INCHECK (1u << 15)
#define SF_HOT_MASK 0x3FFFFFu
#define SF_RARE_SHIFT 22
#define SF_EPISODES (1u << 22)
#define SF_MATES (1u << 23)
#define SF_REPS (1u << 24)
#define SF_CAPS (1u << 25)
#define SF_WEDGED (1u << 26)
#define SF_INVALID (1u << 27)
#define SF_HISTOVF (1u << 28)
#define SF_SLOTOVF (1u << 30)

// Repetition table (the Zobrist-hash history of chess_v2.py:404-407's saved_boards, restricted to the window since the
// last pawn move / capture: an older board cannot recur).  Open addressing over H = history_cap slots of 16 bytes per env,
// slot = bits of the key, linear probing.  An entry is alive iff its generation is the env's current one: an irreversible
// ply or a new episode bumps the generation and thereby empties the table without touching it.  One ply = one probe
// sequence (almost always a single 16-byte load) + one store; nothing is read when the window is empty and nothing is
// written by an irreversible ply.  Returns how often `key` has now occurred in the window, this ply included.
// The table has 2 * history_cap slots, so while the window fits history_cap the load factor stays <= 1/2 and a probe
// sequence of 128 slots cannot be exhausted in practice (expected length 1.5 - 2.5).
#define GCB_REP_MAX_PROBES 128
#ifndef GCB_REP_PREFETCH
#define GCB_REP_PREFETCH 1
#endif
// The entry a ply will probe first is known as soon as the pre-move key is: ask L2 for its line at the START of the step, so
// that the DRAM latency of this one randomly addressed access runs under the action pick instead of stalling the ply.
GCB_HD void rep_prefetch(const EnvView& v, int e, const EnvRegs& s) {
#if defined(__CUDA_ARCH__) && GCB_REP_PREFETCH
    if (s.hist_len != 0) {
        const unsigned mask = (unsigned)v.hist_mask;
        const ulonglong2* p = v.rep + (size_t)e * ((size_t)mask + 1) + ((unsigned)(hist_key(s.zk) >> 24) & mask);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
    }
#else
    (void)v, (void)e, (void)s;
#endif
}
GCB_HD int rep_lookup_insert(const EnvView& v, int e, const EnvRegs& s, u64 key, bool insert, StepStats& st) {
    const unsigned mask = (unsigned)v.hist_mask;
    unsigned i = (unsigned)(key >> 24) & mask;
    const u64 live_tag = (u64)s.gen << 2;
    // env-major: the H entries of an env are contiguous (16 * H bytes), so the 32 envs of a warp touch one small span
    ulonglong2* const tab = v.rep + (size_t)e * ((size_t)mask + 1);
    GCB_CHK((unsigned)e < (unsigned)v.N && i <= mask, CHK_REP_INDEX);
    if (s.hist_len == 0) {  // empty window: every entry is dead, the first slot is free
        if (insert) GCB_STS(&tab[i], make_ulonglong2(key, live_tag | 1ULL));
        return 1;
    }
    const unsigned home = i;
    for (unsigned probes = 0; probes <= mask && probes < GCB_REP_MAX_PROBES; probes++, i = (i + 1) & mask) {
        ulonglong2* const p = &tab[i];
        const ulonglong2 en = GCB_LDS(p);
        const bool alive = (en.y >> 2) == (u64)s.gen && (en.y & 3ULL) != 0;
        if (!alive) {
            if (insert) GCB_STS(p, make_ulonglong2(key, live_tag | 1ULL));
            return 1;
        }
        if (en.x == key) {
            const u64 c = (en.y & 3ULL) < 3ULL ? (en.y & 3ULL) + 1ULL : 3ULL;
            if (insert) GCB_STS(p, make_ulonglong2(key, live_tag | c));
            return (int)c;
        }
        st.scan++;  // a further probe
    }
    // The window has outgrown the table (only an uncapped BLACK-agent episode can get here): the key replaces whatever
    // sits in its home slot -- replacing a live entry by a live entry keeps every probe chain intact -- so the most recent
    // boards, the likely ones to recur, stay findable; the displaced board's later repetition can be missed.
    st.f += SF_HISTOVF;
    if (insert) GCB_STS(&tab[home], make_ulonglong2(key, live_tag | 1ULL));
    return 1;
}

#ifndef GCB_ONE_PICK_SITE  // bot kernels: every sampled pick of a step (agent, bot reply, bot opening) through one code site
#define GCB_ONE_PICK_SITE 1
#endif
#ifndef GCB_SWAR_PICK
#define GCB_SWAR_PICK 1
#endif
// per byte: 0x80 where x <= y (unsigned bytes), else 0
GCB_HD u64 swar_le_u8(u64 x, u64 y) {
    const u64 H = 0x8080808080808080ULL;
    const u64 t = (y | H) - (x & ~H);  // per byte (y & 127) + 128 - (x & 127): no borrow between bytes, top bit = low 7 bits of x <= those of y
    return ((~x & y) | (~(x ^ y) & t)) & H;
}

// The action `possible_moves[idx]` of the reference-ordered list, decoded from the slots (chess_v2.py:116-127:
// the uniform draw indexes the ORDERED list).  idx < n_legal.
template <bool ROLLED = true>
GCB_HD int action_at(const SlotRef& sr, const EnvRegs& s, int idx) {
    // which piece: prefix scan over the 16 count bytes (registers only); pieces beyond 16 (only on crafted initial
    // boards) by reading their slots
    int acc = 0, hit_r = -1, hit_idx = 0;
#if GCB_SWAR_PICK
    if (s.n_legal <= 255) {
        // all 16 prefix sums at once: byte k of (cnt * 0x0101..01) = c0 + ... + ck (no byte overflows: the total is <= 255);
        // the piece is the number of inclusive prefix sums <= idx (they are non-decreasing); branch-free, no unrolled scan
        const u64 K = 0x0101010101010101ULL;
        const u64 p_lo = s.cnt_lo * K, p_hi = (s.cnt_hi + (p_lo >> 56)) * K;
        const u64 I = (u64)(u32)idx * K;
        const int r = gcb_popc(swar_le_u8(p_lo, I)) + gcb_popc(swar_le_u8(p_hi, I));
        acc = (int)(p_hi >> 56);
        if (r < 16) {
            const u64 q = r < 8 ? (p_lo << 8) : ((p_hi << 8) | (p_lo >> 56));  // exclusive prefix sums
            hit_r = r, hit_idx = idx - (int)((q >> (8 * (r & 7))) & 0xFF);
        }
    } else
#endif
    {
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
        for (int r = 0; r < 16; r++) {
            const int c = (int)(((r < 8 ? s.cnt_lo : s.cnt_hi) >> (8 * (r & 7))) & 0xFF);
            if (hit_r < 0 && idx - acc < c) hit_r = r, hit_idx = idx - acc;
            acc += c;
        }
    }
    TgtSink slots(sr, nullptr);
    u64 own = stm_pieces(s);
    if (sr.slots > 16 && hit_r < 0) {
        const int np = gcb_popc(own);
        for (int r = 16; r < np && hit_r < 0; r++) {
            const int c = gcb_popc(slots.get(r));
            if (idx - acc < c) hit_r = r, hit_idx = idx - acc;
            else acc += c;
        }
    }
    if (hit_r >= 0) {
        const u64 T = slots.get(hit_r);  // the one slot this draw needs
        const int sq = gcb_select64(own, hit_r);
        return sq * 64 + nth_target<ROLLED>(piece_code(s.b, sq), !s.stm_black, sq, T, hit_idx);
    }
    // castles come last, queen side first (lib.rs:1473-1479, 992, 1011)
    const int king_side = (s.castle & 1u) ? (idx - acc != 0) : 1;
    return castle_action(!s.stm_black, king_side);
}

// action in possible_actions ? (chess_v2.py:240)
GCB_HD bool action_is_legal(const SlotRef& sr, const EnvRegs& s, int action) {
    if (action < 0) return false;
    if (action < 4096) {
        const int from = action >> 6, to = action & 63;
        const u64 own = stm_pieces(s), fbit = 1ULL << from;
        if (!(own & fbit)) return false;
        TgtSink slots(sr, nullptr);
        return (slots.get(gcb_popc(own & (fbit - 1))) >> to) & 1ULL;
    }
    if (action == castle_action(!s.stm_black, 0)) return s.castle & 1u;
    if (action == castle_action(!s.stm_black, 1)) return (s.castle >> 1) & 1u;
    return false;
}



template <bool FAST> struct SinkOf { typedef TgtSink type; };
template <> struct SinkOf<true> { typedef TgtSinkFast type; };

// One ply = player_move (chess_v2.py:393-412: engine.next_state + repetition count on the PRE-move
// board) + the state setter (315-323) + switch_player (296-299) + get_possible_moves for the new
// side to move (573-582).  apply=false only switches the side and regenerates (BLACK-agent reset
// when White has no move).  Returns the ply reward.
template <bool FAST = false, class G>
GCB_HD int ply_and_movegen(const EnvView& v, int e, EnvRegs& s, int action, bool apply, bool* rep,
                           StepStats& st, CountBytes* scratch, const SlotRef& sr, const G& geo) {
    int r = 0;
    *rep = false;
    if (apply) {
        const u64 key = hist_key(s.zk);  // the board BEFORE the move (chess_v2.py:404-407)
        u32 rights = mask_rights(s.b, s.rights);  // engine entry masks by the INPUT board (Q21)
        int status;
        bool irr;
        r = apply_action(s.b, rights, !s.stm_black, action, &status, &irr, &s.zk, v.zob);
        s.rights = rights;
        st.window += s.hist_len;
        // saved_boards[key] += 1; done when it reaches 3.  An irreversible ply only looks the key up: its window dies with it.
        *rep = rep_lookup_insert(v, e, s, key, !irr, st) >= 3;
        if (irr) {
            s.hist_len = 0, s.gen++;  // the window restarts empty
        } else {
            if (s.hist_len < 0x1FF) s.hist_len++;  // (9-bit field of meta; statistics only)
        }
    }
    s.stm_black ^= 1;
    GenCtx g;
    gen_prepare(s.b, !s.stm_black, g, geo);
    typename SinkOf<FAST>::type sink(sr, scratch);
    gen_targets(s.b, g, g.own, sink, geo);
    st.wrote_slots = true;
    const int n = sink.total();
    if (sink.dropped) st.f += SF_SLOTOVF;
    s.cnt_lo = sink.count_lo(), s.cnt_hi = sink.count_hi();
    s.castle = gen_castles(s.b, g, mask_rights(s.b, s.rights));
    s.n_legal = n + (int)(s.castle & 1u) + (int)(s.castle >> 1);
    // both check flags (update_state, lib.rs:1386-1393): the side to move from the attackers of its king
    // square, the side that just moved from the attack map the generation accumulated
    u32 chk = g.in_check ? (1u << s.stm_black) : 0u;
    const u64 mk = bb_kings(s.b) & g.enemy;
    if (mk && ((g.satt >> ref_king_square(mk)) & 1ULL)) chk |= 1u << (s.stm_black ^ 1);
    s.chk = chk;
    return r;
}

enum { MODE_ACTION = 0, MODE_INDEX = 1, MODE_SAMPLED = 2, MODE_RESET = 3, MODE_BOTPLY = 4 };
enum { PH_AGENT = 0, PH_BOT = 1, PH_FINAL = 2, PH_RESETBOT = 3, PH_END = 4 };

struct StepIO {
    const void* in;      // MODE_ACTION: int32 actions; MODE_INDEX: u32 words; MODE_RESET: uint8 mask or NULL
    int32_t* reward;     // any output may be NULL
    uint8_t* done;
    uint8_t* flags;
    int32_t* act_out;
    int32_t* bot_out;
    u64 tick;            // launch counter (kept for the snapshot ABI; the repetition table needs no clock)
    int ep_inc;
    int e_begin, e_end;  // env range of this launch (host-buffer steps are pipelined in chunks)
    int nsteps;          // MODE_SAMPLED: consecutive steps run by ONE launch (envs are independent: no grid-wide sync needed)
    // packed 16-bit records (host-buffer steps are bound by the bytes that cross PCIe): in16 != 0 -> `in` holds uint16
    // actions / uint16 random words (a word w draws like the 32-bit word w << 16); packed != NULL -> one uint16 result
    // per env: bits 0-7 reward (int8; a reward is always within [-120, 100]), bits 8-14 flags, bit 15 done
    uint16_t* packed = nullptr;
    int in16 = 0;
    // learner-facing output of the step itself: possible_actions of the state the step leaves behind as the 65-word bit
    // mask (uint64[N][bits_stride]); NULL = off
    u64* bits_out = nullptr;
    int bits_stride = 0;
};
// the step's input of env e (MODE_ACTION: the action; MODE_INDEX: the caller's random word as a 32-bit word; MODE_BOTPLY: the
// bot's action): loaded FIRST, together with the state, so that its latency (it may sit in page-locked host memory, read
// through PCIe) is not paid where it is used
template <int MODE>
GCB_HD u32 step_input(const StepIO& io, int e) {
    if (MODE == MODE_ACTION) return io.in16 ? (u32)reinterpret_cast<const uint16_t*>(io.in)[e] : (u32)reinterpret_cast<const int32_t*>(io.in)[e];
    if (MODE == MODE_INDEX) return io.in16 ? (u32)reinterpret_cast<const uint16_t*>(io.in)[e] << 16 : reinterpret_cast<const u32*>(io.in)[e];
    if (MODE == MODE_BOTPLY) return (u32)reinterpret_cast<const int32_t*>(io.in)[e];
    return 0u;
}
GCB_HD uint16_t pack_result(int reward, bool done, u32 flags) {
    return (uint16_t)((u32)(reward & 0xFF) | ((flags & 127u) << 8) | (done ? 0x8000u : 0u));
}

// resident state of env e <-> registers
GCB_HD void env_load(const EnvView& v, int e, EnvRegs& s, u32& ep) {
    GCB_CHK((unsigned)e < (unsigned)v.N, CHK_ENV_INDEX);
    ulonglong2 a = GCB_LDS(&v.bb01[e]), c = GCB_LDS(&v.bb23[e]);
    s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
    ulonglong2 ct = GCB_LDS(&v.cnt[e]);
    s.cnt_lo = ct.x, s.cnt_hi = ct.y;
    unpack_meta(GCB_LDS(&v.meta[e]), s);
    s.zk = GCB_LDS(&v.zkey[e]);
    ep = GCB_LDS(&v.episode[e]);
    s.gen = GCB_LDS(&v.gen[e]);
}
GCB_HD void env_store(const EnvView& v, int e, const EnvRegs& s, u32 ep) {
    GCB_CHK((unsigned)e < (unsigned)v.N, CHK_ENV_INDEX);
    GCB_STS(&v.bb01[e], make_ulonglong2(s.b.t0, s.b.t1));
    GCB_STS(&v.bb23[e], make_ulonglong2(s.b.t2, s.b.w));
    GCB_STS(&v.cnt[e], make_ulonglong2(s.cnt_lo, s.cnt_hi));
    GCB_STS(&v.meta[e], pack_meta(s));
    GCB_STS(&v.zkey[e], s.zk);
    GCB_STS(&v.episode[e], ep);
    GCB_STS(&v.gen[e], s.gen);
}

// chess_v2.py:219-294 for env `e` (plus auto-reset and the episode statistics of this step), state in registers
// SELFPLAY = true: the caller guarantees opponent "none" (one ply per step, no bot, WHITE agent) -- the bot's branches
// are compiled out of the self-play kernel.
// MULTI = true: the step runs inside a multi-step launch (warm caches, a hot loop that has to fit the instruction cache):
// rolled direction scan in the ordered pick, L2 prefetch of the ply's repetition entry at the start of the step.  Single-step
// launches start with cold caches every time and run back to back over an L2-resident state that a prefetch would push out.
template <int MODE, bool SELFPLAY = false, bool FAST = false, bool MULTI = false, class G>
GCB_HD void env_step_regs(const EnvView& v, const StepIO& io, int e, EnvRegs& s, u32& ep, StepStats& st, CountBytes* scratch,
                          const SlotRef& sr, const SlotRef& pick_sr, const G& geo, const u32 input) {
    // sr: where the generation writes the piece slots (and later picks of the same step read them); pick_sr: where the
    // legal set of the state the step STARTS from lives (the same place, except in single-step tile kernels)
    // opponent: 0 none, 1 random (the bot draws on the device), 2 external (the step stops where the bot would move and
    // the caller supplies the bot's ply through MODE_BOTPLY: callable opponents, chess_v2.py:171-179)
    const bool v_bot = SELFPLAY ? false : v.opponent != 0, v_ext = SELFPLAY ? false : v.opponent == 2;
    const bool v_agent_black = SELFPLAY ? false : v.agent_black != 0;
    const u32 genv = v.env_offset + (u32)e;
    int action = ACT_RESIGN, bot_action = -1, R = 0, phase;
    u32 fl = 0;
    bool d_out = false, agent_ply = false, owe_bot = false, agent_draw = false;
    const int n0 = s.n_legal;
    const bool was_done = s.done, capped = s.move_count > v.moves_max;
    const u32 step_idx = (u32)s.step;
    if (MODE == MODE_RESET) {
        phase = PH_FINAL;
    } else if (MODE == MODE_BOTPLY) {
        // the bot's ply of an "external" opponent, applied like the reference applies opponent_policy(env): no
        // membership test (chess_v2.py:277-283, 208-213)
        if (!s.pending) return;  // nothing owed: the env is left alone, no outputs
        s.pending = 0;
        action = bot_action = (int)input;
        agent_ply = true;
        // the opening after a reset is owed at step 0 and only there: a step refused because a ply is owed does not advance
        // step_in_episode, a played step does before it can leave a reply owed (a state import starts at 0 but owes nothing)
        phase = (s.step == 0 && v_agent_black) ? PH_RESETBOT : PH_BOT;
    } else {
        bool valid = false;
        if (MULTI) rep_prefetch(v, e, s);
        if (MODE == MODE_ACTION) {
            action = (int)input;
            valid = action_is_legal(pick_sr, s, action);  // action in possible_actions
        } else {
            if (!SELFPLAY && GCB_ONE_PICK_SITE) {
                // (bot kernels: the agent's draw also goes through the one pick site at the top of the phase loop)
                if (n0 > 0) valid = true, agent_draw = true;
            } else {
                const u32 u = (MODE == MODE_INDEX) ? input : philox_draw(v.seed, genv, ep, step_idx, 0u);
                if (n0 > 0) {
                    action = action_at<MULTI>(pick_sr, s, (int)gcb_umulhi(u, (u32)n0));
                    valid = true;
                }
            }
        }
        // a bot ply is owed first: the agent's action is refused and step_in_episode does not advance; the statistics count
        // the call as a step and as an invalid one
        const bool refused = !SELFPLAY && s.pending;
        if (refused) valid = false;
        st.f += SF_STEPS + (stm_checked(s) ? SF_INCHECK : 0u), st.legal += n0;
        if (!refused) s.step++;
        if (!valid) {  // chess_v2.py:240-242, before the done test (Q16)
            R = -10, d_out = s.done, fl |= EF_INVALID, st.f += SF_INVALID;
            phase = PH_FINAL;
        } else if (s.done) {  // chess_v2.py:245-251
            R = 0, d_out = true;
            phase = PH_FINAL;
        } else if (capped) {  // chess_v2.py:252-258: done is NOT latched (Q12)
            R = 0, d_out = true, fl |= EF_CAP;
            phase = PH_FINAL;
        } else {
            R = -10;  // chess_v2.py:261 (sic)
            phase = PH_AGENT;
        }
    }

    bool do_apply = true;
    int cur = action;  // cur = the action of the ply being executed
    // a bot ply draws its move at the top of the next loop trip: ONE site for the bot's reply (purpose 1) and for the bot's
    // opening ply after a reset (purpose 2) -- the ordered pick is 250 instructions, and the bot kernels wait for
    // instruction fetch more than for anything else
    u32 draw_purpose = 0u, draw_step = 0u;
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
    while (phase != PH_END) {
        if (!SELFPLAY && (draw_purpose || agent_draw)) {
            // agent: purpose 0 at this step (or the caller's random word), from the slots the step found; bot: purpose 1 / 2
            const u32 u = (agent_draw && MODE == MODE_INDEX) ? input : philox_draw(v.seed, genv, ep, agent_draw ? step_idx : draw_step, draw_purpose);
            cur = action_at<MULTI>(agent_draw ? pick_sr : sr, s, (int)gcb_umulhi(u, (u32)s.n_legal));
            if (agent_draw) action = cur;
            else if (draw_purpose == 1u) bot_action = cur;
            draw_purpose = 0u, agent_draw = false;
        }
        if (phase == PH_FINAL) {
            bool terminal;
            if (MODE == MODE_RESET) {
                terminal = true;
            } else {
                if (agent_ply) d_out = s.done;
                terminal = !owe_bot && (d_out || s.n_legal == 0);
                if (!owe_bot && !d_out && s.n_legal == 0) fl |= EF_WEDGED;
                // F_BOT_PENDING = the env owes the bot a ply when the call returns: the reply to this step's ply, a ply still
                // owed (a refused step) or the opening of the BLACK-agent episode an auto-reset starts
                if (v_ext && ((v.auto_reset && terminal) ? v_agent_black : s.pending)) fl |= EF_BOT_PENDING;
                if (n0 == 0 || was_done || owe_bot || (fl & EF_INVALID)) {
                } else if (capped) st.f += SF_CAPS;
                else if (d_out) {
                    if (fl & EF_MATE) st.f += SF_MATES;
                    else st.f += SF_REPS;
                } else if (s.n_legal == 0) st.f += SF_WEDGED;
                if (terminal) st.f += SF_EPISODES;
                st.reward += R;
                if (v.auto_reset && terminal) fl |= EF_RESET;
                GCB_CHK((unsigned)e < (unsigned)v.N, CHK_IO_INDEX);
                if (io.reward) io.reward[e] = R;
                if (io.done) io.done[e] = d_out ? 1 : 0;
                if (io.flags) io.flags[e] = (uint8_t)fl;
                // (self-play sets no flag above F_RESET; saying so keeps the self-play kernels' packing as it was)
                if (io.packed) io.packed[e] = pack_result(R, d_out, SELFPLAY ? fl & 63u : fl);
                if (io.act_out) io.act_out[e] = action;
            }
            if ((MODE == MODE_RESET) || (v.auto_reset && terminal)) {
                // ChessEnvV2.reset, chess_v2.py:183-217: copy the prepared initial state
                const int t = (int)(genv % (u32)v.n_templates);
                ulonglong2 a = v.t_bb01[t], c = v.t_bb23[t];
                s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
                unpack_meta(v.t_meta[t], s);
                s.zk = v.t_zkey[t];
                s.gen++;  // a new episode: the repetition table starts empty
                {
                    ulonglong2 ct = v.t_cnt[t];
                    s.cnt_lo = ct.x, s.cnt_hi = ct.y;
                }
                const int np = gcb_popc(s.b.w);  // White is to move in every initial state
                const u64* ts = v.t_tgt + (size_t)t * v.slots;
                {
                    TgtSink dst(sr, nullptr);
                    for (int r = 0; r < np && r < sr.slots; r++) dst.st(r, ts[r]);
                    st.wrote_slots = true;
                }
                ep += (u32)io.ep_inc;
                if (v_agent_black && v_ext) {
                    s.pending = 1;  // the caller's opponent opens for White (chess_v2.py:208-216): gcb_env_bot_ply
                } else if (v_agent_black) {
                    // the bot opens for White (chess_v2.py:208-216)
                    if (s.n_legal > 0) {
                        draw_purpose = 2u, draw_step = 0u;  // (drawn with the NEW episode counter, at the top of the next trip)
                        do_apply = true;
                    } else {
                        do_apply = false;
                    }
                    phase = PH_RESETBOT;
                    continue;
                }
            }
            phase = PH_END;
            continue;
        }
        bool rep;
        const int r = ply_and_movegen<FAST>(v, e, s, cur, do_apply, &rep, st, scratch, sr, geo);
        if (do_apply) st.f += SF_PLIES;
        const bool mate = s.n_legal == 0 && stm_checked(s);
        if (phase == PH_AGENT) {
            agent_ply = true;
            R += r;
            s.done = rep;
            if (rep) fl |= EF_REPETITION;
            if (mate) s.done = 1, R += 100, fl |= EF_MATE;  // chess_v2.py:270-272
            if (!s.done && v_ext) {
                s.pending = 1, owe_bot = true;  // the step ends here; the reward so far is reported, the bot's ply follows
            } else if (!s.done && v_bot) {
                if (s.n_legal > 0) {  // chess_v2.py:277-288
                    draw_purpose = 1u, draw_step = step_idx;
                    phase = PH_BOT;
                    continue;
                }
                // bot without moves and not in check: the reference raises TypeError (Q9); stop here
            } else if (!s.done) {
                if (!s.stm_black) s.move_count++;  // chess_v2.py:291-292
            }
            phase = PH_FINAL;
        } else if (phase == PH_BOT) {
            R -= r;
            s.done = rep;
            if (rep) fl |= EF_REPETITION;
            if (mate) s.done = 1, R -= 100, fl |= EF_MATE;  // chess_v2.py:286-288
            if (!s.stm_black) s.move_count++;
            phase = PH_FINAL;
        } else {                // PH_RESETBOT
            s.move_count += 1;  // chess_v2.py:214
            s.done = 0;
            if (MODE == MODE_BOTPLY) {
                // the caller's opening ply: the reference's reset discards its reward and clears done, and nothing is owed after it
                GCB_CHK((unsigned)e < (unsigned)v.N, CHK_IO_INDEX);
                if (io.reward) io.reward[e] = 0;
                if (io.done) io.done[e] = 0;
                if (io.flags) io.flags[e] = 0;
                if (io.packed) io.packed[e] = pack_result(0, false, 0u);
                if (io.act_out) io.act_out[e] = action;
            }
            phase = PH_END;
        }
    }
    if (MODE != MODE_RESET && MODE != MODE_BOTPLY && io.bot_out) io.bot_out[e] = bot_action;
}

template <int MODE>
GCB_HD void env_step_one(const EnvView& v, const StepIO& io, int e, StepStats& st, CountBytes* scratch) {
    EnvRegs s;
    u32 ep;
    env_load(v, e, s, ep);
    const SlotRef sr = resident_slots(v, e);
    const u32 input = step_input<MODE>(io, e);
    env_step_regs<MODE, false, false, false>(v, io, e, s, ep, st, scratch, sr, sr, GeomGlobal(), input);
    env_store(v, e, s, ep);
}

// A new episode of env e from an arbitrary position in the reference's wire format (the `state` setter of
// chess_v2.py:315-323 + engine.update_state + get_possible_moves for the side to move): rights masked by king presence,
// both check flags, legal set, empty repetition window, episode counter + 1.
GCB_HD void env_import_one(const EnvView& v, int e, const int8_t* board, int player, u32 rights, int move_count,
                           StepStats& st, CountBytes* scratch) {
    EnvRegs s;
    u32 ep;
    env_load(v, e, s, ep);
    s.b = board_from_mailbox(board);
    s.zk = zobrist_full(s.b);
    s.rights = mask_rights(s.b, rights);
    s.done = 0, s.move_count = move_count, s.step = 0, s.hist_len = 0, s.pending = 0;
    s.gen++;  // a new episode: the repetition table starts empty
    s.stm_black = player < 0 ? 0 : 1;  // ply_and_movegen(apply = false) flips the side, then generates for it
    bool rep;
    ply_and_movegen(v, e, s, 0, false, &rep, st, scratch, resident_slots(v, e), GeomGlobal());
    env_store(v, e, s, ep + 1u);
}

// Clone (gcb_env_clone): env d of `dst` becomes env i of `src` mid-episode -- board, key, meta (done, counters, hist_len,
// bot_pending), count bytes, piece slots and the live entries of the repetition window.  The destination keeps its global id,
// seed, templates and statistics rows; its episode counter advances by one (a re-clone into the same row draws new words) and
// its window moves to a new generation G = its old generation + 1, under which every entry it held before is dead.  The three
// parts below are what one warp of k_env_clone splits among its lanes; env_clone_one runs them in sequence.
//
// The per-env words of the clone.  Returns G; *src_gen / *src_hist receive the source's generation and window length.
GCB_HD u32 env_clone_words(const EnvView& dst, int d, const EnvView& src, int i, u32* src_gen, int* src_hist) {
    EnvRegs s;
    u32 ep;
    env_load(src, i, s, ep);
    *src_gen = s.gen, *src_hist = s.hist_len;
    GCB_CHK((unsigned)d < (unsigned)dst.N, CHK_ENV_INDEX);
    s.gen = GCB_LDS(&dst.gen[d]) + 1u;
    env_store(dst, d, s, GCB_LDS(&dst.episode[d]) + 1u);
    return s.gen;
}
// piece slot r of the clone
GCB_HD void env_clone_slot(const EnvView& dst, int d, const EnvView& src, int i, int r) {
    const TgtSink from(resident_slots(src, i), nullptr);
    TgtSink to(resident_slots(dst, d), nullptr);
    to.st(r, from.get(r));
}
// one repetition-table entry of the source, retagged in place for the destination's generation G: true if it is live (and
// must be written to the SAME slot of the destination's table -- live entries keep their slots and hence their probe chains;
// nothing is ever deleted within a generation, and the overflow replacement of rep_lookup_insert keeps chains intact)
GCB_HD bool rep_clone_entry(ulonglong2& en, u32 src_gen, u32 G) {
    const u64 c = en.y & 3ULL;
    if ((en.y >> 2) != (u64)src_gen || c == 0) return false;
    en.y = ((u64)G << 2) | c;
    return true;
}
GCB_HD void env_clone_one(const EnvView& dst, int d, const EnvView& src, int i) {
    u32 sgen;
    int hist;
    const u32 G = env_clone_words(dst, d, src, i, &sgen, &hist);
    for (int r = 0; r < dst.slots; r++) env_clone_slot(dst, d, src, i, r);
    if (hist == 0) return;  // an empty window: every source entry is dead, nothing to read
    const size_t H2 = (size_t)src.hist_mask + 1;
    const ulonglong2* from = src.rep + (size_t)i * H2;
    ulonglong2* to = dst.rep + (size_t)d * H2;
    for (size_t k = 0; k < H2; k++) {
        ulonglong2 en = GCB_LDS(&from[k]);
        if (rep_clone_entry(en, sgen, G)) GCB_STS(&to[k], en);
    }
}

// initial state of one template board (ChessEnvV2.reset up to the first movegen, chess_v2.py:188-206)
GCB_HD void make_template_one(int i, const int8_t* boards, ulonglong2* bb01, ulonglong2* bb23, u64* meta, u64* zkey,
                              u64* tgt, ulonglong2* cnt, int slots) {
    Board b = board_from_mailbox(boards + (size_t)i * 64);
    EnvRegs s;
    s.b = b;
    s.zk = zobrist_full(b);
    s.rights = mask_rights(b, 15u);  // all four True, then engine.update_state masks them (chess_v2.py:195-204)
    s.chk = check_flags(b);
    s.stm_black = 0, s.done = 0, s.move_count = 0, s.step = 0, s.hist_len = 0, s.pending = 0, s.gen = 0;
    GenCtx g;
    gen_prepare(b, 1, g);
    CountBytes scratch;
    SlotRef tsr = {tgt + (size_t)i * slots, 1u, slots, true};
    TgtSink sink(tsr, &scratch);
    gen_targets(b, g, g.own, sink);
    const int n = sink.total();
    s.castle = gen_castles(b, g, s.rights);
    s.n_legal = n + (int)(s.castle & 1u) + (int)(s.castle >> 1);
    cnt[i] = make_ulonglong2(sink.count_lo(), sink.count_hi());
    bb01[i] = make_ulonglong2(b.t0, b.t1);
    bb23[i] = make_ulonglong2(b.t2, b.w);
    meta[i] = pack_meta(s);
    zkey[i] = s.zk;
}

// Host set-up that gcb_env_create and the host emulation share.  The start position (DEFAULT_BOARD): the template when no
// initial boards are given.
static const int8_t kDefaultBoard[64] = {-3, -5, -4, -2, -1, -4, -5, -3, -6, -6, -6, -6, -6, -6, -6, -6, 0, 0, 0, 0, 0, 0,
                                         0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0, 0, 0, 0, 0, 0,
                                         0,  0,  0,  0,  6,  6,  6,  6,  6,  6,  6,  6,  3,  5,  4,  2,  1, 4, 5, 3};
// The automatic piece-slot count (piece_slots = 0): one slot per own piece of the side to move -- the most pieces either side
// has on any template, at least 16.  Piece counts never grow (no promotion in play, Q1).
static inline int auto_piece_slots(int n_templates, const int8_t* template_boards) {
    int need = 16;
    for (int t = 0; t < n_templates && template_boards; t++) {
        int w = 0, bl = 0;
        for (int sq = 0; sq < 64; sq++) {
            int8_t p = template_boards[(size_t)t * 64 + sq];
            w += p > 0, bl += p < 0;
        }
        need = need < w ? w : need;
        need = need < bl ? bl : need;
    }
    return need;
}

// ordered list -> memory, one uint16 per move at its list position (moves beyond `cap` are dropped, the count is kept)
struct ListOut {
    uint16_t* out;
    int cap;
    GCB_HD void put(int pos, int action) {
        if (pos < cap) out[pos] = (uint16_t)action;
    }
};

// ChessEnvV2.possible_actions (chess_v2.py:333-335) of env e: decode the slots into the reference-ordered list.
// Handles any number of slots by chunks of GCB_SLOTS.  Returns the list length.
// `stage` (may be NULL): GCB_SLOTS words of scratch, element r at stage[r * stage_stride] -- the chunk's slots are copied
// there first (row by row: coalesced across the envs of a warp), so that the decode's per-piece reads do not each pay a
// trip to L2.
template <class Offs, class Out>
GCB_HD int env_legal_list_one(const EnvView& v, int e, Offs& offs, Out& out, u64* stage = nullptr, unsigned stage_stride = 1) {
    EnvRegs s;
    ulonglong2 a = v.bb01[e], c = v.bb23[e];
    s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
    unpack_meta(v.meta[e], s);
    int n = 0, r0 = 0;
    u64 rem = stm_pieces(s);
    while (rem) {
        u64 chunk = rem;
        if (gcb_popc(rem) > GCB_SLOTS) {
            u64 t = rem;
            for (int i = 0; i < GCB_SLOTS; i++) t &= t - 1;
            chunk = rem ^ t;
        }
        rem ^= chunk;
        SlotRef csr = {v.tgt + (size_t)r0 * v.N + e, (unsigned)v.N, v.slots - r0, false};
        if (stage) {
            const int np = gcb_popc(chunk);
            TgtSink src(csr, nullptr);
            for (int r = 0; r < np; r++) stage[(unsigned)r * stage_stride] = src.get(r);
            SlotRef ssr = {stage, stage_stride, np, true};
            csr = ssr;
        }
        TgtSink slots(csr, nullptr);
        n = emit_chunk_typemajor(s.b, !s.stm_black, chunk, slots, offs, out, n);
        r0 += GCB_SLOTS;
    }
    if (s.castle & 1u) out.put(n++, castle_action(!s.stm_black, 0));
    if (s.castle & 2u) out.put(n++, castle_action(!s.stm_black, 1));
    return n;
}

// unpacked view of one env for export: board int8[64] (may be NULL) and info int32[16]
GCB_HD void env_export_one(const EnvView& v, int e, int8_t* board, int32_t* info) {
    EnvRegs s;
    ulonglong2 a = v.bb01[e], c = v.bb23[e];
    s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
    unpack_meta(v.meta[e], s);
    if (board)
        for (int sq = 0; sq < 64; sq++) board[sq] = (int8_t)piece_id(s.b, sq);
    if (info) {
        info[0] = s.stm_black ? -1 : 1, info[1] = s.rights & RT_WK ? 1 : 0, info[2] = s.rights & RT_WQ ? 1 : 0;
        info[3] = s.rights & RT_BK ? 1 : 0, info[4] = s.rights & RT_BQ ? 1 : 0, info[5] = s.chk & 1, info[6] = (s.chk >> 1) & 1;
        info[7] = s.done, info[8] = s.move_count, info[9] = s.n_legal, info[10] = (int)v.episode[e], info[11] = s.step;
        info[12] = s.hist_len, info[13] = (int)s.castle, info[14] = s.pending, info[15] = 0;
    }
}

// ---- Policy sampling (gcb_env_sample_policy): one legal action of the side to move per env, drawn from caller logits.
// L = the resident legal set of env e (slot r of the r-th own piece, plus the castle bits: what gcb_env_legal_bitmask
// exports) in ascending ACTION CODE -- from-square, then to-square, then 4096..4099.  That is the order the slots give for
// free, not the reference's list order.  Only the logits of L are read.  With temperature T > 0: z_a = x_a / T,
// m = max z, w_a = exp(z_a - m), Z = sum w; the action is the first a of L whose inclusive prefix sum of w exceeds u * Z
// (policy_u), or the last a with w_a > 0 if rounding leaves none; logp = z_a - m - log Z.  T == 0: the argmax of x over L,
// ties to the lowest code, logp = 0.  A legal entry of -inf is never chosen; no legal move or no finite legal entry gives
// RESIGN with logp 0.  Below: the pieces the kernel (k_env_policy_sample) and the serial form share.
#if defined(__CUDA_ARCH__)
#define GCB_LDG(p) __ldg(p)
#else
#define GCB_LDG(p) (*(p))
#endif
GCB_HD float gcb_bits_to_float(u32 x) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(x);
#else
    float f;
    __builtin_memcpy(&f, &x, 4);
    return f;
#endif
}
// logit a of a row; DT 0 = fp32, 1 = bf16 (GCB_DT_F32 / GCB_DT_BF16), widened exactly: a bf16 is the high half of an fp32
template <int DT>
GCB_HD float policy_logit(const void* row, int a) {
    GCB_CHK((unsigned)a < 4101u, CHK_POLICY_INDEX);
    if (DT == 1) return gcb_bits_to_float((u32)GCB_LDG(reinterpret_cast<const uint16_t*>(row) + a) << 16);
    return GCB_LDG(reinterpret_cast<const float*>(row) + a);
}
template <int DT>
GCB_HD const void* policy_row(const void* logits, long long row_stride, int e) {
    return reinterpret_cast<const char*>(logits) + (size_t)e * (size_t)row_stride * (DT == 1 ? 2u : 4u);
}
// the draw u in (0, 1] of a random word: (word >> 8) * 2^-24 + 2^-25 in fp32 -- exact while word >> 8 < 2^23, rounded to
// nearest even above (the top value rounds to 1.0, which no prefix sum exceeds); one rounding, the same on host and device
GCB_HD float policy_u(u32 word) { return (float)(word >> 8) * 5.9604644775390625e-08f + 2.98023223876953125e-08f; }
// the default random word: Philox on the env's key, counter (global env id, episode, step in episode, 3 + side to move is
// black) -- purposes 0-2 are the step's draws, and the side to move keeps the agent's and an external bot's draws apart
GCB_HD u32 policy_word(const EnvView& v, int e, const EnvRegs& s, u32 ep) {
    return philox_draw(v.seed, v.env_offset + (u32)e, ep, (u32)s.step, 3u + (u32)s.stm_black);
}
// what a sample reads of the state: board, meta, episode counter (plain loads: a step that follows finds them in L2)
GCB_HD void policy_load(const EnvView& v, int e, EnvRegs& s, u32& ep) {
    GCB_CHK((unsigned)e < (unsigned)v.N, CHK_POLICY_INDEX);
    const ulonglong2 a = v.bb01[e], c = v.bb23[e];
    s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
    unpack_meta(v.meta[e], s);
    ep = v.episode[e];
}
// greedy step: strict > keeps the lowest code of a tie when L is visited in code order; -inf and NaN never win
GCB_HD void policy_argmax(float x, int a, float& best, int& pick) {
    if (x > best) best = x, pick = a;
}
// f(a) for every a of L in code order; pieces beyond the slots have no resident targets (as in gcb_env_legal_bitmask)
template <class F>
GCB_HD void policy_walk(const EnvView& v, int e, const EnvRegs& s, F f) {
    const TgtSink slots(resident_slots(v, e), nullptr);
    int r = 0;
    for (u64 t = stm_pieces(s); t; t &= t - 1, r++) {
        const int from = gcb_lsb(t);
        for (u64 T = slots.get(r); T; T &= T - 1) f(from * 64 + gcb_lsb(T));
    }
    for (u32 c = castle_word(s); c; c &= c - 1) f(4096 + gcb_lsb((u64)c));
}
// The serial form (the host emulation): three walks over L -- max, sum, prefix-sum selection.
template <int DT>
GCB_HD void env_policy_sample_one(const EnvView& v, int e, const void* logits, long long row_stride, float temp, const u32* words,
                                  int32_t* act, float* logp) {
    EnvRegs s;
    u32 ep;
    policy_load(v, e, s, ep);
    const void* row = policy_row<DT>(logits, row_stride, e);
    int pick = -1;
    float lp = 0.f;
    if (temp == 0.f) {
        float best = -INFINITY;
        policy_walk(v, e, s, [&](int a) { policy_argmax(policy_logit<DT>(row, a), a, best, pick); });
    } else {
        float m = -INFINITY;
        policy_walk(v, e, s, [&](int a) {
            const float z = policy_logit<DT>(row, a) / temp;
            if (z > m) m = z;
        });
        if (m > -INFINITY) {
            float Z = 0.f;
            policy_walk(v, e, s, [&](int a) { Z += expf(policy_logit<DT>(row, a) / temp - m); });
            const float target = policy_u(words ? GCB_LDG(words + e) : policy_word(v, e, s, ep)) * Z;
            float acc = 0.f, zp = 0.f, zl = 0.f;
            int last = -1;
            policy_walk(v, e, s, [&](int a) {
                const float z = policy_logit<DT>(row, a) / temp, w = expf(z - m);
                acc += w;
                if (pick < 0 && acc > target) pick = a, zp = z;
                if (w > 0.f) last = a, zl = z;
            });
            if (pick < 0) pick = last, zp = zl;
            lp = zp - m - logf(Z);
        }
    }
    act[e] = pick < 0 ? ACT_RESIGN : pick;
    if (logp) logp[e] = pick < 0 ? 0.f : lp;
}

// ---- Network input (gcb_env_encode): 19 binary planes of 8 x 8 per env, square sq = row * 8 + col (row 0 = rank 8), as
// 64-bit masks (bit sq of mask c = element [c][sq]): 0-5 White K Q R B N P, 6-11 Black K Q R B N P, 12 Black to move,
// 13-16 castle flags wk wq bk bq, 17 the board has occurred >= 1 time and 18 >= 2 times as the pre-move board of a ply of
// this episode.  The count is the repetition table's, probed with the board-only key the step uses, without inserting:
// rep_lookup_insert answers "occurrences including this ply" = stored count + 1, and saturates at 3.  A window that has
// outgrown the table (its overflow branch answers 1) or a key collision can miss a repetition here exactly as in the step.
enum { OBS_PLANES = 19 };
GCB_HD void env_encode_masks(const EnvView& v, int e, u64* m, int* rep) {
    GCB_CHK((unsigned)e < (unsigned)v.N, CHK_ENCODE_INDEX);
    EnvRegs s;
    const ulonglong2 a = v.bb01[e], c = v.bb23[e];
    s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
    unpack_meta(v.meta[e], s);
    const u64 white = s.b.w, black = bb_occ(s.b) & ~s.b.w;
    const u64 kind[6] = {bb_kings(s.b), bb_queens(s.b), bb_rooks(s.b), bb_bishops(s.b), bb_knights(s.b), bb_pawns(s.b)};
    for (int k = 0; k < 6; k++) m[k] = kind[k] & white, m[6 + k] = kind[k] & black;
    m[12] = s.stm_black ? ~0ULL : 0ULL;
    for (int k = 0; k < 4; k++) m[13 + k] = (s.rights >> k) & 1u ? ~0ULL : 0ULL;  // RT_WK, RT_WQ, RT_BK, RT_BQ
    int n = 0;
    if (s.hist_len != 0) {  // an empty window holds no live entry: nothing to read
        s.zk = v.zkey[e], s.gen = v.gen[e];
        StepStats local;
        local.clear();
        n = rep_lookup_insert(v, e, s, hist_key(s.zk), /*insert=*/false, local) - 1;
    }
    m[17] = n >= 1 ? ~0ULL : 0ULL;
    m[18] = n >= 2 ? ~0ULL : 0ULL;
    *rep = n;
}
// element values: DT 0 = fp32, 1 = bf16 (as its 16-bit pattern), 2 = uint8 (GCB_DT_F32 / GCB_DT_BF16 / GCB_DT_U8)
template <int DT> struct EncodeElem { typedef float type; };
template <> struct EncodeElem<1> { typedef uint16_t type; };
template <> struct EncodeElem<2> { typedef uint8_t type; };
template <int DT>
GCB_HD typename EncodeElem<DT>::type encode_value(u32 bit) {
    if (DT == 0) return bit ? 1.0f : 0.0f;
    return (typename EncodeElem<DT>::type)(DT == 1 ? bit * 0x3F80u : bit);  // bf16 1.0 = 0x3F80
}
// The serial form (the host emulation): env e's masks expanded into its row planes[e][19][64]; rep_out[e] (either may be NULL)
template <int DT>
GCB_HD void env_encode_one(const EnvView& v, int e, typename EncodeElem<DT>::type* planes, uint8_t* rep_out) {
    u64 m[OBS_PLANES];
    int rep;
    env_encode_masks(v, e, m, &rep);
    if (planes) {
        typename EncodeElem<DT>::type* row = planes + (size_t)e * OBS_PLANES * 64;
        for (int c = 0; c < OBS_PLANES; c++)
            for (int sq = 0; sq < 64; sq++) row[c * 64 + sq] = encode_value<DT>((u32)(m[c] >> sq) & 1u);
    }
    if (rep_out) rep_out[e] = (uint8_t)rep;
}
