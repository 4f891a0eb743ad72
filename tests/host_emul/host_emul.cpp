// host_emul.cpp -- TEST INFRASTRUCTURE.  Compiles the device rules (gym_chess_b200/csrc/chess_core.cuh,
// env_core.cuh) with g++ so that `pytest -m "not gpu"` can check the bitboard / step / clone / policy / encode LOGIC
// against the oracle on a box without a GPU.  It is never loaded by the product package; the product has no CPU path.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../../gym_chess_b200/csrc/env_core.cuh"

extern "C" {

struct LocalSlots {
    u64 t[GCB_SLOTS];
    void put(int r, u64 v) { t[r] = v; }
    u64 get(int r) const { return t[r]; }
    void replace(int r, u64, u64 v) { t[r] = v; }
};
struct LocalOffs {
    int o[GCB_SLOTS];
    void set(int r, int v) { o[r] = v; }
    int get(int r) const { return o[r]; }
};

void emul_movegen(int n, const int8_t* boards, const int8_t* players, const uint8_t* rights4, int attack, int castles_only,
                  uint16_t* out, int stride, int32_t* counts, uint8_t* incheck) {
    for (int i = 0; i < n; i++) {
        Board b = board_from_mailbox(boards + (size_t)i * 64);
        const uint8_t* q = rights4 + (size_t)i * 4;
        u32 rights = (q[0] ? RT_WK : 0) | (q[1] ? RT_WQ : 0) | (q[2] ? RT_BK : 0) | (q[3] ? RT_BQ : 0);
        rights = mask_rights(b, rights);
        bool chk = false;
        int cnt;
        if (attack) {  // the kernel's form (slots + type-major decode) ...
            LocalSlots slots;
            LocalOffs offs;
            ListOut lo = {out + (size_t)i * stride, stride};
            cnt = gen_attack_list(b, players[i] > 0, slots, offs, lo);
            // ... which must equal the direct square-major generator
            uint16_t tmp[512];
            ListWriter lw(tmp, 512);
            gen_attack_moves(b, players[i] > 0, lw);
            lw.flush();
            bool same = lw.n == cnt;
            for (int k = 0; same && k < cnt && k < stride && k < 512; k++) same = tmp[k] == out[(size_t)i * stride + k];
            if (!same) cnt = -1;
        } else {
            LocalSlots slots;
            LocalOffs offs;
            ListOut lo = {out + (size_t)i * stride, stride};
            cnt = gen_legal_list(b, players[i] > 0, rights, slots, offs, lo, &chk);
        }
        if (castles_only) {
            uint16_t* l = out + (size_t)i * stride;
            int m = 0, lim = cnt < stride ? cnt : stride;
            for (int k = 0; k < lim; k++)
                if (l[k] >= 4096) l[m++] = l[k];
            cnt = m;
        }
        counts[i] = cnt;
        if (incheck) incheck[i] = chk;
    }
}

void emul_next_state(int n, const int8_t* boards, const int8_t* players, const uint8_t* rights4, const int32_t* actions,
                     int8_t* out_boards, uint8_t* out_rights4, uint8_t* out_checks, int32_t* out_reward, int8_t* out_status) {
    for (int i = 0; i < n; i++) {
        Board b = board_from_mailbox(boards + (size_t)i * 64);
        const uint8_t* q = rights4 + (size_t)i * 4;
        u32 rights = (q[0] ? RT_WK : 0) | (q[1] ? RT_WQ : 0) | (q[2] ? RT_BK : 0) | (q[3] ? RT_BQ : 0);
        rights = mask_rights(b, rights);
        Board nb = b;
        int st;
        bool irr;
        int r = apply_action(nb, rights, players[i] > 0, actions[i], &st, &irr);
        if (st) nb = b, r = 0;
        for (int sq = 0; sq < 64; sq++) out_boards[(size_t)i * 64 + sq] = (int8_t)piece_id(nb, sq);
        out_rights4[4 * i] = rights & RT_WK ? 1 : 0, out_rights4[4 * i + 1] = rights & RT_WQ ? 1 : 0;
        out_rights4[4 * i + 2] = rights & RT_BK ? 1 : 0, out_rights4[4 * i + 3] = rights & RT_BQ ? 1 : 0;
        u32 c = check_flags(nb);
        out_checks[2 * i] = c & 1, out_checks[2 * i + 1] = (c >> 1) & 1;
        out_reward[i] = r, out_status[i] = (int8_t)(st ? st : (c == 3u ? 1 : 0));
    }
}

void emul_update_state(int n, const int8_t* boards, const uint8_t* rights4, uint8_t* out_rights4, uint8_t* out_checks) {
    for (int i = 0; i < n; i++) {
        Board b = board_from_mailbox(boards + (size_t)i * 64);
        const uint8_t* q = rights4 + (size_t)i * 4;
        u32 rights = (q[0] ? RT_WK : 0) | (q[1] ? RT_WQ : 0) | (q[2] ? RT_BK : 0) | (q[3] ? RT_BQ : 0);
        rights = mask_rights(b, rights);
        out_rights4[4 * i] = rights & RT_WK ? 1 : 0, out_rights4[4 * i + 1] = rights & RT_WQ ? 1 : 0;
        out_rights4[4 * i + 2] = rights & RT_BK ? 1 : 0, out_rights4[4 * i + 3] = rights & RT_BQ ? 1 : 0;
        u32 c = check_flags(b);
        out_checks[2 * i] = c & 1, out_checks[2 * i + 1] = (c >> 1) & 1;
    }
}

// nth_target (the ordered pick's "idx-th move of this piece") against the walk it abbreviates, emit_piece_moves: for every
// piece class, colour and from-square, the full reach of the class and `rounds` random subsets of it, every idx.
// Returns the number of (class, square, subset, idx) cases checked, or -(1 + first failing case) on a mismatch.
long emul_nth_target_check(uint64_t seed, int rounds) {
    struct Collect {
        int to[64], n;
        void push(int action) { to[n++] = action & 63; }
    };
    const int codes[6] = {PC_KING, PC_QUEEN, PC_ROOK, PC_BISHOP, PC_KNIGHT, PC_PAWN};
    long cases = 0;
    u64 x = seed | 1ULL;
    for (int ci = 0; ci < 6; ci++)
        for (int white = 0; white < 2; white++)
            for (int sq = 0; sq < 64; sq++) {
                const int code = codes[ci], cls = order_class(code, white);
                u64 reach = 0;
                for (int k = 0; k < 8; k++) reach |= g_geom_host.ord[cls][sq][k];
                if (code == PC_ROOK) reach = g_geom_host.line[sq][0] | g_geom_host.line[sq][1];
                if (code == PC_BISHOP) reach = g_geom_host.line[sq][2] | g_geom_host.line[sq][3];
                for (int r = 0; r <= rounds; r++) {
                    x = gcb_splitmix64(x);
                    const u64 T = r == 0 ? reach : (reach & x & gcb_splitmix64(x ^ 0x5555ULL));
                    Collect c;
                    c.n = 0;
                    emit_piece_moves(c, code, white, sq, T);
                    if (c.n != gcb_popc(T)) return -(1 + cases);
                    for (int idx = 0; idx < c.n; idx++, cases++) {
                        if (nth_target<true>(code, white, sq, T, idx) != c.to[idx]) return -(1 + cases);
                        if (nth_target<false>(code, white, sq, T, idx) != c.to[idx]) return -(1 + cases);
                    }
                }
            }
    return cases;
}

uint32_t emul_philox(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step, uint32_t purpose) {
    return philox_draw(seed, env, episode, step, purpose);
}

// ---- env emulation: same SoA arrays, host memory, the same env_step_one()
struct EmulEnv {
    EnvView v;
    u64 tick;
    ulonglong2 *t_bb01, *t_bb23;
    u64 *t_meta, *t_zkey, *t_tgt, *zob;
    ulonglong2* t_cnt;
};

void emul_env_destroy(EmulEnv* E) {
    if (!E) return;
    free(E->v.bb01), free(E->v.bb23), free(E->v.meta), free(E->v.zkey), free(E->v.gen), free(E->v.cnt), free(E->t_cnt), free(E->v.episode), free(E->v.tgt);
    free(E->v.rep), free(E->v.stats), free(E->t_bb01), free(E->t_bb23), free(E->t_meta), free(E->t_zkey), free(E->t_tgt), free(E->zob);
    free(E);
}

// slots 0 = automatic, as gcb_env_config.piece_slots
EmulEnv* emul_env_create(int N, uint32_t env_offset, uint64_t seed, int opponent, int agent_black, int auto_reset, int slots,
                         int hist_cap, int moves_max, int n_templates, const int8_t* template_boards) {
    if (slots == 0) slots = auto_piece_slots(n_templates, template_boards);
    EmulEnv* E = (EmulEnv*)calloc(1, sizeof(EmulEnv));
    int T = n_templates > 0 ? n_templates : 1;
    EnvView& v = E->v;
    v.bb01 = (ulonglong2*)calloc(N, 16), v.bb23 = (ulonglong2*)calloc(N, 16);
    v.meta = (u64*)calloc(N, 8), v.zkey = (u64*)calloc(N, 8), v.episode = (u32*)calloc(N, 4);
    v.gen = (u32*)calloc(N, 4), v.cnt = (ulonglong2*)calloc(N, 16), E->t_cnt = (ulonglong2*)calloc(T, 16);
    v.tgt = (u64*)calloc((size_t)N * slots, 8), v.rep = (ulonglong2*)calloc((size_t)N * 2 * hist_cap, 16);
    v.stats = (u64*)calloc(ST_COUNT, 8);
    E->t_bb01 = (ulonglong2*)calloc(T, 16), E->t_bb23 = (ulonglong2*)calloc(T, 16);
    E->t_meta = (u64*)calloc(T, 8), E->t_zkey = (u64*)calloc(T, 8), E->t_tgt = (u64*)calloc((size_t)T * slots, 8);
    E->zob = (u64*)calloc(GCB_ZOB_ENTRIES, 8);
    for (int i = 0; i < GCB_ZOB_ENTRIES; i++) fill_zobrist_entry(E->zob, i);
    v.t_bb01 = E->t_bb01, v.t_bb23 = E->t_bb23, v.t_meta = E->t_meta, v.t_zkey = E->t_zkey, v.t_tgt = E->t_tgt, v.zob = E->zob, v.t_cnt = E->t_cnt;
    v.seed = seed, v.N = N, v.slots = slots, v.hist_mask = 2 * hist_cap - 1, v.n_templates = T, v.env_offset = env_offset;
    v.moves_max = moves_max, v.opponent = opponent, v.agent_black = agent_black, v.auto_reset = auto_reset;
    v.pps = 1 + (opponent == 1);
    for (int i = 0; i < T; i++)
        make_template_one(i, n_templates > 0 ? template_boards : kDefaultBoard, E->t_bb01, E->t_bb23, E->t_meta, E->t_zkey, E->t_tgt, E->t_cnt, slots);
    StepIO io;
    memset(&io, 0, sizeof(io));
    io.tick = E->tick++, io.e_begin = 0, io.e_end = N, io.nsteps = 1;
    StepStats st;
    CountBytes scratch;
    for (int e = 0; e < N; e++) {
        st.clear();
        env_step_one<MODE_RESET>(v, io, e, st, &scratch);
    }
    return E;
}

// mode: 0 actions, 1 index words, 2 sampled, 3 reset (in = uint8 mask or NULL), 4 the bot ply of an external opponent
void emul_env_step(EmulEnv* E, int mode, const void* in, int32_t* reward, uint8_t* done, uint8_t* flags, int32_t* act_out,
                   int32_t* bot_out) {
    StepIO io;
    io.in = in, io.reward = reward, io.done = done, io.flags = flags, io.act_out = act_out, io.bot_out = bot_out;
    io.tick = E->tick++, io.ep_inc = 1, io.e_begin = 0, io.e_end = E->v.N, io.nsteps = 1;
    StepStats st;
    CountBytes scratch;
    for (int e = 0; e < E->v.N; e++) {
        st.clear();  // the counters of ONE env step (bit fields): summed into the totals env by env
        switch (mode) {
        case 0: env_step_one<MODE_ACTION>(E->v, io, e, st, &scratch); break;
        case 1: env_step_one<MODE_INDEX>(E->v, io, e, st, &scratch); break;
        case 2: env_step_one<MODE_SAMPLED>(E->v, io, e, st, &scratch); break;
        case 4: env_step_one<MODE_BOTPLY>(E->v, io, e, st, &scratch); break;
        default:
            if (!in || ((const uint8_t*)in)[e]) env_step_one<MODE_RESET>(E->v, io, e, st, &scratch);
        }
        if (mode != 3)
            for (int k = 0; k < ST_USED; k++) E->v.stats[k] += (u64)(long long)st.get(k);
    }
}

void emul_env_import(EmulEnv* E, const int8_t* boards, const int8_t* players, const uint8_t* rights4, const int32_t* move_count,
                     const uint8_t* mask) {
    StepStats st;
    CountBytes scratch;
    E->tick++;
    for (int e = 0; e < E->v.N; e++) {
        if (mask && !mask[e]) continue;
        const uint8_t* q = rights4 + (size_t)e * 4;
        u32 rights = (q[0] ? RT_WK : 0) | (q[1] ? RT_WQ : 0) | (q[2] ? RT_BK : 0) | (q[3] ? RT_BQ : 0);
        st.clear();
        env_import_one(E->v, e, boards + (size_t)e * 64, players[e], rights, move_count ? move_count[e] : 0, st, &scratch);
    }
}

void emul_env_export(EmulEnv* E, int8_t* boards, int32_t* info, uint16_t* legal, int legal_stride) {
    for (int e = 0; e < E->v.N; e++) {
        env_export_one(E->v, e, boards ? boards + (size_t)e * 64 : nullptr, info ? info + (size_t)e * 16 : nullptr);
        if (legal) {  // possible_actions: decode of the piece slots
            LocalOffs offs;
            ListOut lo = {legal + (size_t)e * legal_stride, legal_stride};
            env_legal_list_one(E->v, e, offs, lo);
        }
    }
}

void emul_env_stats(EmulEnv* E, uint64_t* out16) { memcpy(out16, E->v.stats, ST_COUNT * 8); }

int emul_env_piece_slots(const EmulEnv* E) { return E->v.slots; }

// the per-env clone (gcb_env_clone): the GCB_HD code of env_core.cuh that k_env_clone splits among the lanes of a warp, run
// row by row.  index int32[dst N]: env d of dst becomes env index[d] of src for 0 <= index[d] < src N; other rows are left untouched
void emul_env_clone(EmulEnv* dst, const EmulEnv* src, const int32_t* index) {
    for (int d = 0; d < dst->v.N; d++) {
        const int i = index[d];
        if (i < 0 || i >= src->v.N) continue;
        env_clone_one(dst->v, d, src->v, i);
    }
}

// policy sampling (gcb_env_sample_policy): env_policy_sample_one, the serial form of the rule that k_env_policy_sample runs
// with one warp per env.
// logits [N][row_stride] of dtype 0 (fp32) / 1 (bf16 as uint16); words uint32[N] or NULL (Philox); logp may be NULL
void emul_env_sample_policy(const EmulEnv* E, const void* logits, int dtype, long long row_stride, float temperature,
                            const uint32_t* words, int32_t* actions, float* logp) {
    for (int e = 0; e < E->v.N; e++) {
        if (dtype == 1) env_policy_sample_one<1>(E->v, e, logits, row_stride, temperature, words, actions, logp);
        else env_policy_sample_one<0>(E->v, e, logits, row_stride, temperature, words, actions, logp);
    }
}

// the network-input encoder (gcb_env_encode): env_encode_one, the serial form of the rule that k_env_encode writes with one
// warp per 32 envs.
// planes [N][19][64] of dtype 0 (fp32) / 1 (bf16 as uint16) / 2 (uint8), or NULL; rep uint8[N] or NULL
void emul_env_encode(const EmulEnv* E, void* planes, int dtype, uint8_t* rep) {
    for (int e = 0; e < E->v.N; e++) {
        if (dtype == 1) env_encode_one<1>(E->v, e, static_cast<uint16_t*>(planes), rep);
        else if (dtype == 2) env_encode_one<2>(E->v, e, static_cast<uint8_t*>(planes), rep);
        else env_encode_one<0>(E->v, e, static_cast<float*>(planes), rep);
    }
}

// the 16-bit result record of the packed step forms (gcb_env_step_packed)
uint16_t emul_pack_result(int reward, int done, uint32_t flags) { return pack_result(reward, done != 0, flags); }

}  // extern "C"
