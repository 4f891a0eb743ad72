// gcb_kernels.cu -- kernels + C ABI of libgymchess_b200.so (sm_100a).  See include/gymchess_b200.h.
//
// The per-env logic lives in env_core.cuh / chess_core.cuh; this file holds the kernels (one thread per env or
// position; the sampled self-play kernel runs up to 64 steps per launch), the per-warp statistics rows and their
// reduction, and the host-side C ABI.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/gymchess_b200.h"
#include "env_core.cuh"

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

static int fail(int code, const char* what, const char* detail) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, detail ? detail : "");
    return code;
}
#define CU(call)                                                                  \
    do {                                                                          \
        cudaError_t e_ = (call);                                                  \
        if (e_ != cudaSuccess) return fail(GCB_E_CUDA, #call, cudaGetErrorString(e_)); \
    } while (0)
#define LAUNCHED()                                                                \
    do {                                                                          \
        g_launches.fetch_add(1, std::memory_order_relaxed);                       \
        cudaError_t e_ = cudaGetLastError();                                      \
        if (e_ != cudaSuccess) return fail(GCB_E_CUDA, "kernel launch", cudaGetErrorString(e_)); \
    } while (0)

extern "C" const char* gcb_last_error(void) { return g_err; }
extern "C" int gcb_version(void) { return 200; }  // round 2: host calls take a stream, bot ply, mask output, guards
extern "C" uint64_t gcb_launch_count(void) { return g_launches.load(); }
extern "C" int gcb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

// the caller's current device is restored when an entry point returns (a process may drive several GPUs)
struct DeviceScope {
    int prev = -1;
    bool switched = false;
    cudaError_t enter(int dev) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) return e;
        if (prev == dev) return cudaSuccess;
        switched = true;
        return cudaSetDevice(dev);
    }
    ~DeviceScope() {
        if (switched) cudaSetDevice(prev);
    }
};

#ifndef GCB_BLOCK
#define GCB_BLOCK 128
#endif
#ifndef GCB_STEP_MIN_BLOCKS  // single-step kernels: 6 resident blocks per SM (80 registers, no spills) measure 3 % faster than 5
#define GCB_STEP_MIN_BLOCKS 6
#endif
#ifndef GCB_FAST_SINK
#define GCB_FAST_SINK 1
#endif
#ifndef GCB_SAMPLED_MIN_BLOCKS
#define GCB_SAMPLED_MIN_BLOCKS 5
#endif
#ifndef GCB_FAST_GENERIC  // unchecked slot stores also in the generic (resident-slot) kernels when the env has 16 slots
#define GCB_FAST_GENERIC 1
#endif
#ifndef GCB_SINGLE_TILE  // single-step launches generate on the shared-memory tile (TILE 2) when the env has 16 piece slots
#define GCB_SINGLE_TILE 1
#endif
#ifndef GCB_BITS_STREAM  // bit-mask rows of the step kernels: streaming (evict-first) stores (1) or default write-back stores (0)
#define GCB_BITS_STREAM 1
#endif
#if GCB_BITS_STREAM
#define GCB_BITS_ST(p, v) __stcs((p), (v))
#else
#define GCB_BITS_ST(p, v) (*(p) = (v))
#endif
static inline int grid_for(int n) { return (n + GCB_BLOCK - 1) / GCB_BLOCK; }

// ------------------------------------------------------------------------------------------------ pack / unpack
__global__ void __launch_bounds__(GCB_BLOCK) k_pack(int n, const int8_t* __restrict__ boards,
                                                    const int8_t* __restrict__ players,
                                                    const uint8_t* __restrict__ rights4, gcb_positions out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int4* src = reinterpret_cast<const int4*>(boards + (size_t)i * 64);
    alignas(16) int8_t m[64];
#pragma unroll
    for (int k = 0; k < 4; k++) *reinterpret_cast<int4*>(m + 16 * k) = __ldg(src + k);
    Board b = board_from_mailbox(m);
    reinterpret_cast<ulonglong2*>(out.bb01)[i] = make_ulonglong2(b.t0, b.t1);
    reinterpret_cast<ulonglong2*>(out.bb23)[i] = make_ulonglong2(b.t2, b.w);
    if (out.player) out.player[i] = players ? (players[i] < 0 ? 1 : 0) : 0;
    if (out.rights) {
        uint8_t r = 0;
        if (rights4) {
            uchar4 q = reinterpret_cast<const uchar4*>(rights4)[i];
            r = (q.x ? RT_WK : 0) | (q.y ? RT_WQ : 0) | (q.z ? RT_BK : 0) | (q.w ? RT_BQ : 0);
        }
        out.rights[i] = r;
    }
}

__device__ __forceinline__ void board_to_mailbox(const Board& b, int8_t* m) {
#pragma unroll
    for (int sq = 0; sq < 64; sq++) m[sq] = (int8_t)piece_id(b, sq);
}

__global__ void __launch_bounds__(GCB_BLOCK) k_unpack(int n, gcb_positions in, int8_t* __restrict__ boards,
                                                      int8_t* __restrict__ players, uint8_t* __restrict__ rights4) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ulonglong2 a = reinterpret_cast<const ulonglong2*>(in.bb01)[i], c = reinterpret_cast<const ulonglong2*>(in.bb23)[i];
    Board b = {a.x, a.y, c.x, c.y};
    if (boards) {
        alignas(16) int8_t m[64];
        board_to_mailbox(b, m);
        int4* dst = reinterpret_cast<int4*>(boards + (size_t)i * 64);
#pragma unroll
        for (int k = 0; k < 4; k++) dst[k] = *reinterpret_cast<int4*>(m + 16 * k);
    }
    if (players && in.player) players[i] = in.player[i] ? -1 : 1;
    if (rights4 && in.rights) {
        uint8_t r = in.rights[i];
        reinterpret_cast<uchar4*>(rights4)[i] = make_uchar4(r & RT_WK ? 1 : 0, r & RT_WQ ? 1 : 0, r & RT_BK ? 1 : 0, r & RT_BQ ? 1 : 0);
    }
}

// ------------------------------------------------------------------------------------------------ engine kernels
// piece slots of one thread in shared memory: slot r of thread t at base[r * GCB_BLOCK + t]
struct SmemSlots {
    u64* base;
    __device__ __forceinline__ void put(int r, u64 t) { base[r * GCB_BLOCK] = t; }
    __device__ __forceinline__ u64 get(int r) const { return base[r * GCB_BLOCK]; }
    __device__ __forceinline__ void replace(int r, u64, u64 t) { base[r * GCB_BLOCK] = t; }
};

// list offsets of one thread's pieces in shared memory
struct SmemOffs {
    uint16_t* base;
    __device__ __forceinline__ void set(int r, int v) { base[r * GCB_BLOCK] = (uint16_t)v; }
    __device__ __forceinline__ int get(int r) const { return base[r * GCB_BLOCK]; }
};

// ATTACK: get_possible_moves(attack=True) -- the attack / defence pseudo-move list (lib.rs:928-933, 1089-1104, 1147-1174).
// Both kinds go through the same two stages: one 64-bit target set per own piece into the thread's shared-memory slots
// (type-major loops), then the type-major ordered decode.
#ifndef GCB_MOVEGEN_MIN_BLOCKS
#define GCB_MOVEGEN_MIN_BLOCKS 6  // measured: 6 resident blocks per SM (80 registers) beat 7-8 (spills) and the compiler default
#endif
template <bool ATTACK>
__global__ void __launch_bounds__(GCB_BLOCK, GCB_MOVEGEN_MIN_BLOCKS) k_movegen(int n, gcb_positions pos, int castles_only,
                                                       uint16_t* __restrict__ actions, int stride,
                                                       int32_t* __restrict__ counts, uint8_t* __restrict__ incheck) {
    __shared__ u64 s_slots[GCB_SLOTS * GCB_BLOCK];
    __shared__ uint16_t s_offs[GCB_SLOTS * GCB_BLOCK];
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ulonglong2 a = reinterpret_cast<const ulonglong2*>(pos.bb01)[i], c = reinterpret_cast<const ulonglong2*>(pos.bb23)[i];
    Board b = {a.x, a.y, c.x, c.y};
    const int white = pos.player[i] == 0;
    const u32 rights = mask_rights(b, pos.rights[i]);  // convert_py_state -> State::new, lib.rs:1267-1274
    bool chk = false;
    int cnt;
    SmemSlots slots = {s_slots + threadIdx.x};
    SmemOffs offs = {s_offs + threadIdx.x};
    ListOut out = {actions + (size_t)i * stride, stride};
    if (ATTACK) cnt = gen_attack_list(b, white, slots, offs, out);
    else cnt = gen_legal_list(b, white, rights, slots, offs, out, &chk);
    if (castles_only) {  // get_castle_moves, lib.rs:1482-1500: the castle tail of the same list
        uint16_t* l = actions + (size_t)i * stride;
        int m = 0, lim = cnt < stride ? cnt : stride;
        for (int k = 0; k < lim; k++) {
            uint16_t v = l[k];
            if (v >= 4096) l[m++] = v;
        }
        cnt = m;
    }
    counts[i] = cnt;
    if (incheck) incheck[i] = chk;
}

__global__ void __launch_bounds__(GCB_BLOCK) k_next_state(int n, gcb_positions pos, const int32_t* __restrict__ actions,
                                                          gcb_positions out, uint8_t* __restrict__ checks,
                                                          int32_t* __restrict__ reward, int8_t* __restrict__ status) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ulonglong2 a = reinterpret_cast<const ulonglong2*>(pos.bb01)[i], c = reinterpret_cast<const ulonglong2*>(pos.bb23)[i];
    Board b = {a.x, a.y, c.x, c.y};
    const int black = pos.player[i] != 0;
    u32 rights = mask_rights(b, pos.rights[i]);  // Q21: masked by the INPUT board, then cloned
    Board nb = b;
    int st;
    bool irr;
    int r = apply_action(nb, rights, !black, actions[i], &st, &irr);
    if (st) nb = b, r = 0;
    reinterpret_cast<ulonglong2*>(out.bb01)[i] = make_ulonglong2(nb.t0, nb.t1);
    reinterpret_cast<ulonglong2*>(out.bb23)[i] = make_ulonglong2(nb.t2, nb.w);
    if (out.player) out.player[i] = st ? black : !black;  // lib.rs:779-780
    if (out.rights) out.rights[i] = (uint8_t)rights;
    const u32 chk = check_flags(nb);  // update_state, lib.rs:1440
    if (checks) checks[i] = (uint8_t)chk;
    if (reward) reward[i] = r;
    // status 1: the move was applied and BOTH kings are in check afterwards -- the reference prints, sets a Python exception
    // and still returns the state (lib.rs:1442-1446, Q19); reported so that a binding can raise like CPython does
    if (status) status[i] = (int8_t)(st ? st : (chk == 3u ? 1 : 0));
}

__global__ void __launch_bounds__(GCB_BLOCK) k_update_state(int n, gcb_positions pos, uint8_t* __restrict__ rights_out,
                                                            uint8_t* __restrict__ checks) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ulonglong2 a = reinterpret_cast<const ulonglong2*>(pos.bb01)[i], c = reinterpret_cast<const ulonglong2*>(pos.bb23)[i];
    Board b = {a.x, a.y, c.x, c.y};
    if (rights_out) rights_out[i] = (uint8_t)mask_rights(b, pos.rights[i]);
    if (checks) checks[i] = (uint8_t)check_flags(b);
}

// possible_actions of the 32 envs of a warp as BIT masks, rows of `stride_words` 64-bit words (include/gymchess_b200.h,
// gcb_env_legal_bitmask): word `from` of an env is exactly the legal-target set of the piece on that square, word 64 holds
// the castles -- at most 17 of the 65 words are non-zero.  The rows of a warp's envs are contiguous, so the warp first
// ZERO-FILLS the whole span with coalesced 16-byte stores, and after a warp barrier (which orders the two stores to the same
// address) every thread SCATTERS its own env's non-zero words: one 8-byte store per own piece, slot index = a running count
// along the ascending square scan.  ~10x fewer instructions than assembling the rows word by word with shuffles, which
// matters because the step kernel that calls this is bound by the integer pipe.  `slots`: the calling thread's piece slots.
__device__ __forceinline__ void write_bits_rows(u64* __restrict__ out, int stride_words, int e0, int e_end, bool active, int e,
                                                u64 own, u32 cword, const SlotRef& slots, int lane) {
    const int nrows = e_end - e0 < 32 ? e_end - e0 : 32;
    if (nrows <= 0) return;
    u64* const span = out + (size_t)e0 * (size_t)stride_words;
    const int words = nrows * stride_words;
    if (((stride_words & 1) == 0) && ((reinterpret_cast<uintptr_t>(span) & 15) == 0)) {
        ulonglong2* q = reinterpret_cast<ulonglong2*>(span);
        for (int i = lane; i < words / 2; i += 32) GCB_BITS_ST(q + i, make_ulonglong2(0ULL, 0ULL));
    } else {
        for (int i = lane; i < words; i += 32) GCB_BITS_ST(span + i, 0ULL);
    }
    __syncwarp();
    if (active) {
        u64* const row = out + (size_t)e * (size_t)stride_words;
        TgtSink src(slots, nullptr);
        int r = 0;
        for (u64 t = own; t; t &= t - 1, r++) {
            const u64 T = src.get(r);
            if (T) GCB_BITS_ST(row + gcb_lsb(t), T);
        }
        if (cword) GCB_BITS_ST(row + 64, (u64)cword);
    }
}

// One UNIT of step work of one block: the envs [e, ...) of the block's tile run `nsteps` consecutive steps.
// TILE selects where the piece slots live while the unit runs:
//   0  in their resident place (any number of slots; the generic path),
//   1  multi-step units: staged into a shared-memory tile at the start, copied back at the end; slot accesses are plain
//      LDS / STS with constant strides, the small geometry tables sit next to them in shared memory,
//   2  single-step units: nothing is staged in -- the step's pick / validity test reads its ONE slot from the resident
//      array -- but the generation still writes the new legal set into the tile (the cheap code path of 1) and the tile is
//      copied out row by row at the end, only for envs whose legal set was rewritten.
// SELFPLAY: opponent "none" is a launch-time fact, so the self-play kernels carry no bot code (a smaller hot loop: the
// kernel's instruction footprint is what it waits for most).
template <int MODE, int TILE, bool SELFPLAY>
__device__ __forceinline__ void run_unit(const EnvView& v, StepIO io, const int e, const int nsteps, u64* s_slots, u64* s_geom,
                                         CountBytes* s_counts) {
    const int lane = threadIdx.x & 31;
    bool active = e < io.e_end;
    if (MODE == MODE_RESET && active && io.in && !reinterpret_cast<const uint8_t*>(io.in)[e]) active = false;  // masked reset
    long long acc = 0;  // lane k accumulates statistics counter k of this warp
    EnvRegs s;          // the env's state stays in registers from step to step
    u32 ep = 0;
    // the block's copy of the small geometry tables: its loads are issued first and stored after the state loads have been
    // issued too, so that the two latencies overlap (a single-step launch pays this start-up once per step)
    u64 gw[(GCB_SGEOM_WORDS + GCB_BLOCK - 1) / GCB_BLOCK];
    if (TILE) {
#pragma unroll
        for (int k = 0; k < (GCB_SGEOM_WORDS + GCB_BLOCK - 1) / GCB_BLOCK; k++) {
            const int i = threadIdx.x + k * GCB_BLOCK;
            gw[k] = i < GCB_SGEOM_WORDS ? GeomShared::source_word(i) : 0ULL;
        }
    }
    u32 input = 0;
    if (active) {
        input = step_input<MODE>(io, e);  // (MODE_RESET's mask byte was read above; sampled runs have no input)
        env_load(v, e, s, ep);
    }
    if (TILE) {
#pragma unroll
        for (int k = 0; k < (GCB_SGEOM_WORDS + GCB_BLOCK - 1) / GCB_BLOCK; k++) {
            const int i = threadIdx.x + k * GCB_BLOCK;
            if (i < GCB_SGEOM_WORDS) s_geom[i] = gw[k];
        }
        __syncthreads();
    }
    const SlotRef gsr = resident_slots(v, e < io.e_end ? e : io.e_begin);
    const SlotRef tsr = {s_slots + threadIdx.x, (unsigned)GCB_BLOCK, GCB_SLOTS, true};
    if (TILE == 1 && active) {
        const int np = gcb_popc(stm_pieces(s));
        for (int r = 0; r < np && r < GCB_SLOTS; r++) s_slots[r * GCB_BLOCK + threadIdx.x] = __ldcs(gsr.base + (unsigned)r * gsr.stride);
    }
    const SlotRef sr = TILE ? tsr : gsr;
    const GeomShared sgeo = {s_geom};
    // at most 16 pieces of either colour (always, from the standard start position: pieces only leave the board): the
    // generation then stores its slots without bounds tests for the whole unit
    const bool small = (TILE || v.slots == GCB_SLOTS) && active && gcb_popc(s.b.w) <= GCB_SLOTS && gcb_popc(bb_occ(s.b) & ~s.b.w) <= GCB_SLOTS;
    (void)small;
    bool wrote = TILE == 1;  // TILE 2: does the tile hold this env's legal set (was it rewritten by this unit)?
#pragma unroll 1
    for (int t = 0; t < nsteps; t++) {
        StepStats st;
        st.clear();
        if (active) {
            // the first pick of a single-step unit reads the resident slot; everything later goes through the tile
            const SlotRef& pick = (TILE == 2 && !wrote) ? gsr : sr;
            if (TILE) {
#if GCB_FAST_SINK
                if (small) env_step_regs<MODE, SELFPLAY, true, TILE == 1>(v, io, e, s, ep, st, &s_counts[threadIdx.x], sr, pick, sgeo, input);
                else
#endif
                    env_step_regs<MODE, SELFPLAY, false, TILE == 1>(v, io, e, s, ep, st, &s_counts[threadIdx.x], sr, pick, sgeo, input);
            } else {
#if GCB_FAST_SINK && GCB_FAST_GENERIC
                if (small) env_step_regs<MODE, SELFPLAY, true, false>(v, io, e, s, ep, st, &s_counts[threadIdx.x], sr, pick, GeomGlobal(), input);
                else
#endif
                    env_step_regs<MODE, SELFPLAY, false, false>(v, io, e, s, ep, st, &s_counts[threadIdx.x], sr, pick, GeomGlobal(), input);
            }
            wrote = wrote || st.wrote_slots;
        }
        if (MODE != MODE_RESET) {
            // episode statistics: warp reduce (REDUX), lane k keeps counter k.  The three counters every step touches are
            // fields of one word wide enough for a warp sum (one REDUX for all three); the rare events (an episode ends,
            // an invalid action, an overflow) are only looked at when some lane of the warp has one
            const u32 f = st.f;
            const u32 hot = __reduce_add_sync(0xffffffffu, f & SF_HOT_MASK);
            const int t_reward = __reduce_add_sync(0xffffffffu, st.reward), t_legal = __reduce_add_sync(0xffffffffu, st.legal);
            const int t_scan = __reduce_add_sync(0xffffffffu, st.scan), t_window = __reduce_add_sync(0xffffffffu, st.window);
            // lane k picks counter k: a chain of selects (a switch on the lane id would run its cases one by one)
            long long mine = 0;
#define GCB_PICK(k_, v_) mine = lane == (k_) ? (long long)(v_) : mine
            GCB_PICK(ST_STEPS, hot & 127u), GCB_PICK(ST_PLIES, (hot >> 7) & 255u), GCB_PICK(ST_INCHECK, (hot >> 15) & 127u);
            GCB_PICK(ST_REWARD, t_reward), GCB_PICK(ST_LEGAL, t_legal), GCB_PICK(ST_HISTSCAN, t_scan), GCB_PICK(ST_WINDOW, t_window);
            if (__any_sync(0xffffffffu, (f >> SF_RARE_SHIFT) != 0u)) {
                const u32 r = f >> SF_RARE_SHIFT;  // episodes, mates, repetitions, caps | wedged, invalid, hist_overflow(2), slot_overflow(2)
                const u32 w0 = (r & 1u) | ((r & 2u) << 7) | ((r & 4u) << 14) | ((r & 8u) << 21);
                const u32 w1 = ((r >> 4) & 1u) | (((r >> 5) & 1u) << 8) | (((r >> 6) & 3u) << 16) | (((r >> 8) & 3u) << 24);
                const u32 r0 = __reduce_add_sync(0xffffffffu, w0), r1 = __reduce_add_sync(0xffffffffu, w1);
                GCB_PICK(ST_EPISODES, r0 & 255u), GCB_PICK(ST_MATES, (r0 >> 8) & 255u), GCB_PICK(ST_REPS, (r0 >> 16) & 255u);
                GCB_PICK(ST_CAPS, r0 >> 24), GCB_PICK(ST_WEDGED, r1 & 255u), GCB_PICK(ST_INVALID, (r1 >> 8) & 255u);
                GCB_PICK(ST_HISTOVF, (r1 >> 16) & 255u), GCB_PICK(ST_SLOTOVF, r1 >> 24);
            }
#undef GCB_PICK
            acc += mine;
        }
        io.tick++;
        if (io.act_out) io.act_out += v.N;
        if (io.bot_out) io.bot_out += v.N;
    }
    if (active) {
        env_store(v, e, s, ep);
        if (TILE && wrote) {  // slots of the side to move back to their resident place
            const int np = gcb_popc(stm_pieces(s));
            for (int r = 0; r < np && r < GCB_SLOTS; r++) __stcs(v.tgt + (size_t)r * v.N + e, s_slots[r * GCB_BLOCK + threadIdx.x]);
        }
    }
    // learner-facing output of the step itself (SURVEY.md 8(f)1): possible_actions of the state the step leaves behind as
    // the 65-word bit mask, written while the legal set still sits in the shared-memory tile (no second kernel, no re-read;
    // envs whose legal set the step did not touch read it from its resident place)
    if (io.bits_out) {
        u64 own = 0;
        u32 cword = 0;
        if (active) own = stm_pieces(s), cword = castle_word(s);
        write_bits_rows(io.bits_out, io.bits_stride, e - lane, io.e_end, active, e, own, cword, (TILE && wrote) ? sr : gsr, lane);
    }
    // one coalesced fire-and-forget add to the warp's own row -- no contention and no block barrier.  A warp that lies wholly
    // past the env range (the idle warps of the last block) owns no row: stat_rows has ceil(N / 32) of them.
    if (MODE != MODE_RESET && lane < ST_USED) {
#if !defined(GCB_SELFTEST_OOB)  // (the self-test build of the checked library leaves the predicate out on purpose)
        if ((e & ~31) < io.e_end)
#endif
        {
            const size_t row = (size_t)(e >> 5);
            GCB_CHK(row < (size_t)v.stat_nrows, CHK_STAT_ROW);
            // (a reduction without a return value: the warp does not wait for the row; the row is this warp's own)
            atomicAdd(reinterpret_cast<unsigned long long*>(v.stat_rows + row * ST_COUNT + lane), (unsigned long long)acc);
        }
    }
}

// one unit per block: the envs [io.e_begin, io.e_end), io.nsteps steps each (one for everything but the sampled mode)
template <int MODE, int TILE = 0, bool SELFPLAY = false>
__global__ void __launch_bounds__(GCB_BLOCK, (MODE == MODE_SAMPLED && TILE == 1) ? GCB_SAMPLED_MIN_BLOCKS : GCB_STEP_MIN_BLOCKS)
    k_env_step(EnvView v, StepIO io) {  // (5 resident blocks at 96 registers for the multi-step tile kernel, 6 at 80 for the rest)
    __shared__ CountBytes s_counts[GCB_BLOCK];
    __shared__ u64 s_slots[TILE ? GCB_SLOTS * GCB_BLOCK : 1];
    __shared__ u64 s_geom[TILE ? GCB_SGEOM_WORDS : 1];
    run_unit<MODE, TILE, SELFPLAY>(v, io, io.e_begin + blockIdx.x * GCB_BLOCK + threadIdx.x, MODE == MODE_SAMPLED ? io.nsteps : 1,
                                   s_slots, s_geom, s_counts);
}

// totals = column sums of the per-warp rows (one block; deterministic order)
__global__ void k_stats_reduce(const u64* __restrict__ rows, int nrows, u64* __restrict__ out) {
    __shared__ u64 s[32][ST_COUNT + 1];
    const int k = threadIdx.x & 15, part = threadIdx.x >> 4;  // 512 threads: 32 partial sums per counter
    u64 acc = 0;
    for (int r = part; r < nrows; r += 32) acc += rows[(size_t)r * ST_COUNT + k];
    s[part][k] = acc;
    __syncthreads();
    if (threadIdx.x < ST_COUNT) {
        u64 t = 0;
        for (int p = 0; p < 32; p++) t += s[p][threadIdx.x];
        out[threadIdx.x] = t;
    }
}

__global__ void k_make_templates(int n, const int8_t* __restrict__ boards, ulonglong2* bb01, ulonglong2* bb23, u64* meta,
                                 u64* zkey, u64* tgt, ulonglong2* cnt, int slots) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    make_template_one(i, boards, bb01, bb23, meta, zkey, tgt, cnt, slots);
}

__global__ void __launch_bounds__(GCB_BLOCK) k_env_import(EnvView v, const int8_t* __restrict__ boards,
                                                          const int8_t* __restrict__ players, const uint8_t* __restrict__ rights4,
                                                          const int32_t* __restrict__ move_count, const uint8_t* __restrict__ mask,
                                                          u64 tick) {
    __shared__ CountBytes s_counts[GCB_BLOCK];
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.N) return;
    if (mask && !mask[e]) return;
    alignas(16) int8_t m[64];
    const int4* src = reinterpret_cast<const int4*>(boards + (size_t)e * 64);
#pragma unroll
    for (int k = 0; k < 4; k++) *reinterpret_cast<int4*>(m + 16 * k) = __ldg(src + k);
    const uchar4 q = reinterpret_cast<const uchar4*>(rights4)[e];
    const u32 rights = (q.x ? RT_WK : 0) | (q.y ? RT_WQ : 0) | (q.z ? RT_BK : 0) | (q.w ? RT_BQ : 0);
    StepStats st;
    st.clear();
    env_import_one(v, e, m, players[e], rights, move_count ? move_count[e] : 0, st, &s_counts[threadIdx.x]);
}

// gcb_env_clone, one warp per destination row d (env_clone_* of env_core.cuh split among the lanes): lane 0 copies the ~70 B
// of per-env words and broadcasts the source's generation and window length, lane r copies piece slot r (slot-major: the
// lanes of neighbouring warps fill the same 32-byte sectors), and when the source's window is non-empty all 32 lanes sweep
// its 2H-entry table, 16 B per lane and load, eight loads in flight per lane before any store, writing only the live entries
// (retagged to the destination's new generation).  is_src (CHECKED build, in-object clones only): 1 where a row is the source
// of some selected destination (k_env_clone_mark).
#define GCB_CLONE_BATCH 8
__global__ void __launch_bounds__(GCB_BLOCK) k_env_clone(EnvView dst, EnvView src, const int32_t* __restrict__ index,
                                                         const uint8_t* __restrict__ is_src) {
    const int d = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (d >= dst.N) return;
    const int i = __ldg(index + d);
    if (i < 0) return;
    GCB_CHK(i < src.N, CHK_CLONE_INDEX);
    if (i >= src.N) return;
    (void)is_src;
#if defined(GCB_CHECKED)
    if (is_src) GCB_CHK(!is_src[d], CHK_CLONE_ALIAS);
#endif
    u32 sgen = 0, G = 0;
    int hist = 0;
    if (lane == 0) G = env_clone_words(dst, d, src, i, &sgen, &hist);
    for (int r = lane; r < dst.slots; r += 32) env_clone_slot(dst, d, src, i, r);
    sgen = __shfl_sync(0xffffffffu, sgen, 0), G = __shfl_sync(0xffffffffu, G, 0), hist = __shfl_sync(0xffffffffu, hist, 0);
    if (hist == 0) return;
    const unsigned H2 = (unsigned)src.hist_mask + 1u;  // 2H >= 16 entries, a multiple of 16
    const ulonglong2* from = src.rep + (size_t)i * H2;
    ulonglong2* to = dst.rep + (size_t)d * H2;
#pragma unroll 1
    for (unsigned k0 = lane; k0 < H2; k0 += 32u * GCB_CLONE_BATCH) {
        ulonglong2 en[GCB_CLONE_BATCH];
#pragma unroll
        for (int b = 0; b < GCB_CLONE_BATCH; b++) {
            const unsigned k = k0 + 32u * b;
            en[b] = k < H2 ? __ldcs(&from[k]) : make_ulonglong2(0ULL, 0ULL);
        }
#pragma unroll
        for (int b = 0; b < GCB_CLONE_BATCH; b++) {
            const unsigned k = k0 + 32u * b;
            if (k < H2 && rep_clone_entry(en[b], sgen, G)) __stcs(&to[k], en[b]);
        }
    }
}

// CHECKED build, in-object clone: mark the source row of every selected destination (the aliasing check of k_env_clone)
__global__ void k_env_clone_mark(int n, int src_n, const int32_t* __restrict__ index, uint8_t* __restrict__ is_src) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n) return;
    const int i = index[d];
    if (i >= 0 && i < src_n) is_src[i] = 1;
}

__global__ void k_init_zobrist(u64* tab) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < GCB_ZOB_ENTRIES) fill_zobrist_entry(tab, i);
}

__global__ void __launch_bounds__(GCB_BLOCK) k_env_export(EnvView v, int8_t* __restrict__ boards, int32_t* __restrict__ info) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.N) return;
    alignas(16) int8_t m[64];
    alignas(16) int32_t inf[16];
    env_export_one(v, e, boards ? m : nullptr, info ? inf : nullptr);
    if (boards) {
        int4* dst = reinterpret_cast<int4*>(boards + (size_t)e * 64);
#pragma unroll
        for (int k = 0; k < 4; k++) dst[k] = *reinterpret_cast<int4*>(m + 16 * k);
    }
    if (info) {
        int4* o = reinterpret_cast<int4*>(info + (size_t)e * 16);
#pragma unroll
        for (int k = 0; k < 4; k++) o[k] = *reinterpret_cast<int4*>(inf + 4 * k);
    }
}

// ChessEnvV2.possible_actions for every env: the reference-ordered list decoded from the resident piece slots
__global__ void __launch_bounds__(GCB_BLOCK) k_env_legal_list(EnvView v, uint16_t* __restrict__ actions, int stride,
                                                              int32_t* __restrict__ counts) {
    __shared__ uint16_t s_offs[GCB_SLOTS * GCB_BLOCK];
    __shared__ u64 s_stage[GCB_SLOTS * GCB_BLOCK];
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.N) return;
    SmemOffs offs = {s_offs + threadIdx.x};
    ListOut out = {actions + (size_t)e * stride, stride};
    const int n = env_legal_list_one(v, e, offs, out, s_stage + threadIdx.x, (unsigned)GCB_BLOCK);
    if (counts) counts[e] = n;
}

struct MaskOut {
    uint8_t* m;
    __device__ __forceinline__ void put(int, int action) { m[action] = 1; }
};
__global__ void __launch_bounds__(GCB_BLOCK) k_env_legal_mask(EnvView v, uint8_t* __restrict__ mask) {
    __shared__ uint16_t s_offs[GCB_SLOTS * GCB_BLOCK];
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= v.N) return;
    SmemOffs offs = {s_offs + threadIdx.x};
    MaskOut mo = {mask + (size_t)e * 4101};
    env_legal_list_one(v, e, offs, mo);
}

// possible_actions as a BIT mask: bit a of a 4101-bit vector per env, in 65 little-endian 64-bit words -- word `from`
// (0..63) is exactly the resident legal-target set of the piece on that square, word 64 holds the four castle actions
// (bit a - 4096).  A streaming kernel (HBM-bound): the thread that owns an env stages its piece slots in shared memory,
// then the warp writes the 32 rows one after the other, lane = from-square, as coalesced 256-byte stores.
// (The stand-alone mask kernel is a pure stream bound by HBM: here every row word is written exactly ONCE, assembled by the
// warp -- the thread that owns an env stages its piece slots in shared memory, then the warp writes the 32 rows one after
// the other, lane = from-square, as coalesced 256-byte stores.  The zero-fill + scatter writer of the step kernels costs
// ~10x fewer instructions but touches the non-zero sectors twice: 111-124 us against 78 us for this kernel alone.)
__global__ void __launch_bounds__(GCB_BLOCK) k_env_legal_bits(EnvView v, u64* __restrict__ out, int stride_words, int e_begin, int e_end) {
    __shared__ u64 s_slots[GCB_SLOTS * GCB_BLOCK];
    const int e = e_begin + blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, wbase = threadIdx.x & ~31;
    u64 own = 0;
    u32 cword = 0;
    if (e < e_end) {
        EnvRegs s;
        ulonglong2 a = __ldcs(&v.bb01[e]), c = __ldcs(&v.bb23[e]);
        s.b.t0 = a.x, s.b.t1 = a.y, s.b.t2 = c.x, s.b.w = c.y;
        unpack_meta(__ldcs(&v.meta[e]), s);
        own = stm_pieces(s), cword = castle_word(s);
        const int np = gcb_popc(own);
        for (int r = 0; r < np && r < GCB_SLOTS; r++) s_slots[r * GCB_BLOCK + threadIdx.x] = __ldcs(v.tgt + (size_t)r * v.N + e);
    }
    __syncwarp();
    const int e0 = e - lane;
#pragma unroll 1
    for (int p = 0; p < 32 && e0 + p < e_end; p++) {
        const u64 own_p = __shfl_sync(0xffffffffu, own, p);
        const u32 c_p = __shfl_sync(0xffffffffu, cword, p);
        u64* row = out + (size_t)(e0 + p) * (size_t)stride_words;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int sq = lane + 32 * h;
            u64 T = 0;
            if ((own_p >> sq) & 1ULL) {
                const int r = gcb_popc(own_p & ((1ULL << sq) - 1));
                T = r < GCB_SLOTS ? s_slots[r * GCB_BLOCK + wbase + p] : (r < v.slots ? __ldcs(v.tgt + (size_t)r * v.N + e0 + p) : 0ULL);
            }
            __stcs(row + sq, T);
        }
        if (lane == 0) __stcs(row + 64, (u64)c_p);
    }
}

// gcb_env_sample_policy, per-env rule in env_core.cuh (policy_*; env_policy_sample_one is the serial form).  A warp takes
// the 32 envs of its lanes: each thread loads its env's board, meta and random word and stages its piece slots in shared
// memory (slot-major, coalesced, as in k_env_legal_bits); then the warp samples the 32 envs one after the other with
// lane = action.  Lane l owns from-squares 2l and 2l+1, so an inclusive warp scan of the lanes' target counts numbers L in
// code order; in round j lane l decodes action k = 32j + l (owner lane by a 5-step binary search over the scan, target by
// gcb_select64) and loads that ONE logit, so the ~23 gathers of an env are in flight together.  Three passes over L: max,
// sum, prefix-sum selection; the first round's logits stay in registers, later rounds re-read theirs.
// GCB_POLICY_THREAD = 1 builds the measured alternative instead: one thread per env runs the serial form (DESIGN 3.10).
#ifndef GCB_POLICY_THREAD
#define GCB_POLICY_THREAD 0
#endif
template <int DT>
__global__ void __launch_bounds__(GCB_BLOCK) k_env_policy_sample(EnvView v, const void* __restrict__ logits, long long row_stride,
                                                                 float temp, const u32* __restrict__ words,
                                                                 int32_t* __restrict__ act, float* __restrict__ logp) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31, wbase = threadIdx.x & ~31;
#if GCB_POLICY_THREAD
    if (e < v.N) env_policy_sample_one<DT>(v, e, logits, row_stride, temp, words, act, logp);
    (void)lane, (void)wbase;
#else
    __shared__ u64 s_slots[GCB_SLOTS * GCB_BLOCK];
    const unsigned FULL = 0xffffffffu;
    u64 own = 0;
    u32 cword = 0, word = 0;
    if (e < v.N) {
        EnvRegs s;
        u32 ep;
        policy_load(v, e, s, ep);
        own = stm_pieces(s), cword = castle_word(s);
        if (temp != 0.f) word = words ? __ldg(words + e) : policy_word(v, e, s, ep);
        const int np = gcb_popc(own);
        for (int r = 0; r < np && r < GCB_SLOTS; r++) s_slots[r * GCB_BLOCK + threadIdx.x] = __ldcs(v.tgt + (size_t)r * v.N + e);
    }
    __syncwarp();
    const int e0 = e - lane;
    int my_act = ACT_RESIGN;
    float my_logp = 0.f;
#pragma unroll 1
    for (int p = 0; p < 32 && e0 + p < v.N; p++) {
        const int ep_ = e0 + p;
        const u64 own_p = __shfl_sync(FULL, own, p);
        const u32 cw = __shfl_sync(FULL, cword, p);
        const void* row = policy_row<DT>(logits, row_stride, ep_);
        auto slot = [&](int r) -> u64 {
            return r < GCB_SLOTS ? s_slots[r * GCB_BLOCK + wbase + p] : (r < v.slots ? __ldcs(v.tgt + (size_t)r * v.N + ep_) : 0ULL);
        };
        const int sqa = 2 * lane, ra = gcb_popc(own_p & ((1ULL << sqa) - 1));
        const bool ha = (own_p >> sqa) & 1ULL, hb = (own_p >> (sqa + 1)) & 1ULL;
        const u64 Ta = ha ? slot(ra) : 0ULL, Tb = hb ? slot(ra + (int)ha) : 0ULL;
        const int ca = gcb_popc(Ta), c = ca + gcb_popc(Tb);
        int incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(FULL, incl, d);
            if (lane >= d) incl += t;
        }
        const int nsq = __shfl_sync(FULL, incl, 31), n = nsq + gcb_popc((u64)cw);
        // the code of action k of L (all 32 lanes call it; -1 for k >= n)
        auto code_at = [&](int k) -> int {
            int pos = 0;  // the owner lane: the number of lanes whose inclusive count is <= k
#pragma unroll
            for (int b = 16; b; b >>= 1)
                if (__shfl_sync(FULL, incl, pos + b - 1) <= k) pos += b;
            const int excl = __shfl_sync(FULL, incl - c, pos), oca = __shfl_sync(FULL, ca, pos);
            const u64 oTa = __shfl_sync(FULL, Ta, pos), oTb = __shfl_sync(FULL, Tb, pos);
            if (k < nsq) {
                const int i = k - excl;
                return i < oca ? 128 * pos + gcb_select64(oTa, i) : 128 * pos + 64 + gcb_select64(oTb, i - oca);
            }
            return k < n ? 4096 + gcb_select64((u64)cw, k - nsq) : -1;
        };
        const int a0 = code_at(lane);
        int pick = -1;
        float lp = 0.f;
        if (temp == 0.f) {
            float best = -INFINITY;
            if (a0 >= 0) policy_argmax(policy_logit<DT>(row, a0), a0, best, pick);
            for (int base = 32; base < n; base += 32) {
                const int a = code_at(base + lane);
                if (a >= 0) policy_argmax(policy_logit<DT>(row, a), a, best, pick);
            }
#pragma unroll
            for (int d = 16; d; d >>= 1) {  // warp argmax: the larger logit, then the lower code
                const float ob = __shfl_xor_sync(FULL, best, d);
                const int oi = __shfl_xor_sync(FULL, pick, d);
                if (oi >= 0 && (pick < 0 || ob > best || (ob == best && oi < pick))) best = ob, pick = oi;
            }
        } else {
            const float z0 = a0 >= 0 ? policy_logit<DT>(row, a0) / temp : 0.f;
            float m = a0 >= 0 && z0 > -INFINITY ? z0 : -INFINITY;
            for (int base = 32; base < n; base += 32) {
                const int a = code_at(base + lane);
                if (a >= 0) {
                    const float z = policy_logit<DT>(row, a) / temp;
                    if (z > m) m = z;
                }
            }
#pragma unroll
            for (int d = 16; d; d >>= 1) {
                const float o = __shfl_xor_sync(FULL, m, d);
                if (o > m) m = o;
            }
            if (m > -INFINITY) {
                float Z = a0 >= 0 ? expf(z0 - m) : 0.f;
                for (int base = 32; base < n; base += 32) {
                    const int a = code_at(base + lane);
                    if (a >= 0) Z += expf(policy_logit<DT>(row, a) / temp - m);
                }
#pragma unroll
                for (int d = 16; d; d >>= 1) Z += __shfl_xor_sync(FULL, Z, d);
                Z = __shfl_sync(FULL, Z, 0);  // (lanes may round the butterfly differently: lane 0's sum for all)
                const float target = policy_u(__shfl_sync(FULL, word, p)) * Z;
                float carry = 0.f, zp = 0.f;
                int last = -1;
                for (int base = 0; base < n && pick < 0; base += 32) {
                    const int a = base == 0 ? a0 : code_at(base + lane);
                    const float z = base == 0 ? z0 : (a >= 0 ? policy_logit<DT>(row, a) / temp : 0.f);
                    const float w = a >= 0 ? expf(z - m) : 0.f;
                    float pre = w;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const float t = __shfl_up_sync(FULL, pre, d);
                        if (lane >= d) pre += t;
                    }
                    pre += carry;
                    const unsigned hit = __ballot_sync(FULL, a >= 0 && pre > target), pos = __ballot_sync(FULL, a >= 0 && w > 0.f);
                    if (hit) {
                        pick = __shfl_sync(FULL, a, __ffs(hit) - 1), zp = __shfl_sync(FULL, z, __ffs(hit) - 1);
                    } else if (pos) {  // (the last a with w > 0 so far: the pick if rounding leaves no prefix sum above target)
                        last = __shfl_sync(FULL, a, 31 - __clz(pos)), zp = __shfl_sync(FULL, z, 31 - __clz(pos));
                    }
                    carry = __shfl_sync(FULL, pre, 31);
                }
                if (pick < 0) pick = last;
                lp = zp - m - logf(Z);
            }
        }
        if (lane == p) my_act = pick < 0 ? ACT_RESIGN : pick, my_logp = pick < 0 ? 0.f : lp;
    }
    if (e < v.N) {
        act[e] = my_act;
        if (logp) logp[e] = my_logp;
    }
#endif
}

// gcb_env_encode, per-env rule in env_core.cuh (env_encode_masks; env_encode_one is the serial form).  The output rows of the
// 32 envs of a warp are ONE contiguous span of 32 x 19 x 64 elements.  Each lane puts its env's 19 masks into shared memory,
// env-major, so that mask word w of the warp holds elements [64 w, 64 w + 64) of the span; then the warp writes the span
// flat, one 16-byte vector per lane per iteration (4 / 8 / 16 elements from one broadcast mask word; a vector never straddles
// two words), with streaming stores.  A pure write stream: the state it reads is 40 B per env plus the table probe of envs
// with a non-empty window.
template <int DT>
__device__ __forceinline__ uint4 encode_vec(u32 bits) {  // the 16 / 8 / 4 low bits of `bits` -> one 16-byte vector
    uint4 r;
    if (DT == 2) {  // bit i of a nibble -> byte i: the copies of the nibble shifted by 7 do not overlap
        r.x = ((bits & 15u) * 0x204081u) & 0x01010101u, r.y = (((bits >> 4) & 15u) * 0x204081u) & 0x01010101u;
        r.z = (((bits >> 8) & 15u) * 0x204081u) & 0x01010101u, r.w = ((bits >> 12) * 0x204081u) & 0x01010101u;
    } else if (DT == 1) {  // two bf16 per word, 1.0 = 0x3F80
        r.x = (bits & 1u) * 0x3F80u + ((bits >> 1) & 1u) * 0x3F800000u, r.y = ((bits >> 2) & 1u) * 0x3F80u + ((bits >> 3) & 1u) * 0x3F800000u;
        r.z = ((bits >> 4) & 1u) * 0x3F80u + ((bits >> 5) & 1u) * 0x3F800000u, r.w = ((bits >> 6) & 1u) * 0x3F80u + (bits >> 7) * 0x3F800000u;
    } else {  // fp32 1.0 = 0x3F800000
        r.x = (bits & 1u) * 0x3F800000u, r.y = ((bits >> 1) & 1u) * 0x3F800000u;
        r.z = ((bits >> 2) & 1u) * 0x3F800000u, r.w = (bits >> 3) * 0x3F800000u;
    }
    return r;
}
template <int DT>
__global__ void __launch_bounds__(GCB_BLOCK) k_env_encode(EnvView v, void* __restrict__ planes, uint8_t* __restrict__ rep_out) {
    __shared__ u64 s_masks[GCB_BLOCK * OBS_PLANES];
    const int e = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
    u64* const wm = s_masks + (threadIdx.x & ~31) * OBS_PLANES;
    if (e < v.N) {
        u64 m[OBS_PLANES];
        int rep;
        env_encode_masks(v, e, m, &rep);
#pragma unroll
        for (int c = 0; c < OBS_PLANES; c++) wm[lane * OBS_PLANES + c] = m[c];
        if (rep_out) rep_out[e] = (uint8_t)rep;
    }
    if (!planes) return;
    __syncwarp();
    constexpr int V = 16 / (int)sizeof(typename EncodeElem<DT>::type), PER_ENV = OBS_PLANES * 64 / V;
    const int e0 = e - lane, nvec = min(32, v.N - e0) * PER_ENV;  // a partial last warp writes only its envs' rows
    uint4* const out = reinterpret_cast<uint4*>(planes) + (size_t)e0 * PER_ENV;
#pragma unroll 4
    for (int j = lane; j < nvec; j += 32) {
        const int k = j * V;
        const u32 bits = (u32)(wm[k >> 6] >> (k & 63)) & ((1u << V) - 1u);
        GCB_CHK((size_t)e0 * PER_ENV + (size_t)j < (size_t)v.N * PER_ENV, CHK_ENCODE_INDEX);
        __stcs(out + j, encode_vec<DT>(bits));
    }
}

// ------------------------------------------------------------------------------------------------ host side
static int need_gpu() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return fail(GCB_E_NOGPU, "no CUDA device", "this library has no CPU fallback");
    return GCB_OK;
}

extern "C" int gcb_pack(int n, const int8_t* d_boards, const int8_t* d_players, const uint8_t* d_rights4, gcb_positions out,
                        void* stream) {
    if (n < 0 || !d_boards || !out.bb01 || !out.bb23) return fail(GCB_E_ARG, "gcb_pack", "null pointer or n < 0");
    if (n == 0) return GCB_OK;
    k_pack<<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, d_boards, d_players, d_rights4, out);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_unpack(int n, gcb_positions in, int8_t* d_boards, int8_t* d_players, uint8_t* d_rights4, void* stream) {
    if (n < 0 || !in.bb01 || !in.bb23) return fail(GCB_E_ARG, "gcb_unpack", "null pointer or n < 0");
    if (n == 0) return GCB_OK;
    k_unpack<<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, in, d_boards, d_players, d_rights4);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_get_possible_moves(int n, gcb_positions pos, int attack, int castles_only, uint16_t* d_actions, int stride,
                                      int32_t* d_counts, uint8_t* d_incheck, void* stream) {
    if (n < 0 || !pos.bb01 || !pos.bb23 || !pos.player || !pos.rights || !d_actions || !d_counts || stride <= 0 || (stride & 1))
        return fail(GCB_E_ARG, "gcb_get_possible_moves", "null pointer, n < 0 or odd stride");
    if (n == 0) return GCB_OK;
    if (attack)
        k_movegen<true><<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, pos, 0, d_actions, stride, d_counts, d_incheck);
    else
        k_movegen<false><<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, pos, castles_only, d_actions, stride, d_counts,
                                                                               d_incheck);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_next_state(int n, gcb_positions pos, const int32_t* d_actions, gcb_positions out, uint8_t* d_checks,
                              int32_t* d_reward, int8_t* d_status, void* stream) {
    if (n < 0 || !pos.bb01 || !pos.bb23 || !pos.player || !pos.rights || !d_actions || !out.bb01 || !out.bb23)
        return fail(GCB_E_ARG, "gcb_next_state", "null pointer or n < 0");
    if (n == 0) return GCB_OK;
    k_next_state<<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, pos, d_actions, out, d_checks, d_reward, d_status);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_update_state(int n, gcb_positions pos, uint8_t* d_rights_out, uint8_t* d_checks, void* stream) {
    if (n < 0 || !pos.bb01 || !pos.bb23 || !pos.rights) return fail(GCB_E_ARG, "gcb_update_state", "null pointer or n < 0");
    if (n == 0) return GCB_OK;
    k_update_state<<<grid_for(n), GCB_BLOCK, 0, (cudaStream_t)stream>>>(n, pos, d_rights_out, d_checks);
    LAUNCHED();
    return GCB_OK;
}

// ---- host-buffer engine calls: one scratch arena per call (these are the convenience / binding entry points)
struct Arena {
    char* base = nullptr;
    size_t used = 0, cap = 0;
    int init(size_t bytes) {
        cap = bytes;
        return cudaMalloc(&base, bytes ? bytes : 256) == cudaSuccess ? 0 : -1;
    }
    template <class T>
    T* take(size_t count) {
        size_t off = (used + 255) & ~(size_t)255;
        used = off + count * sizeof(T);
        return reinterpret_cast<T*>(base + off);
    }
    ~Arena() {
        if (base) cudaFree(base);
    }
};
static size_t al(size_t x) { return ((x + 255) & ~(size_t)255) + 256; }

static gcb_positions arena_positions(Arena& A, int n) {
    gcb_positions p;
    p.bb01 = A.take<uint64_t>((size_t)n * 2);
    p.bb23 = A.take<uint64_t>((size_t)n * 2);
    p.player = A.take<uint8_t>(n);
    p.rights = A.take<uint8_t>(n);
    return p;
}
static size_t positions_bytes(int n) { return al((size_t)n * 16) * 2 + al(n) * 2; }

extern "C" int gcb_host_get_possible_moves(int n, const int8_t* boards, const int8_t* players, const uint8_t* rights4, int attack,
                                           int castles_only, uint16_t* actions, int stride, int32_t* counts, uint8_t* incheck) {
    if (int rc = need_gpu()) return rc;
    if (n < 0 || !boards || !players || !rights4 || !actions || !counts || stride <= 0 || (stride & 1))
        return fail(GCB_E_ARG, "gcb_host_get_possible_moves", "null pointer, n < 0 or odd stride");
    if (n == 0) return GCB_OK;
    Arena A;
    size_t bytes = al((size_t)n * 64) + al(n) + al((size_t)n * 4) + positions_bytes(n) + al((size_t)n * stride * 2) +
                   al((size_t)n * 4) + al(n);
    if (A.init(bytes)) return fail(GCB_E_NOMEM, "cudaMalloc", "scratch");
    int8_t* d_b = A.take<int8_t>((size_t)n * 64);
    int8_t* d_p = A.take<int8_t>(n);
    uint8_t* d_r = A.take<uint8_t>((size_t)n * 4);
    gcb_positions pos = arena_positions(A, n);
    uint16_t* d_a = A.take<uint16_t>((size_t)n * stride);
    int32_t* d_c = A.take<int32_t>(n);
    uint8_t* d_i = A.take<uint8_t>(n);
    CU(cudaMemcpyAsync(d_b, boards, (size_t)n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_p, players, n, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_r, rights4, (size_t)n * 4, cudaMemcpyHostToDevice, 0));
    CU(cudaMemsetAsync(d_a, 0, (size_t)n * stride * 2, 0));
    if (int rc = gcb_pack(n, d_b, d_p, d_r, pos, 0)) return rc;
    if (int rc = gcb_get_possible_moves(n, pos, attack, castles_only, d_a, stride, d_c, d_i, 0)) return rc;
    CU(cudaMemcpyAsync(actions, d_a, (size_t)n * stride * 2, cudaMemcpyDeviceToHost, 0));
    CU(cudaMemcpyAsync(counts, d_c, (size_t)n * 4, cudaMemcpyDeviceToHost, 0));
    if (incheck) CU(cudaMemcpyAsync(incheck, d_i, n, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return GCB_OK;
}

extern "C" int gcb_host_next_state(int n, const int8_t* boards, const int8_t* players, const uint8_t* rights4,
                                   const int32_t* actions, int8_t* out_boards, uint8_t* out_rights4, uint8_t* out_checks,
                                   int32_t* out_reward, int8_t* out_status) {
    if (int rc = need_gpu()) return rc;
    if (n < 0 || !boards || !players || !rights4 || !actions || !out_boards || !out_rights4 || !out_checks || !out_reward ||
        !out_status)
        return fail(GCB_E_ARG, "gcb_host_next_state", "null pointer or n < 0");
    if (n == 0) return GCB_OK;
    Arena A;
    size_t bytes = al((size_t)n * 64) * 2 + al(n) * 2 + al((size_t)n * 4) * 4 + positions_bytes(n) * 2 + al(n) * 2;
    if (A.init(bytes)) return fail(GCB_E_NOMEM, "cudaMalloc", "scratch");
    int8_t* d_b = A.take<int8_t>((size_t)n * 64);
    int8_t* d_p = A.take<int8_t>(n);
    uint8_t* d_r = A.take<uint8_t>((size_t)n * 4);
    int32_t* d_a = A.take<int32_t>(n);
    gcb_positions pos = arena_positions(A, n), out = arena_positions(A, n);
    int8_t* d_ob = A.take<int8_t>((size_t)n * 64);
    uint8_t* d_or = A.take<uint8_t>((size_t)n * 4);
    uint8_t* d_oc = A.take<uint8_t>(n);
    int32_t* d_rw = A.take<int32_t>(n);
    int8_t* d_st = A.take<int8_t>(n);
    CU(cudaMemcpyAsync(d_b, boards, (size_t)n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_p, players, n, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_r, rights4, (size_t)n * 4, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_a, actions, (size_t)n * 4, cudaMemcpyHostToDevice, 0));
    if (int rc = gcb_pack(n, d_b, d_p, d_r, pos, 0)) return rc;
    if (int rc = gcb_next_state(n, pos, d_a, out, d_oc, d_rw, d_st, 0)) return rc;
    if (int rc = gcb_unpack(n, out, d_ob, nullptr, d_or, 0)) return rc;
    CU(cudaMemcpyAsync(out_boards, d_ob, (size_t)n * 64, cudaMemcpyDeviceToHost, 0));
    CU(cudaMemcpyAsync(out_rights4, d_or, (size_t)n * 4, cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    // checks come back as 2 bytes per position (wchk, bchk) like the oracle's batch call
    uint8_t* tmp = new (std::nothrow) uint8_t[n];
    if (!tmp) return fail(GCB_E_NOMEM, "new", "host scratch");
    cudaError_t e1 = cudaMemcpy(tmp, d_oc, n, cudaMemcpyDeviceToHost);
    for (int i = 0; i < n && e1 == cudaSuccess; i++) out_checks[2 * i] = tmp[i] & 1, out_checks[2 * i + 1] = (tmp[i] >> 1) & 1;
    delete[] tmp;
    if (e1 != cudaSuccess) return fail(GCB_E_CUDA, "cudaMemcpy", cudaGetErrorString(e1));
    CU(cudaMemcpy(out_reward, d_rw, (size_t)n * 4, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(out_status, d_st, n, cudaMemcpyDeviceToHost));
    return GCB_OK;
}

extern "C" int gcb_host_update_state(int n, const int8_t* boards, const uint8_t* rights4, uint8_t* out_rights4,
                                     uint8_t* out_checks) {
    if (int rc = need_gpu()) return rc;
    if (n < 0 || !boards || !rights4 || !out_rights4 || !out_checks) return fail(GCB_E_ARG, "gcb_host_update_state", "null pointer");
    if (n == 0) return GCB_OK;
    Arena A;
    size_t bytes = al((size_t)n * 64) + al((size_t)n * 4) + positions_bytes(n) + al(n) * 2;
    if (A.init(bytes)) return fail(GCB_E_NOMEM, "cudaMalloc", "scratch");
    int8_t* d_b = A.take<int8_t>((size_t)n * 64);
    uint8_t* d_r = A.take<uint8_t>((size_t)n * 4);
    gcb_positions pos = arena_positions(A, n);
    uint8_t* d_or = A.take<uint8_t>(n);
    uint8_t* d_oc = A.take<uint8_t>(n);
    CU(cudaMemcpyAsync(d_b, boards, (size_t)n * 64, cudaMemcpyHostToDevice, 0));
    CU(cudaMemcpyAsync(d_r, rights4, (size_t)n * 4, cudaMemcpyHostToDevice, 0));
    if (int rc = gcb_pack(n, d_b, nullptr, d_r, pos, 0)) return rc;
    if (int rc = gcb_update_state(n, pos, d_or, d_oc, 0)) return rc;
    uint8_t* tmp = new (std::nothrow) uint8_t[2 * (size_t)n];
    if (!tmp) return fail(GCB_E_NOMEM, "new", "host scratch");
    cudaError_t e1 = cudaMemcpy(tmp, d_or, n, cudaMemcpyDeviceToHost);
    cudaError_t e2 = cudaMemcpy(tmp + n, d_oc, n, cudaMemcpyDeviceToHost);
    for (int i = 0; i < n; i++) {
        uint8_t r = tmp[i], c = tmp[n + i];
        out_rights4[4 * i] = r & 1, out_rights4[4 * i + 1] = (r >> 1) & 1, out_rights4[4 * i + 2] = (r >> 2) & 1,
                        out_rights4[4 * i + 3] = (r >> 3) & 1;
        out_checks[2 * i] = c & 1, out_checks[2 * i + 1] = (c >> 1) & 1;
    }
    delete[] tmp;
    if (e1 != cudaSuccess || e2 != cudaSuccess) return fail(GCB_E_CUDA, "cudaMemcpy", "update_state results");
    return GCB_OK;
}

// ------------------------------------------------------------------------------------------------ env object
struct gcb_env {
    gcb_env_config cfg;
    EnvView v;
    ulonglong2 *t_bb01 = nullptr, *t_bb23 = nullptr;
    u64 *t_meta = nullptr, *t_zkey = nullptr, *t_tgt = nullptr, *zob = nullptr;
    ulonglong2* t_cnt = nullptr;
    u64 tick = 0;
    // staging for the host-buffer step calls
    int32_t *d_in = nullptr, *d_reward = nullptr;
    uint8_t *d_done = nullptr, *d_flags = nullptr;
    cudaStream_t streams[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t events[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    // every device array of the env: `user` is what the kernels see; with guard regions (GCB_GUARD_BYTES=<n> in the
    // environment at create time -- a test-only mode) it sits between two regions filled with 0xA5 that
    // gcb_env_check_guards() verifies
    struct Alloc {
        const char* name;
        char* base;
        char* user;
        size_t bytes;
    };
    std::vector<Alloc> allocs;
    size_t guard = 0;
    // optional learner-facing output of every step call (gcb_env_step_mask_output)
    u64* bits_out = nullptr;
    int bits_stride = 0;
};
#define GCB_GUARD_BYTE 0xA5

static cudaError_t env_alloc(gcb_env* env, const char* name, void** out, size_t bytes) {
    const size_t G = env->guard;  // a multiple of 256: `user` keeps cudaMalloc's alignment
    char* base = nullptr;
    cudaError_t e = cudaMalloc((void**)&base, bytes + 2 * G + (G ? 256 : 0));
    if (e != cudaSuccess) return e;
    if (G) {
        e = cudaMemset(base, GCB_GUARD_BYTE, G);
        if (e == cudaSuccess) e = cudaMemset(base + G + bytes, GCB_GUARD_BYTE, G + 256);  // starts at the first byte past the array
        if (e != cudaSuccess) {
            cudaFree(base);
            return e;
        }
    }
    env->allocs.push_back({name, base, base + G, bytes});
    *out = base + G;
    return cudaSuccess;
}

static const int8_t kDefaultBoard[64] = {-3, -5, -4, -2, -1, -4, -5, -3, -6, -6, -6, -6, -6, -6, -6, -6, 0, 0, 0, 0, 0, 0,
                                         0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0,  0, 0, 0, 0, 0, 0,
                                         0,  0,  0,  0,  6,  6,  6,  6,  6,  6,  6,  6,  3,  5,  4,  2,  1, 4, 5, 3};

// single-step launches: with the default 16 piece slots the generation runs on the shared-memory tile (TILE 2)
template <int MODE>
static int launch_io(gcb_env* env, StepIO& io, cudaStream_t s) {
    const int grid = grid_for(io.e_end - io.e_begin);
    // (measured: without the mask output the generic kernel -- with unchecked slot stores -- is faster at one step per launch:
    // 90 vs 105 us per step of 524,288 envs; with it the tile wins, 166 vs 191 us, because the mask is scattered from shared memory)
    const bool tile = GCB_SINGLE_TILE && env->bits_out != nullptr && env->v.slots == GCB_SLOTS && MODE != MODE_RESET && MODE != MODE_BOTPLY;
    const bool selfplay = MODE != MODE_RESET && MODE != MODE_BOTPLY && env->v.opponent == 0 && !env->v.agent_black;
    io.bits_out = (MODE != MODE_RESET) ? env->bits_out : nullptr, io.bits_stride = env->bits_stride;
    if constexpr (MODE == MODE_RESET || MODE == MODE_BOTPLY) {
        k_env_step<MODE, 0, false><<<grid, GCB_BLOCK, 0, s>>>(env->v, io);
    } else {
        if (tile && selfplay) k_env_step<MODE, 2, true><<<grid, GCB_BLOCK, 0, s>>>(env->v, io);
        else if (tile) k_env_step<MODE, 2, false><<<grid, GCB_BLOCK, 0, s>>>(env->v, io);
        else if (selfplay) k_env_step<MODE, 0, true><<<grid, GCB_BLOCK, 0, s>>>(env->v, io);
        else k_env_step<MODE, 0, false><<<grid, GCB_BLOCK, 0, s>>>(env->v, io);
    }
    LAUNCHED();
    return GCB_OK;
}

template <int MODE>
static int launch_range(gcb_env* env, const void* in, int32_t* reward, uint8_t* done, uint8_t* flags, int32_t* act_out,
                        int32_t* bot_out, int ep_inc, int e_begin, int e_end, cudaStream_t s) {
    StepIO io;
    io.in = in, io.reward = reward, io.done = done, io.flags = flags, io.act_out = act_out, io.bot_out = bot_out;
    io.tick = env->tick, io.ep_inc = ep_inc, io.e_begin = e_begin, io.e_end = e_end, io.nsteps = 1;
    return launch_io<MODE>(env, io, s);
}

template <int MODE>
static int launch_step(gcb_env* env, const void* in, int32_t* reward, uint8_t* done, uint8_t* flags, int32_t* act_out,
                       int32_t* bot_out, int ep_inc, cudaStream_t s) {
    int rc = launch_range<MODE>(env, in, reward, done, flags, act_out, bot_out, ep_inc, 0, env->v.N, s);
    env->tick++;
    return rc;
}

extern "C" int gcb_env_destroy(gcb_env* env) {
    if (!env) return GCB_OK;
    DeviceScope dev;
    dev.enter(env->cfg.device);
    for (const gcb_env::Alloc& a : env->allocs) cudaFree(a.base);
    for (int c = 0; c < 8; c++)
        if (env->streams[c]) cudaStreamDestroy(env->streams[c]);
    for (int c = 0; c < 9; c++)
        if (env->events[c]) cudaEventDestroy(env->events[c]);
    delete env;
    return GCB_OK;
}

extern "C" int gcb_env_create(const gcb_env_config* cfg_in, gcb_env** out) {
    if (!cfg_in || !out) return fail(GCB_E_ARG, "gcb_env_create", "null pointer");
    if (int rc = need_gpu()) return rc;
    gcb_env_config cfg = *cfg_in;
    if (cfg.num_envs <= 0) return fail(GCB_E_ARG, "gcb_env_create", "num_envs <= 0");
    // piece slots: one per own piece of the side to move; piece counts never grow (no promotion in play, Q1)
    {
        int need = 16;
        for (int t = 0; t < cfg.n_templates && cfg.template_boards; t++) {
            int w = 0, bl = 0;
            for (int sq = 0; sq < 64; sq++) {
                int8_t p = cfg.template_boards[(size_t)t * 64 + sq];
                w += p > 0, bl += p < 0;
            }
            need = need < w ? w : need;
            need = need < bl ? bl : need;
        }
        if (cfg.piece_slots == 0) cfg.piece_slots = need;
        if (cfg.piece_slots < need || cfg.piece_slots > 64)
            return fail(GCB_E_ARG, "gcb_env_create", "piece_slots must be 0 (auto) or in [max pieces per side, 64]");
        if ((long long)cfg.piece_slots * cfg.num_envs >= (1LL << 31))
            return fail(GCB_E_ARG, "gcb_env_create", "num_envs * piece_slots must stay below 2^31 (shard the envs)");
    }
    if (cfg.history_cap == 0) cfg.history_cap = 512;
    if (cfg.moves_max < 0) cfg.moves_max = 149;
    if (cfg.history_cap < 8 || cfg.history_cap > 1024 || (cfg.history_cap & (cfg.history_cap - 1)))
        return fail(GCB_E_ARG, "gcb_env_create", "history_cap must be a power of two in [8, 1024]");
    if (cfg.opponent < 0 || cfg.opponent > 2) return fail(GCB_E_ARG, "gcb_env_create", "opponent must be 0 (none), 1 (random) or 2 (external)");
    if (cfg.agent_black && cfg.opponent == 0)  // chess_v2.py:208-209 calls opponent_policy(None) -> TypeError (Q23)
        return fail(GCB_E_ARG, "gcb_env_create", "player_color BLACK needs an opponent (the reference raises TypeError)");
    if (cfg.n_templates < 0 || (cfg.n_templates > 0 && !cfg.template_boards))
        return fail(GCB_E_ARG, "gcb_env_create", "template_boards missing");
    DeviceScope dev;
    CU(dev.enter(cfg.device));
    gcb_env* env = new (std::nothrow) gcb_env();
    if (!env) return fail(GCB_E_NOMEM, "new", "gcb_env");
    if (const char* gv = getenv("GCB_GUARD_BYTES")) {  // test-only: guard regions around every env array
        const long g = atol(gv);
        env->guard = g > 0 ? (((size_t)g + 255) & ~(size_t)255) : 0;
    }
    const int N = cfg.num_envs, T = cfg.n_templates > 0 ? cfg.n_templates : 1, S = cfg.piece_slots, H = cfg.history_cap;
    env->cfg = cfg;
    env->cfg.template_boards = nullptr;
    EnvView& v = env->v;
    memset(&v, 0, sizeof(v));
    int8_t* d_tb = nullptr;
    cudaError_t e = cudaSuccess;
#define ALLOC(ptr, bytes) \
    if (e == cudaSuccess) e = env_alloc(env, #ptr, (void**)&(ptr), (bytes))
    ALLOC(v.bb01, (size_t)N * 16);
    ALLOC(v.bb23, (size_t)N * 16);
    ALLOC(v.meta, (size_t)N * 8);
    ALLOC(v.zkey, (size_t)N * 8);
    ALLOC(v.gen, (size_t)N * 4);
    ALLOC(v.cnt, (size_t)N * 16);
    ALLOC(env->t_cnt, (size_t)T * 16);
    ALLOC(v.episode, (size_t)N * 4);
    ALLOC(v.tgt, (size_t)N * S * 8);
    ALLOC(v.rep, (size_t)N * 2 * H * 16);  // twice history_cap slots: load factor <= 1/2 while the window fits
    ALLOC(v.stats, ST_COUNT * 8);
    ALLOC(v.stat_rows, (size_t)((N + 31) / 32) * ST_COUNT * 8);
    ALLOC(env->t_bb01, (size_t)T * 16);
    ALLOC(env->t_bb23, (size_t)T * 16);
    ALLOC(env->t_meta, (size_t)T * 8);
    ALLOC(env->t_zkey, (size_t)T * 8);
    ALLOC(env->t_tgt, (size_t)T * S * 8);
    ALLOC(env->zob, (size_t)GCB_ZOB_ENTRIES * 8);
    ALLOC(env->d_in, (size_t)N * 4);
    ALLOC(env->d_reward, (size_t)N * 4);
    ALLOC(env->d_done, (size_t)N);
    ALLOC(env->d_flags, (size_t)N);
#undef ALLOC
    if (e == cudaSuccess) e = cudaMalloc((void**)&d_tb, (size_t)T * 64);
    if (e != cudaSuccess) {
        cudaFree(d_tb);
        gcb_env_destroy(env);
        return fail(GCB_E_NOMEM, "cudaMalloc", cudaGetErrorString(e));
    }
    v.t_bb01 = env->t_bb01, v.t_bb23 = env->t_bb23, v.t_meta = env->t_meta, v.t_zkey = env->t_zkey, v.t_tgt = env->t_tgt;
    v.zob = env->zob, v.t_cnt = env->t_cnt;
    v.seed = cfg.seed, v.N = N, v.slots = S, v.hist_mask = 2 * H - 1, v.n_templates = T, v.env_offset = cfg.env_id_offset;
    v.stat_nrows = (N + 31) / 32;
    v.moves_max = cfg.moves_max, v.opponent = cfg.opponent, v.agent_black = cfg.agent_black, v.auto_reset = cfg.auto_reset;
    v.pps = 1 + (cfg.opponent == 1 ? 1 : 0);  // ring slots per step: agent ply, bot ply (a reset-bot ply reuses the bot slot)
    int rc = GCB_OK;
    do {
        if (cudaMemcpy(d_tb, cfg.n_templates > 0 ? cfg.template_boards : kDefaultBoard, (size_t)T * 64, cudaMemcpyHostToDevice) !=
                cudaSuccess ||
            cudaMemset(v.stats, 0, ST_COUNT * 8) != cudaSuccess ||
            cudaMemset(v.stat_rows, 0, (size_t)((N + 31) / 32) * ST_COUNT * 8) != cudaSuccess || cudaMemset(v.episode, 0, (size_t)N * 4) != cudaSuccess ||
            cudaMemset(v.meta, 0, (size_t)N * 8) != cudaSuccess || cudaMemset(v.bb01, 0, (size_t)N * 16) != cudaSuccess ||
            cudaMemset(v.bb23, 0, (size_t)N * 16) != cudaSuccess || cudaMemset(v.zkey, 0, (size_t)N * 8) != cudaSuccess ||
            cudaMemset(v.gen, 0, (size_t)N * 4) != cudaSuccess || cudaMemset(v.rep, 0, (size_t)N * 2 * H * 16) != cudaSuccess || cudaMemset(v.cnt, 0, (size_t)N * 16) != cudaSuccess || cudaMemset(v.tgt, 0, (size_t)N * S * 8) != cudaSuccess ||
            cudaMemset(env->t_tgt, 0, (size_t)T * S * 8) != cudaSuccess) {
            rc = fail(GCB_E_CUDA, "cudaMemcpy/cudaMemset", "env init");
            break;
        }
        k_init_zobrist<<<(GCB_ZOB_ENTRIES + 127) / 128, 128>>>(env->zob);
        k_make_templates<<<(T + 63) / 64, 64>>>(T, d_tb, env->t_bb01, env->t_bb23, env->t_meta, env->t_zkey, env->t_tgt, env->t_cnt, S);
        g_launches.fetch_add(2);
        // episode 0 starts with a reset that does not advance the episode counter
        StepIO io;
        memset(&io, 0, sizeof(io));
        io.tick = env->tick, io.e_begin = 0, io.e_end = N, io.nsteps = 1;
        k_env_step<MODE_RESET, 0, false><<<grid_for(N), GCB_BLOCK>>>(v, io);
        env->tick++;
        g_launches.fetch_add(1);
        cudaError_t e2 = cudaDeviceSynchronize();
        if (e2 != cudaSuccess) rc = fail(GCB_E_CUDA, "env init kernels", cudaGetErrorString(e2));
    } while (0);
    cudaFree(d_tb);
    if (rc) {
        gcb_env_destroy(env);
        return rc;
    }
    *out = env;
    return GCB_OK;
}

#define ENV_CHECK(env)                                               \
    if (!(env)) return fail(GCB_E_ARG, __func__, "null env");        \
    DeviceScope dev_scope_;                                          \
    CU(dev_scope_.enter((env)->cfg.device))

// a registered mask output (gcb_env_step_mask_output) is kept current by everything that changes the legal set: the step
// kernels write it themselves, reset and import run the mask kernel behind them
static int refresh_mask_output(gcb_env* env, cudaStream_t s);

extern "C" int gcb_env_reset(gcb_env* env, const uint8_t* d_mask, void* stream) {
    ENV_CHECK(env);
    if (int rc = launch_step<MODE_RESET>(env, d_mask, nullptr, nullptr, nullptr, nullptr, nullptr, 1, (cudaStream_t)stream)) return rc;
    return refresh_mask_output(env, (cudaStream_t)stream);
}

extern "C" int gcb_env_step(gcb_env* env, const int32_t* d_actions, int32_t* d_reward, uint8_t* d_done, uint8_t* d_flags,
                            void* stream) {
    ENV_CHECK(env);
    if (!d_actions) return fail(GCB_E_ARG, "gcb_env_step", "null actions");
    return launch_step<MODE_ACTION>(env, d_actions, d_reward, d_done, d_flags, nullptr, nullptr, 1, (cudaStream_t)stream);
}

extern "C" int gcb_env_bot_ply(gcb_env* env, const int32_t* d_bot_actions, int32_t* d_reward, uint8_t* d_done, uint8_t* d_flags,
                               void* stream) {
    ENV_CHECK(env);
    if (!d_bot_actions) return fail(GCB_E_ARG, "gcb_env_bot_ply", "null actions");
    if (env->v.opponent != 2) return fail(GCB_E_ARG, "gcb_env_bot_ply", "the env was not created with opponent 2 (external)");
    return launch_step<MODE_BOTPLY>(env, d_bot_actions, d_reward, d_done, d_flags, nullptr, nullptr, 1, (cudaStream_t)stream);
}

extern "C" int gcb_env_step_index(gcb_env* env, const uint32_t* d_u32, int32_t* d_reward, uint8_t* d_done, uint8_t* d_flags,
                                  void* stream) {
    ENV_CHECK(env);
    if (!d_u32) return fail(GCB_E_ARG, "gcb_env_step_index", "null random words");
    return launch_step<MODE_INDEX>(env, d_u32, d_reward, d_done, d_flags, nullptr, nullptr, 1, (cudaStream_t)stream);
}

#define GCB_MAX_STEPS_PER_LAUNCH 64
#define GCB_HOST_CHUNKS 8
static int ensure_streams(gcb_env* env) {
    if (!env->streams[0]) {
        for (int c = 0; c < GCB_HOST_CHUNKS; c++) CU(cudaStreamCreateWithFlags(&env->streams[c], cudaStreamNonBlocking));
        for (int c = 0; c <= GCB_HOST_CHUNKS; c++) CU(cudaEventCreateWithFlags(&env->events[c], cudaEventDisableTiming));
    }
    return GCB_OK;
}

extern "C" int gcb_env_step_sampled(gcb_env* env, int nsteps, int32_t* d_reward, uint8_t* d_done, uint8_t* d_flags,
                                    int32_t* d_actions_out, int32_t* d_bot_out, void* stream) {
    ENV_CHECK(env);
    if (nsteps < 0) return fail(GCB_E_ARG, "gcb_env_step_sampled", "nsteps < 0");
    if (env->v.opponent == 2) return fail(GCB_E_ARG, "gcb_env_step_sampled", "an env with an external opponent is stepped with gcb_env_step + gcb_env_bot_ply");
    const size_t N = (size_t)env->v.N;
    // A run of several launches is issued as a few env RANGES on their own streams (forked from / joined to the caller's
    // stream): every launch ends with a partly filled last wave of blocks (524,288 envs = 5.5 waves of 740 resident
    // blocks), and with independent ranges the next launch of one range fills the tail of the other.  Envs never read
    // each other, so ranges need no ordering among themselves.
    static const int want = [] {  // (function-local static: initialised once, thread-safe)
        const char* ev = getenv("GCB_SAMPLED_RANGES");
        const int w = ev ? atoi(ev) : 2;
        return (w < 1 || w > GCB_HOST_CHUNKS) ? 2 : w;
    }();
    // (Cutting a short run of 16..64 steps into two launches so that it, too, runs as two ranges was measured: 67.6 against
    // 66.3 us per step at 20 steps -- the extra trip of the state through memory costs more than half a last wave.)
    const int per_launch = GCB_MAX_STEPS_PER_LAUNCH;
    const int nlaunch = (nsteps + per_launch - 1) / per_launch;
    const int R = (nlaunch >= 2 && N >= (size_t)want * 65536) ? want : 1;
    const int per = (int)((((N + R - 1) / R) + GCB_BLOCK - 1) / GCB_BLOCK * GCB_BLOCK);  // whole blocks (and whole stat rows)
    cudaStream_t cs = (cudaStream_t)stream;
    if (R > 1) {
        if (int rc = ensure_streams(env)) return rc;
        CU(cudaEventRecord(env->events[GCB_HOST_CHUNKS], cs));
        for (int r = 0; r < R; r++) CU(cudaStreamWaitEvent(env->streams[r], env->events[GCB_HOST_CHUNKS], 0));
    }
    const bool selfplay = env->v.opponent == 0 && !env->v.agent_black, tiled = env->v.slots == GCB_SLOTS;
    int rc = GCB_OK;
    for (int t = 0; t < nsteps && rc == GCB_OK;) {
        const int k = nsteps - t < per_launch ? nsteps - t : per_launch;
        StepIO io;
        io.in = nullptr, io.reward = d_reward, io.done = d_done, io.flags = d_flags;
        io.act_out = d_actions_out ? d_actions_out + t * N : nullptr, io.bot_out = d_bot_out ? d_bot_out + t * N : nullptr;
        io.tick = env->tick, io.ep_inc = 1, io.nsteps = k;
        // the mask output belongs to the state the RUN leaves behind: only the last launch writes it
        io.bits_out = (t + k == nsteps) ? env->bits_out : nullptr, io.bits_stride = env->bits_stride;
        for (int r = 0; r < R; r++) {
            io.e_begin = r * per, io.e_end = (r + 1) * per < (int)N ? (r + 1) * per : (int)N;
            if (io.e_begin >= io.e_end) break;
            cudaStream_t ls = R > 1 ? env->streams[r] : cs;
            const int grid = grid_for(io.e_end - io.e_begin);
            // several steps: the slots are staged into the tile once (TILE 1); a few steps that also write the bit mask:
            // generation on the tile without stage-in (TILE 2); a few plain steps: the generic kernel (measured fastest)
            if (tiled && k >= 4 && selfplay) k_env_step<MODE_SAMPLED, 1, true><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            else if (tiled && k >= 4) k_env_step<MODE_SAMPLED, 1, false><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            else if (tiled && io.bits_out && selfplay) k_env_step<MODE_SAMPLED, 2, true><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            else if (tiled && io.bits_out) k_env_step<MODE_SAMPLED, 2, false><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            else if (selfplay) k_env_step<MODE_SAMPLED, 0, true><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            else k_env_step<MODE_SAMPLED, 0, false><<<grid, GCB_BLOCK, 0, ls>>>(env->v, io);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            const cudaError_t le = cudaGetLastError();
            if (le != cudaSuccess) {
                rc = fail(GCB_E_CUDA, "kernel launch", cudaGetErrorString(le));
                break;
            }
        }
        env->tick += (u64)k;
        t += k;
    }
    if (R > 1) {  // the forked streams are joined on EVERY path, also after a failed launch
        for (int r = 0; r < R; r++) {
            const cudaError_t e1 = cudaEventRecord(env->events[r], env->streams[r]);
            const cudaError_t e2 = e1 == cudaSuccess ? cudaStreamWaitEvent(cs, env->events[r], 0) : e1;
            if (e2 != cudaSuccess && rc == GCB_OK) rc = fail(GCB_E_CUDA, "join of the range streams", cudaGetErrorString(e2));
        }
    }
    return rc;
}

// Host-buffer step: the batch is cut into chunks that travel on their own streams, so the H2D copy of chunk k+1, the
// kernel of chunk k and the D2H copies of chunk k-1 overlap (PCIe is full duplex).  Envs are independent, so a step may
// be issued range by range; all chunks share the step's ring tick.  Pass page-locked host buffers to get the overlap
// (pageable memory still works, the copies then serialise).
// device-visible alias of a page-locked host buffer (NULL for pageable memory)
static void* mapped_ptr(const void* host) {
    if (!host) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, host) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}

static int step_host_common(gcb_env* env, int mode, const void* in, int32_t* reward, uint8_t* done, uint8_t* flags, cudaStream_t cs) {
    const int N = env->v.N;
    // Zero-copy path: when every buffer is page-locked, the step kernel reads the actions and writes reward / done /
    // flags straight through PCIe (coalesced 128-byte rows per warp) -- one launch, no staging copies, the transfers
    // overlap the move generation of the other warps.
    static const int zero_copy = [] {
        const char* ev = getenv("GCB_HOST_ZEROCOPY");
        return ev ? atoi(ev) : 1;
    }();
    if (zero_copy) {
        void* m_in = mapped_ptr(in);
        void* m_r = mapped_ptr(reward);
        void* m_d = mapped_ptr(done);
        void* m_f = mapped_ptr(flags);
        if (m_in && (m_r || !reward) && (m_d || !done) && (m_f || !flags)) {
            int rc = mode == MODE_ACTION
                         ? launch_step<MODE_ACTION>(env, m_in, (int32_t*)m_r, (uint8_t*)m_d, (uint8_t*)m_f, nullptr, nullptr, 1, cs)
                         : launch_step<MODE_INDEX>(env, m_in, (int32_t*)m_r, (uint8_t*)m_d, (uint8_t*)m_f, nullptr, nullptr, 1, cs);
            if (rc) return rc;
            CU(cudaStreamSynchronize(cs));
            return GCB_OK;
        }
    }
    static const int want = [] {  // GCB_HOST_CHUNKS=<1..8> overrides the default pipelining depth
        const char* ev = getenv("GCB_HOST_CHUNKS");
        const int w = ev ? atoi(ev) : 4;
        return (w < 1 || w > GCB_HOST_CHUNKS) ? 4 : w;
    }();
    int chunks = N >= want * 16384 ? want : (N >= 32768 ? 2 : 1);
    int per = (((N + chunks - 1) / chunks) + GCB_BLOCK - 1) / GCB_BLOCK * GCB_BLOCK;  // whole blocks (and whole stat rows)
    if (int rc = ensure_streams(env)) return rc;
    // the chunk streams start after everything enqueued on the caller's stream so far
    CU(cudaEventRecord(env->events[GCB_HOST_CHUNKS], cs));
    for (int c = 0; c < chunks; c++) CU(cudaStreamWaitEvent(env->streams[c], env->events[GCB_HOST_CHUNKS], 0));
    const char* src = reinterpret_cast<const char*>(in);
    for (int c = 0; c < chunks; c++) {
        const int b = c * per, e = (b + per < N) ? b + per : N;
        if (b >= e) break;
        cudaStream_t s = env->streams[c];
        CU(cudaMemcpyAsync(env->d_in + b, src + (size_t)b * 4, (size_t)(e - b) * 4, cudaMemcpyHostToDevice, s));
        int rc = mode == MODE_ACTION ? launch_range<MODE_ACTION>(env, env->d_in, env->d_reward, env->d_done, env->d_flags, nullptr,
                                                                  nullptr, 1, b, e, s)
                                     : launch_range<MODE_INDEX>(env, env->d_in, env->d_reward, env->d_done, env->d_flags, nullptr,
                                                                 nullptr, 1, b, e, s);
        if (rc) return rc;
        if (reward) CU(cudaMemcpyAsync(reward + b, env->d_reward + b, (size_t)(e - b) * 4, cudaMemcpyDeviceToHost, s));
        if (done) CU(cudaMemcpyAsync(done + b, env->d_done + b, (size_t)(e - b), cudaMemcpyDeviceToHost, s));
        if (flags) CU(cudaMemcpyAsync(flags + b, env->d_flags + b, (size_t)(e - b), cudaMemcpyDeviceToHost, s));
    }
    env->tick++;
    cudaError_t first = cudaSuccess;  // every chunk stream is drained, also after an error on one of them
    for (int c = 0; c < chunks; c++) {
        const cudaError_t ce = cudaStreamSynchronize(env->streams[c]);
        if (first == cudaSuccess) first = ce;
    }
    if (first != cudaSuccess) return fail(GCB_E_CUDA, "host-buffer step", cudaGetErrorString(first));
    return GCB_OK;
}

extern "C" int gcb_env_step_host(gcb_env* env, const int32_t* actions, int32_t* reward, uint8_t* done, uint8_t* flags, void* stream) {
    ENV_CHECK(env);
    if (!actions) return fail(GCB_E_ARG, "gcb_env_step_host", "null actions");
    return step_host_common(env, MODE_ACTION, actions, reward, done, flags, (cudaStream_t)stream);
}

extern "C" int gcb_env_step_index_host(gcb_env* env, const uint32_t* u32, int32_t* reward, uint8_t* done, uint8_t* flags, void* stream) {
    ENV_CHECK(env);
    if (!u32) return fail(GCB_E_ARG, "gcb_env_step_index_host", "null random words");
    return step_host_common(env, MODE_INDEX, u32, reward, done, flags, (cudaStream_t)stream);
}

// Asynchronous host-buffer steps: page-locked buffers only (their device aliases are read / written in place by the step
// kernel); the launch is enqueued on `stream` and the call returns.  Two or more env objects (shards of one device) can
// be kept in flight this way: the device steps one while the host consumes the other's results and writes its actions.
static int step_host_async(gcb_env* env, int mode, const void* in, int32_t* reward, uint8_t* done, uint8_t* flags, void* stream) {
    void* m_in = mapped_ptr(in);
    void* m_r = mapped_ptr(reward);
    void* m_d = mapped_ptr(done);
    void* m_f = mapped_ptr(flags);
    if (!m_in || (reward && !m_r) || (done && !m_d) || (flags && !m_f))
        return fail(GCB_E_ARG, "gcb_env_step_*_host_async", "buffers must be page-locked (cudaHostAlloc / cudaHostRegister / pin_memory)");
    return mode == MODE_ACTION
               ? launch_step<MODE_ACTION>(env, m_in, (int32_t*)m_r, (uint8_t*)m_d, (uint8_t*)m_f, nullptr, nullptr, 1, (cudaStream_t)stream)
               : launch_step<MODE_INDEX>(env, m_in, (int32_t*)m_r, (uint8_t*)m_d, (uint8_t*)m_f, nullptr, nullptr, 1, (cudaStream_t)stream);
}

extern "C" int gcb_env_step_host_async(gcb_env* env, const int32_t* actions, int32_t* reward, uint8_t* done, uint8_t* flags,
                                       void* stream) {
    ENV_CHECK(env);
    if (!actions) return fail(GCB_E_ARG, "gcb_env_step_host_async", "null actions");
    return step_host_async(env, MODE_ACTION, actions, reward, done, flags, stream);
}

extern "C" int gcb_env_step_index_host_async(gcb_env* env, const uint32_t* u32, int32_t* reward, uint8_t* done, uint8_t* flags,
                                             void* stream) {
    ENV_CHECK(env);
    if (!u32) return fail(GCB_E_ARG, "gcb_env_step_index_host_async", "null random words");
    return step_host_async(env, MODE_INDEX, u32, reward, done, flags, stream);
}

// Packed 16-bit records: the same step with 2 bytes in and 2 bytes out per env (10 with the int32 / uint8 arrays).  The
// pointers may be device memory or page-locked host memory (the device alias is used: read / written in place through PCIe).
static void* device_view(const void* p) {
    if (!p) return nullptr;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) return const_cast<void*>(p);
    return a.type == cudaMemoryTypeHost ? a.devicePointer : nullptr;
}
template <int MODE>
static int step_packed(gcb_env* env, const uint16_t* in16, uint16_t* result16, void* stream) {
    void* d_in = device_view(in16);
    void* d_out = device_view(result16);
    if (!d_in || (result16 && !d_out))
        return fail(GCB_E_ARG, "gcb_env_step_*_packed", "buffers must be device memory or page-locked host memory");
    StepIO io;
    io.in = d_in, io.in16 = 1, io.packed = (uint16_t*)d_out;
    io.reward = nullptr, io.done = nullptr, io.flags = nullptr, io.act_out = nullptr, io.bot_out = nullptr;
    io.tick = env->tick, io.ep_inc = 1, io.e_begin = 0, io.e_end = env->v.N, io.nsteps = 1;
    const int rc = launch_io<MODE>(env, io, (cudaStream_t)stream);
    env->tick++;
    return rc;
}
extern "C" int gcb_env_step_packed(gcb_env* env, const uint16_t* actions16, uint16_t* result16, void* stream) {
    ENV_CHECK(env);
    return step_packed<MODE_ACTION>(env, actions16, result16, stream);
}
extern "C" int gcb_env_step_index_packed(gcb_env* env, const uint16_t* u16, uint16_t* result16, void* stream) {
    ENV_CHECK(env);
    return step_packed<MODE_INDEX>(env, u16, result16, stream);
}

extern "C" int gcb_env_wait(gcb_env* env, void* stream) {
    ENV_CHECK(env);
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return GCB_OK;
}

extern "C" int gcb_env_import(gcb_env* env, const int8_t* d_boards, const int8_t* d_players, const uint8_t* d_rights4,
                              const int32_t* d_move_count, const uint8_t* d_mask, void* stream) {
    ENV_CHECK(env);
    if (!d_boards || !d_players || !d_rights4) return fail(GCB_E_ARG, "gcb_env_import", "null pointer");
    k_env_import<<<grid_for(env->v.N), GCB_BLOCK, 0, (cudaStream_t)stream>>>(env->v, d_boards, d_players, d_rights4, d_move_count,
                                                                               d_mask, env->tick);
    env->tick++;
    LAUNCHED();
    return refresh_mask_output(env, (cudaStream_t)stream);
}

extern "C" int gcb_env_clone(gcb_env* dst, const gcb_env* src, const int32_t* d_src_index, void* stream) {
    ENV_CHECK(dst);
    if (!src || !d_src_index) return fail(GCB_E_ARG, "gcb_env_clone", "null pointer");
    const gcb_env_config &a = dst->cfg, &b = src->cfg;
    if (a.device != b.device) return fail(GCB_E_ARG, "gcb_env_clone", "source and destination live on different devices");
    if (a.piece_slots != b.piece_slots || a.history_cap != b.history_cap || a.opponent != b.opponent ||
        a.agent_black != b.agent_black || a.moves_max != b.moves_max)
        return fail(GCB_E_ARG, "gcb_env_clone", "source and destination differ in piece_slots, history_cap, opponent, agent colour or moves_max");
    const cudaStream_t s = (cudaStream_t)stream;
    uint8_t* is_src = nullptr;
#if defined(GCB_CHECKED)
    if (src == dst) {  // the aliasing check: which rows are sources of this call
        CU(cudaMallocAsync((void**)&is_src, (size_t)dst->v.N, s));
        CU(cudaMemsetAsync(is_src, 0, (size_t)dst->v.N, s));
        k_env_clone_mark<<<grid_for(dst->v.N), GCB_BLOCK, 0, s>>>(dst->v.N, src->v.N, d_src_index, is_src);
        LAUNCHED();
    }
#endif
    const int warps_per_block = GCB_BLOCK / 32;
    k_env_clone<<<(dst->v.N + warps_per_block - 1) / warps_per_block, GCB_BLOCK, 0, s>>>(dst->v, src->v, d_src_index, is_src);
    LAUNCHED();
    if (is_src) CU(cudaFreeAsync(is_src, s));
    return refresh_mask_output(dst, s);
}

// ---- checkpoint / resume: the resident state is plain arrays; a snapshot is their concatenation in one device buffer
struct SnapPart {
    void* ptr;
    size_t bytes;
};
static int snap_parts(gcb_env* env, SnapPart* p) {
    const size_t N = (size_t)env->v.N, S = (size_t)env->v.slots, H = (size_t)env->v.hist_mask + 1;
    int k = 0;
    p[k++] = {env->v.bb01, N * 16}, p[k++] = {env->v.bb23, N * 16}, p[k++] = {env->v.meta, N * 8}, p[k++] = {env->v.zkey, N * 8};
    p[k++] = {env->v.gen, N * 4}, p[k++] = {env->v.cnt, N * 16}, p[k++] = {env->v.episode, N * 4};
    p[k++] = {env->v.tgt, N * S * 8}, p[k++] = {env->v.rep, N * H * 16};
    p[k++] = {env->v.stat_rows, ((N + 31) / 32) * ST_COUNT * 8};
    return k;
}

extern "C" int gcb_env_snapshot_bytes(gcb_env* env, uint64_t* bytes) {
    if (!env || !bytes) return fail(GCB_E_ARG, "gcb_env_snapshot_bytes", "null pointer");
    SnapPart p[16];
    const int k = snap_parts(env, p);
    size_t tot = 0;
    for (int i = 0; i < k; i++) tot += (p[i].bytes + 255) & ~(size_t)255;
    *bytes = tot;
    return GCB_OK;
}

extern "C" int gcb_env_snapshot(gcb_env* env, void* d_buf, uint64_t* tick, void* stream) {
    ENV_CHECK(env);
    if (!d_buf || !tick) return fail(GCB_E_ARG, "gcb_env_snapshot", "null pointer");
    SnapPart p[16];
    const int k = snap_parts(env, p);
    char* dst = reinterpret_cast<char*>(d_buf);
    for (int i = 0; i < k; i++) {
        CU(cudaMemcpyAsync(dst, p[i].ptr, p[i].bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        dst += (p[i].bytes + 255) & ~(size_t)255;
    }
    *tick = env->tick;
    return GCB_OK;
}

extern "C" int gcb_env_restore(gcb_env* env, const void* d_buf, uint64_t tick, void* stream) {
    ENV_CHECK(env);
    if (!d_buf) return fail(GCB_E_ARG, "gcb_env_restore", "null pointer");
    SnapPart p[16];
    const int k = snap_parts(env, p);
    const char* src = reinterpret_cast<const char*>(d_buf);
    for (int i = 0; i < k; i++) {
        CU(cudaMemcpyAsync(p[i].ptr, src, p[i].bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
        src += (p[i].bytes + 255) & ~(size_t)255;
    }
    env->tick = tick;
    return GCB_OK;
}

extern "C" int gcb_env_export(gcb_env* env, int8_t* d_boards, int32_t* d_info, void* stream) {
    ENV_CHECK(env);
    k_env_export<<<grid_for(env->v.N), GCB_BLOCK, 0, (cudaStream_t)stream>>>(env->v, d_boards, d_info);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_legal_mask(gcb_env* env, uint8_t* d_mask, void* stream) {
    ENV_CHECK(env);
    if (!d_mask) return fail(GCB_E_ARG, "gcb_env_legal_mask", "null mask");
    CU(cudaMemsetAsync(d_mask, 0, (size_t)env->v.N * 4101, (cudaStream_t)stream));
    k_env_legal_mask<<<grid_for(env->v.N), GCB_BLOCK, 0, (cudaStream_t)stream>>>(env->v, d_mask);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_legal_bitmask(gcb_env* env, uint64_t* d_bits, int stride_words, void* stream) {
    ENV_CHECK(env);
    if (!d_bits || stride_words < 65) return fail(GCB_E_ARG, "gcb_env_legal_bitmask", "null pointer or stride_words < 65");
    k_env_legal_bits<<<grid_for(env->v.N), GCB_BLOCK, 0, (cudaStream_t)stream>>>(env->v, reinterpret_cast<u64*>(d_bits), stride_words, 0, env->v.N);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_sample_policy(const gcb_env* env, const void* d_logits, int dtype, int64_t row_stride, float temperature,
                                     const uint32_t* d_u32, int32_t* d_actions, float* d_logp, void* stream) {
    ENV_CHECK(env);
    if (dtype != GCB_DT_F32 && dtype != GCB_DT_BF16) return fail(GCB_E_ARG, "gcb_env_sample_policy", "dtype must be GCB_DT_F32 or GCB_DT_BF16");
    if (row_stride < 4101) return fail(GCB_E_ARG, "gcb_env_sample_policy", "row_stride < 4101");
    if (!(temperature >= 0.f && temperature < INFINITY)) return fail(GCB_E_ARG, "gcb_env_sample_policy", "temperature must be finite and >= 0");
    if (!d_logits || !d_actions) return fail(GCB_E_ARG, "gcb_env_sample_policy", "null logits or actions");
    const cudaStream_t s = (cudaStream_t)stream;
    if (dtype == GCB_DT_F32)
        k_env_policy_sample<0><<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, d_logits, (long long)row_stride, temperature, d_u32, d_actions, d_logp);
    else
        k_env_policy_sample<1><<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, d_logits, (long long)row_stride, temperature, d_u32, d_actions, d_logp);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_encode(const gcb_env* env, void* d_planes, int dtype, uint8_t* d_rep, void* stream) {
    ENV_CHECK(env);
    if (dtype != GCB_DT_F32 && dtype != GCB_DT_BF16 && dtype != GCB_DT_U8)
        return fail(GCB_E_ARG, "gcb_env_encode", "dtype must be GCB_DT_F32, GCB_DT_BF16 or GCB_DT_U8");
    if (!d_planes && !d_rep) return fail(GCB_E_ARG, "gcb_env_encode", "d_planes and d_rep are both NULL");
    if (reinterpret_cast<uintptr_t>(d_planes) & 15u) return fail(GCB_E_ARG, "gcb_env_encode", "d_planes is not 16-byte aligned");
    const cudaStream_t s = (cudaStream_t)stream;
    if (dtype == GCB_DT_F32) k_env_encode<0><<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, d_planes, d_rep);
    else if (dtype == GCB_DT_BF16) k_env_encode<1><<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, d_planes, d_rep);
    else k_env_encode<2><<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, d_planes, d_rep);
    LAUNCHED();
    return GCB_OK;
}

static int refresh_mask_output(gcb_env* env, cudaStream_t s) {
    if (!env->bits_out) return GCB_OK;
    k_env_legal_bits<<<grid_for(env->v.N), GCB_BLOCK, 0, s>>>(env->v, env->bits_out, env->bits_stride, 0, env->v.N);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_step_mask_output(gcb_env* env, uint64_t* d_bits, int stride_words) {
    if (!env) return fail(GCB_E_ARG, "gcb_env_step_mask_output", "null env");
    if (d_bits && stride_words < 65) return fail(GCB_E_ARG, "gcb_env_step_mask_output", "stride_words < 65");
    env->bits_out = reinterpret_cast<u64*>(d_bits), env->bits_stride = d_bits ? stride_words : 0;
    return GCB_OK;
}

extern "C" int gcb_env_legal_actions(gcb_env* env, uint16_t* d_actions, int stride, int32_t* d_counts, void* stream) {
    ENV_CHECK(env);
    if (!d_actions || stride <= 0 || (stride & 1)) return fail(GCB_E_ARG, "gcb_env_legal_actions", "null pointer or odd stride");
    k_env_legal_list<<<grid_for(env->v.N), GCB_BLOCK, 0, (cudaStream_t)stream>>>(env->v, d_actions, stride, d_counts);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_piece_slots(gcb_env* env, uint64_t** d_slots, int32_t* n_slots) {
    if (!env) return fail(GCB_E_ARG, "gcb_env_piece_slots", "null env");
    if (d_slots) *d_slots = reinterpret_cast<uint64_t*>(env->v.tgt);
    if (n_slots) *n_slots = env->v.slots;
    return GCB_OK;
}

extern "C" int gcb_env_positions(gcb_env* env, gcb_positions* out) {
    if (!env || !out) return fail(GCB_E_ARG, "gcb_env_positions", "null pointer");
    out->bb01 = reinterpret_cast<uint64_t*>(env->v.bb01);
    out->bb23 = reinterpret_cast<uint64_t*>(env->v.bb23);
    out->player = nullptr, out->rights = nullptr;
    return GCB_OK;
}

// ---- memory-safety net (test support): guard regions around every env array, index checks of the CHECKED build
extern "C" int gcb_env_check_guards(gcb_env* env, uint64_t* n_bad_bytes) {
    ENV_CHECK(env);
    if (!n_bad_bytes) return fail(GCB_E_ARG, "gcb_env_check_guards", "null pointer");
    *n_bad_bytes = 0;
    if (!env->guard) return fail(GCB_E_ARG, "gcb_env_check_guards", "the env was created without GCB_GUARD_BYTES");
    CU(cudaDeviceSynchronize());
    const size_t G = env->guard;
    std::vector<unsigned char> h(G + 256);
    char first[160] = "";
    for (const gcb_env::Alloc& a : env->allocs) {
        for (int side = 0; side < 2; side++) {
            const size_t n = side ? G + 256 : G;
            CU(cudaMemcpy(h.data(), side ? a.user + a.bytes : a.base, n, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < n; i++)
                if (h[i] != GCB_GUARD_BYTE) {
                    if (!*n_bad_bytes) snprintf(first, sizeof(first), "%s: byte %zu %s the array", a.name, side ? i : G - i, side ? "past the end of" : "before");
                    ++*n_bad_bytes;
                }
        }
    }
    if (*n_bad_bytes) snprintf(g_err, sizeof(g_err), "guard regions overwritten, first: %s", first);
    return GCB_OK;
}

extern "C" int gcb_debug_violations(uint64_t* out, int reset) {
    if (!out) return fail(GCB_E_ARG, "gcb_debug_violations", "null pointer");
    if (int rc = need_gpu()) return rc;
    unsigned long long v = 0;
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpyFromSymbol(&v, g_violations, sizeof(v)));
    if (reset) {
        const unsigned long long z = 0;
        CU(cudaMemcpyToSymbol(g_violations, &z, sizeof(z)));
    }
    *out = v;
    return GCB_OK;
}
extern "C" int gcb_build_is_checked(void) {
#if defined(GCB_CHECKED)
    return 1;
#else
    return 0;
#endif
}

static int stats_reduce(gcb_env* env, cudaStream_t s) {
    k_stats_reduce<<<1, 512, 0, s>>>(env->v.stat_rows, (env->v.N + 31) / 32, env->v.stats);
    LAUNCHED();
    return GCB_OK;
}

extern "C" int gcb_env_stats(gcb_env* env, uint64_t* out16, void* stream) {
    ENV_CHECK(env);
    if (!out16) return fail(GCB_E_ARG, "gcb_env_stats", "null out");
    if (int rc = stats_reduce(env, (cudaStream_t)stream)) return rc;
    CU(cudaMemcpyAsync(out16, env->v.stats, ST_COUNT * 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CU(cudaStreamSynchronize((cudaStream_t)stream));
    return GCB_OK;
}

extern "C" int gcb_env_stats_reset(gcb_env* env, void* stream) {
    ENV_CHECK(env);
    CU(cudaMemsetAsync(env->v.stats, 0, ST_COUNT * 8, (cudaStream_t)stream));
    CU(cudaMemsetAsync(env->v.stat_rows, 0, (size_t)((env->v.N + 31) / 32) * ST_COUNT * 8, (cudaStream_t)stream));
    return GCB_OK;
}

extern "C" int gcb_env_stats_ptr(gcb_env* env, uint64_t** d_stats, void* stream) {
    if (!env || !d_stats) return fail(GCB_E_ARG, "gcb_env_stats_ptr", "null pointer");
    DeviceScope dev;
    CU(dev.enter(env->cfg.device));
    if (int rc = stats_reduce(env, (cudaStream_t)stream)) return rc;  // totals are current once `stream` reaches here
    *d_stats = reinterpret_cast<uint64_t*>(env->v.stats);
    return GCB_OK;
}
