// clone_emul.cpp -- TEST INFRASTRUCTURE.  The host emulation of host_emul.cpp plus the per-env clone (gcb_env_clone):
// the same GCB_HD code of env_core.cuh that k_env_clone splits among the lanes of a warp, run row by row on the CPU.
#include "host_emul.cpp"

extern "C" {

// index int32[dst N]: env d of dst becomes env index[d] of src for 0 <= index[d] < src N; other rows are left untouched
void emul_env_clone(EmulEnv* dst, const EmulEnv* src, const int32_t* index) {
    for (int d = 0; d < dst->v.N; d++) {
        const int i = index[d];
        if (i < 0 || i >= src->v.N) continue;
        env_clone_one(dst->v, d, src->v, i);
    }
}

}  // extern "C"
