// encode_emul.cpp -- TEST INFRASTRUCTURE.  The host emulation of host_emul.cpp plus the network-input encoder (gcb_env_encode):
// env_encode_one of env_core.cuh, the serial form of the rule that k_env_encode writes with one warp per 32 envs.
#include "host_emul.cpp"

extern "C" {

// planes [N][19][64] of dtype 0 (fp32) / 1 (bf16 as uint16) / 2 (uint8), or NULL; rep uint8[N] or NULL
void emul_env_encode(const EmulEnv* E, void* planes, int dtype, uint8_t* rep) {
    for (int e = 0; e < E->v.N; e++) {
        if (dtype == 1) env_encode_one<1>(E->v, e, static_cast<uint16_t*>(planes), rep);
        else if (dtype == 2) env_encode_one<2>(E->v, e, static_cast<uint8_t*>(planes), rep);
        else env_encode_one<0>(E->v, e, static_cast<float*>(planes), rep);
    }
}

}  // extern "C"
