// policy_emul.cpp -- TEST INFRASTRUCTURE.  The host emulation of host_emul.cpp plus policy sampling (gcb_env_sample_policy):
// env_policy_sample_one of env_core.cuh, the serial form of the rule that k_env_policy_sample runs with one warp per env.
#include "host_emul.cpp"

extern "C" {

// logits [N][row_stride] of dtype 0 (fp32) / 1 (bf16 as uint16); words uint32[N] or NULL (Philox); logp may be NULL
void emul_env_sample_policy(const EmulEnv* E, const void* logits, int dtype, long long row_stride, float temperature,
                            const uint32_t* words, int32_t* actions, float* logp) {
    for (int e = 0; e < E->v.N; e++) {
        if (dtype == 1) env_policy_sample_one<1>(E->v, e, logits, row_stride, temperature, words, actions, logp);
        else env_policy_sample_one<0>(E->v, e, logits, row_stride, temperature, words, actions, logp);
    }
}

}  // extern "C"
