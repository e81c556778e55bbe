/*
 * log_prob_reference.c -- C restatement of the log-probability of the behaviour-policy record
 * (dexsim_rollout_mlp_record; include/dexsim.h), the arithmetic reference of tests/test_policy_record.py.
 * TEST INFRASTRUCTURE ONLY.
 *
 * Built by the test with the oracle's flags (gcc -O2 -ffp-contract=off -fno-fast-math, SSE2): every product and sum is
 * rounded as written; fmaf is glibc's correctly rounded fused multiply-add, log glibc's double log.
 */
#include <math.h>
#include <stdint.h>

#if defined(__FLT_EVAL_METHOD__) && __FLT_EVAL_METHOD__ != 0
#error "the reference needs FLT_EVAL_METHOD == 0 (SSE2 arithmetic)"
#endif

#define NJ 15

/* c = (float)(-S - 7.5 L), S the ascending double sum from 0 of log((double)std_j), L = double log(2 pi); per row
 * lp = fmaf(-0.5f, s, c), s the ascending fmaf chain from 0 of z_j * z_j.  std [15], z [n,15], out [n] */
void log_prob_reference(const float* std, const float* z, int64_t n, float* out) {
    double S = 0.0;
    for (int32_t j = 0; j < NJ; ++j) S = S + log((double)std[j]);
    const float c = (float)(-S - 7.5 * 1.8378770664093453);
    for (int64_t r = 0; r < n; ++r) {
        float s = 0.0f;
        for (int32_t j = 0; j < NJ; ++j) s = fmaf(z[r * NJ + j], z[r * NJ + j], s);
        out[r] = fmaf(-0.5f, s, c);
    }
}
