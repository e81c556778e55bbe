/*
 * mlp_reference.c -- C restatement of the MLP policy's mean (dexsim_rollout_mlp, dexsim_mlp_policy_mean;
 * include/dexsim.h), the arithmetic reference of tests/test_rollout_mlp.py.  TEST INFRASTRUCTURE ONLY.
 *
 * Built by the test with the oracle's flags (gcc -O2 -ffp-contract=off -fno-fast-math, SSE2): every product and sum is
 * rounded as written; fmaf is glibc's correctly rounded fused multiply-add, tanhf glibc's.
 */
#include <math.h>
#include <stdint.h>

#if defined(__FLT_EVAL_METHOD__) && __FLT_EVAL_METHOD__ != 0
#error "the reference needs FLT_EVAL_METHOD == 0 (SSE2 arithmetic)"
#endif

#define OBS 45
#define NJ 15

/* acc = 0; acc = fmaf(W[j,i], x[i], acc) for ascending i; y = acc + b[j]; act 0 ReLU (NaN propagates), 1 tanhf,
 * -1 none (the output layer) */
static void layer(const float* W, const float* b, int32_t nin, int32_t nout, const float* x, float* y, int32_t act) {
    for (int32_t j = 0; j < nout; ++j) {
        float acc = 0.0f;
        for (int32_t i = 0; i < nin; ++i) acc = fmaf(W[(int64_t)j * nin + i], x[i], acc);
        float v = acc + b[j];
        if (act == 0) v = (v > 0.0f || v != v) ? v : 0.0f;
        else if (act == 1) v = tanhf(v);
        y[j] = v;
    }
}

/* params packed in torch's layout: W1 [h1,45], b1, (W2 [h2,h1], b2,) W3 [15,h_last], b3; obs [n,45], out [n,15] */
void mlp_reference_mean(const float* params, int32_t num_hidden, const int32_t* hidden, int32_t activation,
                        const float* obs, int64_t n, float* out) {
    const int32_t h1 = hidden[0], h2 = num_hidden == 2 ? hidden[1] : 0, hl = num_hidden == 2 ? h2 : h1;
    const float* W1 = params;
    const float* b1 = W1 + (int64_t)h1 * OBS;
    const float* W2 = b1 + h1;
    const float* b2 = W2 + (int64_t)h2 * h1;
    const float* W3 = num_hidden == 2 ? b2 + h2 : W2;
    const float* b3 = W3 + (int64_t)NJ * hl;
    for (int64_t r = 0; r < n; ++r) {
        float a1[64], a2[64];
        layer(W1, b1, OBS, h1, obs + r * OBS, a1, activation);
        if (num_hidden == 2) layer(W2, b2, h1, h2, a1, a2, activation);
        layer(W3, b3, hl, NJ, num_hidden == 2 ? a2 : a1, out + r * NJ, -1);
    }
}
