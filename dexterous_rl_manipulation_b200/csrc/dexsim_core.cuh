// dexsim_core.cuh -- per-env arithmetic of the batched manipulation simulator (sm_100a).
//
// One env's state lives in registers (EnvRegs); the kernels in dexsim_kernels.cu move it
// between HBM and registers.  Everything here mirrors, operation for operation and rounding
// for rounding, what the reference computes under numpy 2.3.5 (NEP 50):
//   envs/manipulation_env.py:124-182 (reset), :184-252 (step), :285-310 (contacts),
//   rewards/reward_shaping.py:50-187 (dense), :205-242 (sparse),
//   evaluation/metrics.py:39-96 and evaluation/failure_taxonomy.py:156-239 (failure labels).
// Joints and velocities are float32; the object position, the fingertip distances and the
// contact test are float64 because the reference's are (SURVEY.md 8a-3, 8a-4).  Every product
// and sum the reference rounds separately is written with __f*_rn / __d*_rn intrinsics, which
// nvcc never contracts into FMA (the file is also compiled with -fmad=false).
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/dexsim.h"

namespace dexsim {

constexpr int NJ = DEXSIM_NJ;
constexpr int NF = DEXSIM_NF;
constexpr int NOBS = DEXSIM_OBS;

#if defined(__CUDACC__)
#define DEXSIM_HD __host__ __device__ __forceinline__
#define DEXSIM_D __device__ __forceinline__
#else
#define DEXSIM_HD inline
#define DEXSIM_D inline
#endif

#if defined(__CUDACC__)
// n_c / num_fingers for n_c = 0..5, rounded once like the reference's int / int true division
__constant__ double kContactReward[6] = {0.0 / 5.0, 1.0 / 5.0, 2.0 / 5.0, 3.0 / 5.0, 4.0 / 5.0, 5.0 / 5.0};
// clip(float32(1 - float32(k / 5)), 0, 1) for k = 0..5 flipped contact bits, the float32 arithmetic of
// rewards/reward_shaping.py:178-183 folded at compile time (IEEE single-precision division and subtraction)
__constant__ float kStabilityReward[6] = {1.0f - 0.0f / 5.0f, 1.0f - 1.0f / 5.0f, 1.0f - 2.0f / 5.0f,
                                          1.0f - 3.0f / 5.0f, 1.0f - 4.0f / 5.0f, 1.0f - 5.0f / 5.0f};
#endif

struct EnvRegs {
    float    jp[NJ];
    float    jv[NJ];
    double   op[3];
    float    ov[3];
    double   thr;     // object_size * 1.5
    float    damp;    // float32(1.0 - friction * 0.1 * 0.01)
    int      sc;      // step_count; sc == 0 <=> object_position is still the float32 array of reset()
    unsigned cmask;   // bit f: finger f in contact after the last contact update
};

struct StepResult {
    double total, distance, contact, closure, stability;
    int    n_c;
    bool   terminated, truncated;
};

// np.clip == minimum(maximum(x, lo), hi): NaN propagates (fminf/fmaxf would swallow it)
DEXSIM_D float clip_f32(float x, float lo, float hi) {
    const float y = (x < lo) ? lo : x;
    return (y > hi) ? hi : y;
}
DEXSIM_D double clip_f64(double x, double lo, double hi) {
    const double y = (x < lo) ? lo : x;
    return (y > hi) ? hi : y;
}

// envs/manipulation_env.py:285-310.  Returns the contact mask and count; with NEED_DMIN also the
// minimum fingertip distance (rewards/reward_shaping.py:111-113).
//
// The reference tests RN(sqrt(sq)) < thr in float64.  sqrt is monotone and correctly rounded, so
//   sq < thr^2 (1 - 2^-50)  =>  sqrt(sq) < thr (1 - 2^-52) <= pred(thr)  =>  contact
//   sq > thr^2 (1 + 2^-50)  =>  sqrt(sq) > thr                           =>  no contact
// (thr^2 itself carries one rounding, 2^-53, absorbed by the 2^-50 margins).  Only inside that band --
// relative width 2^-49, the "contact branch" -- is the square root evaluated; the decision is
// bit-identical to the reference's for every threshold (0, negative, thr^2 underflowing or overflowing, inf, NaN) on the
// domain stepping produces: fingertips and object positions lie on the float32 grid (multiples of 2^-149), so sq is 0
// or >= 2^-298 (or inf / NaN from such inputs).  tests/test_contact_boundary.py puts fingers in the band and on
// d == thr exactly, through this function and split_contact (dexsim_rollout_split.cuh).  Likewise min_i RN(sqrt(sq_i)) == RN(sqrt(min_i sq_i)),
// so the dense reward needs one square root, not five.
// One finger of the test below (shared by update_contacts and the warp-cooperative reset): returns the contact bit,
// sq = squared fingertip-object distance.
DEXSIM_D bool finger_contact(const float j0, const float j1, const float j2, const double op0, const double op1, const double op2,
                             const double thr, const double lo2, const double hi2, const bool thr_pos, double& sq) {
    // :301-302 float32 sequential sum of 3 joints, "* 0.1" stays float32, then widened (:300)
    const float s = __fadd_rn(__fadd_rn(j0, j1), j2);
    const double tip = (double)__fmul_rn(s, 0.1f);
    // :309 np.linalg.norm(axis=1) in float64, left to right
    const double dx = __dsub_rn(tip, op0);
    const double dy = __dsub_rn(tip, op1);
    const double dz = __dsub_rn(tip, op2);
    sq = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    // two compares and a select for all but the tie band: lanes of a warp differ in their contact state all the
    // time, so an if / else-if chain here diverges (ncu: 26 of 32 lanes active on these lines); the band does not
    const bool below = sq < lo2, above = sq > hi2;
    bool c = below;
    if (!(below || above)) c = __dsqrt_rn(sq) < thr;           // tie band (and NaN): exact test, :310
    return c && thr_pos;
}

template <bool NEED_DMIN>
DEXSIM_D unsigned update_contacts(const EnvRegs& e, int& n_c, double& dmin) {
    unsigned mask = 0u;
    n_c = 0;
    const double thr2 = __dmul_rn(e.thr, e.thr);
    const double lo2 = __dmul_rn(thr2, 1.0 - 0x1p-50), hi2 = __dmul_rn(thr2, 1.0 + 0x1p-50);
    const bool thr_pos = e.thr > 0.0;                              // d >= 0 can never be below thr <= 0
    double sqmin = 0.0;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        double sq;
        const bool c = finger_contact(e.jp[3 * f], e.jp[3 * f + 1], e.jp[3 * f + 2], e.op[0], e.op[1], e.op[2], e.thr, lo2, hi2,
                                      thr_pos, sq);
        mask |= (c ? 1u : 0u) << f;
        n_c += c ? 1 : 0;
        if (NEED_DMIN) sqmin = (f == 0) ? sq : ((sq < sqmin || sq != sq) ? sq : sqmin);   // np.min propagates NaN
    }
    dmin = NEED_DMIN ? __dsqrt_rn(sqmin) : 0.0;
    return mask;
}

// envs/manipulation_env.py:124-182 with the draws supplied (reference order: joints, size,
// mass, friction, x, y, z).  keep_pos: reused env object, position re-cast to float32 (:160-161).
DEXSIM_D void env_reset(EnvRegs& e, const float* jp0, double size, double friction,
                        const float* pos, bool keep_pos) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) { e.jp[j] = jp0[j]; e.jv[j] = 0.0f; }
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        e.op[i] = keep_pos ? (double)(float)e.op[i] : (double)pos[i];
        e.ov[i] = 0.0f;
    }
    e.thr = __dmul_rn(size, 1.5);                                            // :293
    e.damp = (float)__dsub_rn(1.0, __dmul_rn(__dmul_rn(friction, 0.1), 0.01)); // :215
    e.sc = 0;
    int n_c; double dmin;
    e.cmask = update_contacts<false>(e, n_c, dmin);                          // :176
}

// envs/manipulation_env.py:184-252 + rewards/reward_shaping.py (compute)
// CLIP_ACTION = false only when the caller has already produced actions inside [-1, 1] (in-kernel random /
// heuristic policy, or an action it clipped itself): np.clip is then the identity and is skipped.
template <bool DENSE, bool CLIP_ACTION = true>
DEXSIM_D void env_step(EnvRegs& e, const float* a, const DexsimParams& p, StepResult& r) {
    // :199-207
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const float aj = CLIP_ACTION ? clip_f32(a[j], -1.0f, 1.0f) : a[j];
        e.jv[j] = __fadd_rn(__fmul_rn(0.9f, e.jv[j]), __fmul_rn(0.1f, aj));
        e.jp[j] = clip_f32(__fadd_rn(e.jp[j], __fmul_rn(e.jv[j], 0.01f)), -1.0f, 1.0f);
    }
    // :211-219  (gravity is a float64 array: the += happens in float64, rounded back to float32)
    constexpr double kGravZ = -9.81 * 0.01;
    e.ov[0] = (float)__dadd_rn((double)__fmul_rn(e.ov[0], e.damp), 0.0);
    e.ov[1] = (float)__dadd_rn((double)__fmul_rn(e.ov[1], e.damp), 0.0);
    e.ov[2] = (float)__dadd_rn((double)__fmul_rn(e.ov[2], e.damp), kGravZ);
    // :222  float32 in-place add on the first step after reset, float64 afterwards
    const bool first = (e.sc == 0);
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const float dq = __fmul_rn(e.ov[i], 0.01f);
        const double p32 = (double)__fadd_rn((float)e.op[i], dq);
        const double p64 = __dadd_rn(e.op[i], (double)dq);
        e.op[i] = first ? p32 : p64;
    }
    // :225-235
    const double lo[3] = {-0.2, -0.2, 0.0};
    const double hi[3] = {0.2, 0.2, 0.3};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        e.op[i] = clip_f64(e.op[i], lo[i], hi[i]);
        if ((e.op[i] <= lo[i] && e.ov[i] < 0.0f) || (e.op[i] >= hi[i] && e.ov[i] > 0.0f)) e.ov[i] = 0.0f;
    }
    // :238
    double dmin;
    const unsigned prev = e.cmask;
    e.cmask = update_contacts<DENSE>(e, r.n_c, dmin);
    // :241
    if (DENSE) {
        r.distance = exp(__dmul_rn(-5.0, dmin));                              // reward_shaping.py:116
        r.contact = kContactReward[r.n_c];                                    // :134 n_c / 5 (correctly rounded constants)
        float msum = -0.0f;                                                   // :149-162
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            float s = -0.0f;
#pragma unroll
            for (int j = 0; j < 3; ++j) {
                // adding fminf(v, 0) == adding v only when v < 0 (NaN joints add 0, like the reference's mask);
                // the result can differ only in the sign of an all-zero sum, which nothing downstream sees
                s = __fadd_rn(s, fminf(e.jp[3 * f + j], 0.0f));
            }
            msum = __fadd_rn(msum, -s);
        }
        const float avg = __fdiv_rn(msum, 5.0f);
        r.closure = (double)clip_f32(__fdiv_rn(avg, 5.0f), 0.0f, 1.0f);
        if (first) {                                                          // :172-175
            r.stability = 0.0;
        } else {                                                              // :178-183
            r.stability = (double)kStabilityReward[__popc((prev ^ e.cmask) & 31u)];
        }
        r.total = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(p.w_distance, r.distance),
                                                __dmul_rn(p.w_contact, r.contact)),
                                      __dmul_rn(p.w_closure, r.closure)),
                            __dmul_rn(p.w_stability, r.stability));           // :86-91
    } else {
        r.total = (r.n_c >= 3) ? 1.0 : -0.01;                                 // :231-234
        r.distance = r.contact = r.closure = r.stability = 0.0;
    }
    r.terminated = r.n_c >= p.success_threshold;                              // :244
    r.truncated = e.sc >= p.max_episode_steps;                                // :245
    e.sc += 1;                                                                // :247
}

// ---- counter-based RNG: Philox4x32-10 (Salmon et al. SC'11), DESIGN.md "RNG" -----------------
struct U4 { uint32_t x, y, z, w; };

DEXSIM_D U4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return U4{c0, c1, c2, c3};
}

enum : uint32_t { STREAM_RESET = 0, STREAM_POLICY = 1, STREAM_DYN = 2, STREAM_OBS = 3, STREAM_LEARNER_ACT = 4,
                  STREAM_LEARNER_UPD = 5 };

DEXSIM_D U4 rng_block(uint64_t seed, uint32_t gid, uint32_t episode, uint32_t step, uint32_t stream,
                      uint32_t block) {
    return philox4x32_10(gid, episode, step, stream | (block << 8), (uint32_t)seed, (uint32_t)(seed >> 32));
}

DEXSIM_D float u24(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }
DEXSIM_D double u53(uint32_t a, uint32_t b) {
    // division by 2^53 == multiplication by 2^-53 (exact power-of-two scaling)
    return __dmul_rn(__dadd_rn(__dmul_rn((double)(a >> 5), 67108864.0), (double)(b >> 6)), 0x1p-53);
}
DEXSIM_D double lerp_rn(double lo, double hi, double u) {   // low + (high - low) * u, as Generator.uniform
    return __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u));
}

// Philox stand-in for the PCG64 draws of envs/manipulation_env.py:143-161 + experiments/config.py:44-113
// (DESIGN.md "RNG"): blocks 0-3 -> 15 joints (24-bit uniforms); block 4 -> spawn x, y, z (32-bit uniforms: the
// position is cast to float32 anyway); blocks 5-6 -> size, mass, friction (53-bit uniforms), generated only
// when the group actually randomises one of them -- fixed curricula (easy / medium / hard, held-out
// objects) reset with five Philox blocks instead of seven.
DEXSIM_D void reset_draws(uint64_t seed, uint32_t gid, uint32_t episode, const DexsimGroup& g, float* jp0,
                          double& size, double& mass, double& friction, float* pos) {
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b) {
        const U4 o = rng_block(seed, gid, episode, 0u, STREAM_RESET, b);
        const uint32_t w[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (4 * (int)b + k < NJ) jp0[4 * b + k] = (float)__dadd_rn(-0.1, __dmul_rn(0.2, (double)u24(w[k])));
    }
    {
        const U4 o = rng_block(seed, gid, episode, 0u, STREAM_RESET, 4u);
        const uint32_t w[3] = {o.x, o.y, o.z};
#pragma unroll
        for (int i = 0; i < 3; ++i)
            pos[i] = (float)lerp_rn(g.spawn_lo[i], g.spawn_hi[i], __dmul_rn((double)w[i], 0x1p-32));
    }
    size = g.size; mass = g.mass; friction = g.friction;
    if (g.size_ranged | g.mass_ranged | g.fric_ranged) {
        const U4 a = rng_block(seed, gid, episode, 0u, STREAM_RESET, 5u);
        const U4 b = rng_block(seed, gid, episode, 0u, STREAM_RESET, 6u);
        if (g.size_ranged) size = lerp_rn(g.size_lo, g.size_hi, u53(a.x, a.y));
        if (g.mass_ranged) mass = lerp_rn(g.mass_lo, g.mass_hi, u53(a.z, a.w));
        if (g.fric_ranged) friction = lerp_rn(g.fric_lo, g.fric_hi, u53(b.x, b.y));
    }
}

// policies/random_policy.py:40 and policies/heuristic_policy.py:55-62 on Philox bits
DEXSIM_D void policy_action(uint64_t seed, uint32_t gid, uint32_t episode, uint32_t step, int kind, float* a) {
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b) {
        const U4 o = rng_block(seed, gid, episode, step, STREAM_POLICY, b);
        const uint32_t w[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            // 2 * u24 - 1 == (x >> 8) * 2^-23 - 1: every intermediate is exact in float32, so the fused form
            // returns the same bits as the separately rounded one
            if (4 * (int)b + k < NJ) a[4 * b + k] = __fmaf_rn((float)(w[k] >> 8), 0x1p-23f, -1.0f);
        }
    }
    if (kind == DEXSIM_POLICY_HEURISTIC) {              // warp-uniform: only the selected policy's arithmetic runs
#pragma unroll
        for (int j = 0; j < NJ; ++j) a[j] = clip_f32(__fadd_rn(-0.5f, __fmul_rn(a[j], 0.1f)), -1.0f, 1.0f);
    }
}

// float32 N(0,1) pairs by Box-Muller on Philox words (device-only; parity runs pre-draw noise
// with dexsim_fill_normal and hand the same tensors to the oracle).
DEXSIM_D void normal_pair(uint32_t wa, uint32_t wb, float& z0, float& z1) {
    const float u1 = (float)((wa >> 8) + 1u) * 5.9604644775390625e-08f;   // (0, 1]
    const float u2 = u24(wb);
    const float rad = sqrtf(-2.0f * __logf(u1));
    // uniform angle in [-pi, pi): the range in which the hardware sine / cosine keep ~2^-21 absolute error
    const float theta = 6.2831855f * (u2 - 0.5f);
    const float s = __sinf(theta), c = __cosf(theta);
    z0 = rad * c; z1 = rad * s;
}
template <int ROWS>
DEXSIM_D void normal_rows(uint64_t seed, uint32_t gid, uint32_t episode, uint32_t step, uint32_t stream,
                          float sigma, float* out) {
    constexpr int NBLK = (ROWS + 3) / 4;
#pragma unroll
    for (int b = 0; b < NBLK; ++b) {
        const U4 o = rng_block(seed, gid, episode, step, stream, (uint32_t)b);
        float z[4];
        normal_pair(o.x, o.y, z[0], z[1]);
        normal_pair(o.z, o.w, z[2], z[3]);
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (4 * b + k < ROWS) out[4 * b + k] = sigma * z[k];
    }
}

// ---- episode history summary + failure labels --------------------------------------------------
// Packed per-env summary of the per-step contact COUNTS an Evaluator would have collected
// (evaluation/evaluator.py:148-150): enough to run both classifiers without the history.
//   w0: [15:0] sum of counts   [20:16] sum of the first five   [23:21] max count
//   w1: [16:0] sum of squares  [31:17] last five counts, 3 bits each (newest in the low bits)
struct EpStats { uint32_t w0, w1; };

// The packed sums hold episodes of up to EPSTATS_MAX_STEPS steps (5,242 steps of 5 contacts reach 2^17 - 1 in the sum of
// squares); the entry points reject longer tracked episodes (DEXSIM_E_PARAM) and the fields saturate instead of wrapping
// if a caller steps a tracked env past that without resetting it.
constexpr int EPSTATS_MAX_STEPS = 5242;

DEXSIM_HD void epstats_push(EpStats& s, int hist_len_before, int n_c) {
    uint32_t sum = s.w0 & 0xFFFFu, first5 = (s.w0 >> 16) & 0x1Fu, mx = (s.w0 >> 21) & 0x7u;
    uint32_t sq = s.w1 & 0x1FFFFu, ring = s.w1 >> 17;
    sum += (uint32_t)n_c; sq += (uint32_t)(n_c * n_c);
    sum = sum > 0xFFFFu ? 0xFFFFu : sum; sq = sq > 0x1FFFFu ? 0x1FFFFu : sq;
    if (hist_len_before < 5) first5 += (uint32_t)n_c;
    mx = ((uint32_t)n_c > mx) ? (uint32_t)n_c : mx;
    ring = ((ring << 3) | (uint32_t)n_c) & 0x7FFFu;
    s.w0 = (sum & 0xFFFFu) | (first5 << 16) | (mx << 21);
    s.w1 = (sq & 0x1FFFFu) | (ring << 17);
}

DEXSIM_HD void epstats_unpack(const EpStats& s, int& sum, int& sq, int& first5, int& last5, int& mx) {
    sum = (int)(s.w0 & 0xFFFFu); first5 = (int)((s.w0 >> 16) & 0x1Fu); mx = (int)((s.w0 >> 21) & 0x7u);
    sq = (int)(s.w1 & 0x1FFFFu);
    const uint32_t ring = s.w1 >> 17;
    last5 = (int)((ring & 7u) + ((ring >> 3) & 7u) + ((ring >> 6) & 7u) + ((ring >> 9) & 7u) + ((ring >> 12) & 7u));
}

// ---- np.var of the per-step contact counts, bit for bit -----------------------------------------------------
// Both classifiers threshold np.var(contact_counts) (evaluation/metrics.py:77-78, evaluation/failure_taxonomy.py:189,
// :219-230).  For a list of ints NumPy computes (numpy/_core/_methods.py::_var, numpy 2.3.5): float64 mean = sum / n
// (the integer sum is exact), x = (count - mean)^2 element-wise, then the float64 PAIRWISE sum of x
// (numpy/_core/src/umath/loops_utils.h.src: plain loop below 8 elements, 8 interleaved accumulators up to 128,
// recursive halving rounded down to a multiple of 8 above), divided by n.  The order of the counts matters for the
// last bits, so this needs the history itself; the packed summary cannot reproduce it.
struct CountsView {               // per-step contact counts of ONE episode: count(k) = base[k * stride]
    const uint8_t* base;
    int64_t stride;
    DEXSIM_HD double sq_dev(int64_t k, double mean) const {
#if defined(__CUDA_ARCH__)
        const double d = __dsub_rn((double)base[k * stride], mean);
        return __dmul_rn(d, d);
#else
        const double d = (double)base[k * stride] - mean;
        return d * d;
#endif
    }
};

DEXSIM_HD double np_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// pairwise sum of the squared deviations of counts [lo, lo + n).  Recursive like NumPy's (depth log2(n / 128): 1 for the
// 200-step episodes of every shipped config); only ever reached on an exact variance tie, so it is kept out of line.
#if defined(__CUDACC__)
__host__ __device__ __noinline__
#endif
static double np_pairwise_sq_sum(const CountsView& c, int64_t lo, int64_t n, double mean) {
    if (n < 8) {
        double res = -0.0;
        for (int64_t i = 0; i < n; ++i) res = np_add(res, c.sq_dev(lo + i, mean));
        return res;
    }
    if (n <= 128) {
        double r[8];
        for (int k = 0; k < 8; ++k) r[k] = c.sq_dev(lo + k, mean);
        int64_t i;
        for (i = 8; i < n - (n % 8); i += 8)
            for (int k = 0; k < 8; ++k) r[k] = np_add(r[k], c.sq_dev(lo + i + k, mean));
        double res = np_add(np_add(np_add(r[0], r[1]), np_add(r[2], r[3])), np_add(np_add(r[4], r[5]), np_add(r[6], r[7])));
        for (; i < n; ++i) res = np_add(res, c.sq_dev(lo + i, mean));
        return res;
    }
    int64_t n2 = n / 2;
    n2 -= n2 % 8;
    const double left = np_pairwise_sq_sum(c, lo, n2, mean);
    return np_add(left, np_pairwise_sq_sum(c, lo + n2, n - n2, mean));
}

#if defined(__CUDACC__)
__host__ __device__ __noinline__
#endif
static double np_var_counts(const CountsView& c, int64_t n) {
    long long isum = 0;
    for (int64_t i = 0; i < n; ++i) isum += c.base[i * c.stride];
#if defined(__CUDA_ARCH__)
    const double mean = __ddiv_rn((double)isum, (double)n);
    return __ddiv_rn(np_pairwise_sq_sum(c, 0, n, mean), (double)n);
#else
    const double mean = (double)isum / (double)n;
    return np_pairwise_sq_sum(c, 0, n, mean) / (double)n;
#endif
}

// Both classifiers from the summary.  var = (n*Q - S^2)/n^2 is compared as integers, which decides every case
// except an EXACT tie with a threshold: there NumPy's float64 pairwise sum may land on either side
// (SURVEY.md 8a-12).  With the history at hand (`counts`, hist_len entries) a tie is decided by np.var itself
// (np_var_counts) and var_tie = 2; without it the tie is resolved as in exact arithmetic and var_tie = 1 flags the
// label as unconfirmed (DEXSIM_CNT_VAR_TIES counts those).  The slippage trend reproduces
// np.mean(last5) - np.mean(first5) with two IEEE divisions and one subtraction.
DEXSIM_HD void classify_summary(const DexsimEpisodeSummary& e, int max_steps, int thr,
                                int& label_a, int& label_b, int& var_tie, const CountsView* counts = nullptr) {
    var_tie = 0;
    label_a = label_b = DEXSIM_LABEL_NONE;
    if (e.success) return;                                        // metrics.py:53-55, failure_taxonomy.py:171-173
    const long long n = e.hist_len;
    const long long vnum = n * (long long)e.sum_sq_counts - (long long)e.sum_counts * e.sum_counts;  // var * n^2
    bool var_gt2 = vnum > 2 * n * n, var_lt1 = vnum < n * n;
    const bool tie2 = (n > 5) && (vnum == 2 * n * n), tie1 = (n > 1) && (vnum == n * n);
    const int tie_flag = (counts && counts->base) ? 2 : 1;
    if ((tie2 || tie1) && tie_flag == 2) {
        const double v = np_var_counts(*counts, n);
        var_gt2 = v > 2.0;                                        // metrics.py:78, failure_taxonomy.py:219
        var_lt1 = v < 1.0;                                        // failure_taxonomy.py:228
    }
#if defined(__CUDA_ARCH__)
    const double trend = __dsub_rn(__ddiv_rn((double)e.last5_sum, 5.0), __ddiv_rn((double)e.first5_sum, 5.0));
#else
    const double trend = (double)e.last5_sum / 5.0 - (double)e.first5_sum / 5.0;
#endif
    // EvaluationMetrics.classify_failure, evaluation/metrics.py:63-96
    {
        int lab;
        if (e.episode_steps >= max_steps) lab = DEXSIM_LABEL_TIMEOUT;
        else if (e.final_contacts == 0) lab = DEXSIM_LABEL_DROPPED;
        else {
            lab = -1;
            if (n > 5) {
                if (tie2) var_tie = tie_flag;
                if (var_gt2) lab = DEXSIM_LABEL_UNSTABLE;
                else if (n > 10 && trend < -1.0) lab = DEXSIM_LABEL_SLIPPAGE;
            }
            if (lab < 0) lab = (e.num_contacts > 0 && e.num_contacts < thr) ? DEXSIM_LABEL_MISALIGNED
                                                                            : DEXSIM_LABEL_INSUFFICIENT;
        }
        label_a = lab;
    }
    // FailureClassifier.classify, evaluation/failure_taxonomy.py:183-239
    {
        const int max_c = (n > 0) ? e.max_count : e.num_contacts;
        const bool has_var = n > 1;                                // :187 (variance is 0.0 otherwise)
        int lab;
        if (e.episode_steps >= max_steps) lab = DEXSIM_LABEL_TIMEOUT;
        else if (e.final_contacts == 0 && max_c > 0) lab = DEXSIM_LABEL_DROPPED;
        else {
            lab = -1;
            if (n > 5) {
                if (n > 10 && trend < -1.0 && max_c >= 1) lab = DEXSIM_LABEL_SLIPPAGE;
                else {
                    if (tie2) var_tie = tie_flag;
                    if (var_gt2) lab = DEXSIM_LABEL_UNSTABLE;
                }
            }
            if (lab < 0 && e.num_contacts >= 1 && e.num_contacts <= 2) {
                const bool lt1 = has_var ? var_lt1 : true;
                if (has_var && tie1) var_tie = tie_flag;
                if (lt1) lab = DEXSIM_LABEL_MISALIGNED;
            }
            if (lab < 0) lab = DEXSIM_LABEL_INSUFFICIENT;
        }
        label_b = lab;
    }
}

}  // namespace dexsim
