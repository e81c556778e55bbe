/*
 * dexsim_oracle.c -- CPU restatement of the reference's hot path.  TEST INFRASTRUCTURE ONLY.
 * See dexsim_oracle.h for the rules on who may load this and how parity is pinned.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -fno-fast-math; x86-64 SSE2 evaluates
 * float expressions in float and double expressions in double, FLT_EVAL_METHOD == 0, which is
 * what NumPy's loops do).  No FMA contraction anywhere: the reference rounds every product.
 *
 * Dtype notes are for the reference under numpy 2.3.5 (NEP 50: Python scalars are "weak").
 */
#include "dexsim_oracle.h"

#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#if defined(__FLT_EVAL_METHOD__) && __FLT_EVAL_METHOD__ != 0
#error "oracle needs FLT_EVAL_METHOD == 0 (SSE2 arithmetic)"
#endif

/* np.clip(x, lo, hi) == minimum(maximum(x, lo), hi); NaN propagates. */
static inline float clip_f32(float x, float lo, float hi) {
    float y = (x < lo) ? lo : x;
    return (y > hi) ? hi : y;
}
static inline double clip_f64(double x, double lo, double hi) {
    double y = (x < lo) ? lo : x;
    return (y > hi) ? hi : y;
}

/* envs/manipulation_env.py:119 */
static const double WS_LO[3] = {-0.2, -0.2, 0.0};
static const double WS_HI[3] = {0.2, 0.2, 0.3};

void dexo_default_params(dexo_params* p, int dense) {
    /* rewards/reward_shaping.py:20-25 defaults; envs/manipulation_env.py:29,53,336 */
    p->w_distance = 1.0; p->w_contact = 0.5; p->w_closure = 0.3; p->w_stability = 0.2;
    p->reward_type = dense ? 1 : 0;
    p->max_episode_steps = 200;
    p->success_threshold = 3;
    p->pad_ = 0;
}

/* envs/manipulation_env.py:285-310 (_update_contacts).  Returns distances for the reward. */
static void update_contacts(dexo_env* e, double dist[DEXO_NF]) {
    const double thr = e->size * 1.5;                         /* :293, float64 */
    int n = 0;
    for (int f = 0; f < DEXO_NF; ++f) {
        /* :301-302  np.sum of a 3-element float32 slice is sequential; "* 0.1" stays float32 */
        float s = e->jp[3 * f] + e->jp[3 * f + 1];
        s = s + e->jp[3 * f + 2];
        const float tip32 = s * 0.1f;
        const double tip = (double)tip32;                     /* finger_base is float64 zeros, :300 */
        /* :309  np.linalg.norm(axis=1): sqrt(add.reduce(x*x)) in float64, left to right */
        const double dx = tip - e->op[0], dy = tip - e->op[1], dz = tip - e->op[2];
        const double sq = (dx * dx + dy * dy) + dz * dz;
        dist[f] = sqrt(sq);
        e->c[f] = (dist[f] < thr) ? 1.0f : 0.0f;              /* :310 */
        n += (e->c[f] > 0.5f);
    }
    e->num_contacts = n;                                      /* :272 */
}

/* envs/manipulation_env.py:124-182 with the RNG draws supplied by the caller in the
 * reference's draw order (joints, size, mass, friction, x, y, z; SURVEY.md 8a-10). */
void dexo_reset_predrawn(dexo_env* e, const float* jp0, double size, double mass,
                         double friction, const float* pos) {
    for (int j = 0; j < DEXO_NJ; ++j) { e->jp[j] = jp0[j]; e->jv[j] = 0.0f; }   /* :143-148 */
    e->size = size; e->mass = mass; e->friction = friction;                     /* :151-153 */
    if (pos) { for (int i = 0; i < 3; ++i) e->op[i] = (double)pos[i]; }         /* :156-159 */
    else     { for (int i = 0; i < 3; ++i) e->op[i] = (double)(float)e->op[i]; }/* :160-161 */
    e->op_is_f32 = 1;
    for (int i = 0; i < 3; ++i) e->ov[i] = 0.0f;                                /* :167 */
    for (int f = 0; f < DEXO_NF; ++f) e->c[f] = 0.0f;                           /* :170 */
    e->step_count = 0;                                                          /* :173 */
    double dist[DEXO_NF];
    update_contacts(e, dist);                                                   /* :176 */
    e->has_prev = 0;                                                            /* :177 -> reward_shaping.py:45-48 */
    for (int f = 0; f < DEXO_NF; ++f) e->prev_c[f] = 0.0f;
    e->ep_return = 0.0; e->ep_steps = 0;
}

/* envs/manipulation_env.py:254-264 */
void dexo_observation(const dexo_env* e, float* obs) {
    for (int j = 0; j < DEXO_NJ; ++j) { obs[j] = e->jp[j]; obs[DEXO_NJ + j] = e->jv[j]; }
    for (int i = 0; i < 3; ++i) obs[30 + i] = (float)e->op[i];
    obs[33] = 1.0f; obs[34] = 0.0f; obs[35] = 0.0f; obs[36] = 0.0f;             /* :164 */
    for (int i = 0; i < 3; ++i) obs[37 + i] = e->ov[i];
    for (int f = 0; f < DEXO_NF; ++f) obs[40 + f] = e->c[f];
}

/* rewards/reward_shaping.py:50-99 (dense) and :205-242 (sparse) */
static void compute_reward(dexo_env* e, const dexo_params* p, const double dist[DEXO_NF],
                           dexo_reward* r) {
    const int n_c = e->num_contacts;
    if (p->reward_type == 0) {                                /* SparseReward.compute :228-242 */
        r->total = (n_c >= 3) ? 1.0 : -0.01;
        r->distance = r->contact = r->closure = r->stability = 0.0;
        return;
    }
    /* _compute_distance_reward :101-118 (same float64 distances as _update_contacts) */
    double dmin = dist[0];
    for (int f = 1; f < DEXO_NF; ++f) dmin = (dist[f] < dmin || isnan(dist[f])) ? dist[f] : dmin;   /* np.min propagates NaN */
    r->distance = exp(-5.0 * dmin);
    /* _compute_contact_reward :120-136 */
    r->contact = (double)n_c / (double)DEXO_NF;
    /* _compute_closure_reward :138-164: float32 per-finger sums of the negative joints,
     * float32 mean over 5 fingers (:159), then "/ num_fingers" AGAIN (:162), clip to [0,1] */
    float msum = -0.0f;
    for (int f = 0; f < DEXO_NF; ++f) {
        float s = -0.0f;
        for (int j = 0; j < DEXO_JPF; ++j) {
            const float v = e->jp[3 * f + j];
            if (v < 0.0f) s = s + v;
        }
        msum = msum + (-s);
    }
    const float avg = msum / 5.0f;
    r->closure = (double)clip_f32(avg / 5.0f, 0.0f, 1.0f);
    /* _compute_stability_reward :166-187 */
    if (!e->has_prev) {
        r->stability = 0.0;
        e->has_prev = 1;
    } else {
        float changes = -0.0f;
        for (int f = 0; f < DEXO_NF; ++f) changes = changes + fabsf(e->c[f] - e->prev_c[f]);
        const float st = 1.0f - (changes / 5.0f);
        r->stability = (double)clip_f32(st, 0.0f, 1.0f);
    }
    for (int f = 0; f < DEXO_NF; ++f) e->prev_c[f] = e->c[f];
    /* :86-91, Python floats, left to right */
    r->total = ((p->w_distance * r->distance + p->w_contact * r->contact)
                + p->w_closure * r->closure) + p->w_stability * r->stability;
}

/* envs/manipulation_env.py:184-252 */
void dexo_step(dexo_env* e, const dexo_params* p, const float* action,
               float* obs, dexo_reward* rew, int32_t* terminated, int32_t* truncated) {
    /* :199-207 all float32; two rounded products and a rounded sum, no FMA */
    for (int j = 0; j < DEXO_NJ; ++j) {
        const float a = clip_f32(action[j], -1.0f, 1.0f);
        const float t1 = 0.9f * e->jv[j];
        const float t2 = 0.1f * a;
        e->jv[j] = t1 + t2;
        const float dq = e->jv[j] * 0.01f;
        e->jp[j] = clip_f32(e->jp[j] + dq, -1.0f, 1.0f);
    }
    /* :211-219  damping factor is a Python float rounded once to float32 by "*=";
     * gravity is a float64 array, so "+=" adds in float64 and rounds back to float32 */
    const double damp64 = 1.0 - (e->friction * 0.1 * 0.01);
    const float damp = (float)damp64;
    const double grav[3] = {0.0, 0.0, -9.81 * 0.01};
    for (int i = 0; i < 3; ++i) {
        e->ov[i] = e->ov[i] * damp;
        e->ov[i] = (float)((double)e->ov[i] + grav[i]);
    }
    /* :222  first step after reset: object_position is float32 (in-place float32 add);
     * afterwards it is the float64 array np.clip returned */
    if (e->op_is_f32) {
        for (int i = 0; i < 3; ++i) {
            const float t = e->ov[i] * 0.01f;
            const float pnew = (float)e->op[i] + t;
            e->op[i] = (double)pnew;
        }
        e->op_is_f32 = 0;
    } else {
        for (int i = 0; i < 3; ++i) e->op[i] = e->op[i] + (double)(e->ov[i] * 0.01f);
    }
    /* :225-235 */
    for (int i = 0; i < 3; ++i) {
        e->op[i] = clip_f64(e->op[i], WS_LO[i], WS_HI[i]);
        if ((e->op[i] <= WS_LO[i] && e->ov[i] < 0.0f) || (e->op[i] >= WS_HI[i] && e->ov[i] > 0.0f))
            e->ov[i] = 0.0f;
    }
    double dist[DEXO_NF];
    update_contacts(e, dist);                                  /* :238 */
    compute_reward(e, p, dist, rew);                           /* :241 */
    *terminated = (e->num_contacts >= p->success_threshold);   /* :244, :332-336 */
    *truncated = (e->step_count >= p->max_episode_steps);      /* :245 (before the increment) */
    e->step_count += 1;                                        /* :247 */
    if (obs) dexo_observation(e, obs);                         /* :249 */
}

/* evaluation/robustness_tests.py:177-207 (CombinedNoiseWrapper.step) with the wrapper's
 * normal draws supplied by the caller already scaled by sigma and cast to float32. */
void dexo_step_noisy(dexo_env* e, const dexo_params* p, const float* action,
                     const float* dyn_noise, const float* obs_noise,
                     float* obs, dexo_reward* rew, int32_t* terminated, int32_t* truncated) {
    float a[DEXO_NJ];
    for (int j = 0; j < DEXO_NJ; ++j)
        a[j] = dyn_noise ? clip_f32(action[j] + dyn_noise[j], -1.0f, 1.0f) : action[j];  /* :180-189 */
    dexo_step(e, p, a, obs, rew, terminated, truncated);                                  /* :192 */
    if (obs && obs_noise)
        for (int k = 0; k < DEXO_OBS; ++k) obs[k] = obs[k] + obs_noise[k];                /* :204-205 */
}

/* ---- batch wrappers ------------------------------------------------------------------- */
void dexo_reset_predrawn_batch(dexo_env* e, int64_t n, const float* jp0, const double* size,
                               const double* mass, const double* friction, const float* pos) {
    for (int64_t i = 0; i < n; ++i)
        dexo_reset_predrawn(&e[i], jp0 + i * DEXO_NJ, size[i], mass[i], friction[i],
                            pos ? pos + i * 3 : NULL);
}

typedef struct {
    dexo_env* e; int64_t lo, hi; const dexo_params* p; const float* action;
    const float* dyn_noise; const float* obs_noise; float* obs; double* reward; double* comps;
    uint8_t* terminated; uint8_t* truncated; uint8_t* num_contacts;
} step_job;

static void* step_worker(void* arg) {
    step_job* j = (step_job*)arg;
    for (int64_t i = j->lo; i < j->hi; ++i) {
        dexo_reward r; int32_t te, tr;
        dexo_step_noisy(&j->e[i], j->p, j->action + i * DEXO_NJ,
                        j->dyn_noise ? j->dyn_noise + i * DEXO_NJ : NULL,
                        j->obs_noise ? j->obs_noise + i * DEXO_OBS : NULL,
                        j->obs ? j->obs + i * DEXO_OBS : NULL, &r, &te, &tr);
        if (j->reward) j->reward[i] = r.total;
        if (j->comps) {
            j->comps[4 * i + 0] = r.distance; j->comps[4 * i + 1] = r.contact;
            j->comps[4 * i + 2] = r.closure;  j->comps[4 * i + 3] = r.stability;
        }
        if (j->terminated) j->terminated[i] = (uint8_t)te;
        if (j->truncated) j->truncated[i] = (uint8_t)tr;
        if (j->num_contacts) j->num_contacts[i] = (uint8_t)j->e[i].num_contacts;
    }
    return NULL;
}

void dexo_step_batch(dexo_env* e, int64_t n, const dexo_params* p, const float* action,
                     const float* dyn_noise, const float* obs_noise, float* obs, double* reward,
                     double* comps, uint8_t* terminated, uint8_t* truncated,
                     uint8_t* num_contacts, int32_t threads) {
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    if ((int64_t)threads > n) threads = (int32_t)(n > 0 ? n : 1);
    step_job jobs[256]; pthread_t tid[256];
    for (int t = 0; t < threads; ++t) {
        step_job j = {e, n * t / threads, n * (t + 1) / threads, p, action, dyn_noise, obs_noise,
                      obs, reward, comps, terminated, truncated, num_contacts};
        jobs[t] = j;
    }
    if (threads == 1) { step_worker(&jobs[0]); return; }
    for (int t = 0; t < threads; ++t) pthread_create(&tid[t], NULL, step_worker, &jobs[t]);
    for (int t = 0; t < threads; ++t) pthread_join(tid[t], NULL);
}

/* ---- failure labels --------------------------------------------------------------------- */

/* NumPy's float64 pairwise summation (numpy/_core/src/umath/loops_utils.h.src,
 * DOUBLE_pairwise_sum; third-party, numpy 2.3.5, not vendored by the reference): plain loop
 * below 8 elements, 8 interleaved accumulators up to 128, recursive halving above. */
static double np_pairwise_sum(const double* a, int64_t n) {
    if (n < 8) {
        double res = -0.0;
        for (int64_t i = 0; i < n; ++i) res += a[i];
        return res;
    } else if (n <= 128) {
        double r[8];
        for (int k = 0; k < 8; ++k) r[k] = a[k];
        int64_t i;
        for (i = 8; i < n - (n % 8); i += 8)
            for (int k = 0; k < 8; ++k) r[k] += a[i + k];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res += a[i];
        return res;
    } else {
        int64_t n2 = n / 2;
        n2 -= n2 % 8;
        return np_pairwise_sum(a, n2) + np_pairwise_sum(a + n2, n - n2);
    }
}

/* np.var of a list of ints (numpy/_core/_methods.py:_var): float64 mean = sum/n, deviations,
 * squares, pairwise float64 sum, divided by n.  Used by evaluation/metrics.py:77 and
 * evaluation/failure_taxonomy.py:187. */
double dexo_np_var_counts(const uint8_t* counts, int64_t n) {
    if (n <= 0) return NAN;
    double* x = (double*)malloc(sizeof(double) * (size_t)n);
    int64_t isum = 0;
    for (int64_t i = 0; i < n; ++i) isum += counts[i];
    const double mean = (double)isum / (double)n;            /* integer sum is exact in float64 */
    for (int64_t i = 0; i < n; ++i) { const double d = (double)counts[i] - mean; x[i] = d * d; }
    const double v = np_pairwise_sum(x, n) / (double)n;
    free(x);
    return v;
}

static double mean5(const uint8_t* c) {                      /* np.mean of 5 ints: exact sum / 5 */
    int s = 0;
    for (int i = 0; i < 5; ++i) s += c[i];
    return (double)s / 5.0;
}

/* evaluation/metrics.py:39-96 (EvaluationMetrics.classify_failure) */
int32_t dexo_classify_metrics(int32_t success, int32_t episode_steps, int32_t num_contacts,
                              int32_t final_contacts, const uint8_t* counts, int64_t len,
                              int32_t max_steps, int32_t success_threshold) {
    if (success) return -1;                                           /* :53-55 */
    if (episode_steps >= max_steps) return DEXO_TIMEOUT;              /* :63-64 */
    if (final_contacts == 0) return DEXO_DROPPED;                     /* :67-68 */
    if (len > 0) {                                                    /* :71 */
        if (len > 5) {                                                /* :74 */
            if (dexo_np_var_counts(counts, len) > 2.0) return DEXO_UNSTABLE;     /* :76-78 */
            if (len > 10) {                                           /* :81 */
                const double trend = mean5(counts + len - 5) - mean5(counts);    /* :82 */
                if (trend < -1.0) return DEXO_SLIPPAGE;               /* :83-84 */
            }
        }
    }
    if (num_contacts > 0 && num_contacts < success_threshold) return DEXO_MISALIGNED;  /* :87-88 */
    return DEXO_INSUFFICIENT;                                         /* :91-96 */
}

/* evaluation/failure_taxonomy.py:156-239 (FailureClassifier.classify); thresholds from the
 * definitions table :53-57 (trend -1.0, min contacts 1), :70-74 (variance 2.0), :87-91 (1..2) */
int32_t dexo_classify_taxonomy(int32_t success, int32_t episode_steps, int32_t num_contacts,
                               int32_t final_contacts, const uint8_t* counts, int64_t len,
                               int32_t max_steps, int32_t success_threshold, double* confidence) {
    double conf_dummy;
    if (!confidence) confidence = &conf_dummy;
    *confidence = 0.0;
    if (success) return -1;                                           /* :171-173 */
    int max_c; double var;
    if (len > 0) {                                                    /* :183-189 */
        max_c = 0;
        for (int64_t i = 0; i < len; ++i) if (counts[i] > max_c) max_c = counts[i];
        var = (len > 1) ? dexo_np_var_counts(counts, len) : 0.0;
    } else {                                                          /* :190-193 */
        max_c = num_contacts; var = 0.0;
    }
    if (episode_steps >= max_steps) { *confidence = 1.0; return DEXO_TIMEOUT; }          /* :196-198 */
    if (final_contacts == 0 && max_c > 0) { *confidence = 1.0; return DEXO_DROPPED; }    /* :201-203 */
    if (len > 5) {                                                    /* :206 */
        if (len > 10) {                                               /* :208 */
            const double trend = mean5(counts + len - 5) - mean5(counts);                /* :209-211 */
            if (trend < -1.0 && max_c >= 1) {                         /* :214 */
                const double a = fabs(trend) / 2.0;
                *confidence = a < 1.0 ? a : 1.0;
                return DEXO_SLIPPAGE;
            }
        }
        if (var > 2.0) {                                              /* :219-222 */
            const double a = var / 5.0;
            *confidence = a < 1.0 ? a : 1.0;
            return DEXO_UNSTABLE;
        }
    }
    if (1 <= num_contacts && num_contacts <= 2) {                     /* :225-226 */
        if (var < 1.0) { *confidence = 0.8; return DEXO_MISALIGNED; } /* :228-230 */
    }
    if (max_c < success_threshold) { *confidence = 1.0; return DEXO_INSUFFICIENT; }      /* :233-235 */
    *confidence = 0.5;                                                /* :238-239 */
    return DEXO_INSUFFICIENT;
}

/* ---- counter-based RNG specification ---------------------------------------------------- *
 * Philox4x32-10 (Salmon et al., SC'11; same constants as Random123 / cuRAND).  The device
 * implements this specification independently; DESIGN.md "RNG" is the shared definition.
 *   key = (seed lo, seed hi);  counter = (env global id, episode, step, stream | block << 8)
 *   streams: 0 reset, 1 policy, 2 dynamics noise, 3 observation noise, 4 learner exploration,
 *   5 learner update                                                                        */
void dexo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3];
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

static void philox_block(uint64_t seed, uint32_t env_gid, uint32_t episode, uint32_t step,
                         uint32_t stream, uint32_t block, uint32_t out[4]) {
    const uint32_t ctr[4] = {env_gid, episode, step, stream | (block << 8)};
    const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    dexo_philox4x32_10(ctr, key, out);
}

static inline float u24(uint32_t x) { return (float)(x >> 8) * 5.9604644775390625e-08f; }  /* 2^-24 */
static inline double u53(uint32_t a, uint32_t b) {
    return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) / 9007199254740992.0;
}

/* Device-side replacement for the PCG64 draws of envs/manipulation_env.py:143-161 and
 * experiments/config.py:44-113: same draw ORDER and distributions, Philox bits. */
void dexo_reset_draws(uint64_t seed, uint32_t env_gid, uint32_t episode, const dexo_group* g,
                      float* jp0, double* size, double* mass, double* friction, float* pos) {
    /* blocks 0-3: joints; block 4: spawn x, y, z from 32-bit uniforms; blocks 5-6: size / mass / friction
     * from 53-bit uniforms, only for groups that randomise them (DESIGN.md "RNG") */
    uint32_t w[28];
    for (uint32_t b = 0; b < 7; ++b) philox_block(seed, env_gid, episode, 0u, 0u, b, w + 4 * b);
    for (int j = 0; j < DEXO_NJ; ++j)
        jp0[j] = (float)(-0.1 + 0.2 * (double)u24(w[j]));     /* U(-0.1, 0.1) -> float32, :143-145 */
    for (int i = 0; i < 3; ++i) {
        const double d = (double)w[16 + i] * 0x1p-32;
        pos[i] = (float)(g->spawn_lo[i] + (g->spawn_hi[i] - g->spawn_lo[i]) * d);
    }
    *size     = g->size_ranged ? g->size_lo + (g->size_hi - g->size_lo) * u53(w[20], w[21]) : g->size;
    *mass     = g->mass_ranged ? g->mass_lo + (g->mass_hi - g->mass_lo) * u53(w[22], w[23]) : g->mass;
    *friction = g->fric_ranged ? g->fric_lo + (g->fric_hi - g->fric_lo) * u53(w[24], w[25]) : g->friction;
}

/* policies/random_policy.py:40 (U(-1,1) float32) and policies/heuristic_policy.py:55-62
 * (clip(-0.5 + float32 U(-0.1,0.1))) with Philox bits. */
void dexo_policy_action(uint64_t seed, uint32_t env_gid, uint32_t episode, uint32_t step,
                        int32_t policy_kind, float* action) {
    uint32_t w[16];
    for (uint32_t b = 0; b < 4; ++b) philox_block(seed, env_gid, episode, step, 1u, b, w + 4 * b);
    for (int j = 0; j < DEXO_NJ; ++j) {
        const float u = 2.0f * u24(w[j]) - 1.0f;              /* exact in float32 */
        if (policy_kind == 2) {
            const float noise = u * 0.1f;
            action[j] = clip_f32(-0.5f + noise, -1.0f, 1.0f);
        } else {
            action[j] = u;
        }
    }
}

/* Box-Muller normals (streams 2-5), in double precision on the spec's exact inputs (DESIGN.md "RNG"):
 *   u1 = ((wa >> 8) + 1)·2^-24 in (0, 1],  u2 = (wb >> 8)·2^-24,  theta = 2·pi·(u2 - 1/2)
 *   z0 = sqrt(-2 ln u1)·cos(theta),  z1 = sqrt(-2 ln u1)·sin(theta)
 * The device evaluates the same formula in float32 with the hardware log / sin / cos; tests bound the difference. */
void dexo_normal_pair_ref(const uint32_t* wa, const uint32_t* wb, int64_t n, double* z0, double* z1) {
    const double two_pi = 6.283185307179586476925286766559;
    for (int64_t i = 0; i < n; ++i) {
        const double u1 = ((double)(wa[i] >> 8) + 1.0) * 0x1p-24;
        const double u2 = (double)(wb[i] >> 8) * 0x1p-24;
        const double r = sqrt(-2.0 * log(u1)), theta = two_pi * (u2 - 0.5);
        z0[i] = r * cos(theta);
        z1[i] = r * sin(theta);
    }
}

/* sigma·N(0,1) rows of one env: Philox block b of counter (gid, episode, step, stream | b << 8) gives rows
 * 4b .. 4b+3 from the word pairs (x, y) and (z, w). */
void dexo_normal_rows_ref(uint64_t seed, const uint32_t* env_gid, const uint32_t* episode, const uint32_t* step,
                          int64_t n, uint32_t stream, int32_t rows, double sigma, double* out) {
    for (int64_t i = 0; i < n; ++i) {
        for (int32_t b = 0; 4 * b < rows; ++b) {
            uint32_t w[4];
            double z[4];
            philox_block(seed, env_gid[i], episode[i], step[i], stream, (uint32_t)b, w);
            dexo_normal_pair_ref(&w[0], &w[1], 1, &z[0], &z[1]);
            dexo_normal_pair_ref(&w[2], &w[3], 1, &z[2], &z[3]);
            for (int k = 0; k < 4 && 4 * b + k < rows; ++k) out[i * rows + 4 * b + k] = sigma * z[k];
        }
    }
}

/* ---- fused rollout restatement --------------------------------------------------------- *
 * Loop shape of evaluation/evaluator.py:135-158 / training/episode_utils.py:42-53 applied to
 * every env independently, with the batched env's auto-reset in place of "construct a new env"
 * (respawn=1, evaluator.py:91) or "reuse the env object" (respawn=0, robustness_tests.py:260). */
typedef struct {
    dexo_env* e; int64_t lo, hi, n; const dexo_params* p; const dexo_group* groups;
    const uint16_t* group_of_env; const dexo_rollout_cfg* cfg; const float* actions;
    const float* dyn_noise; int64_t* counters; double* ret_sums; const dexo_learner* learner;
    int32_t err;
} rollout_job;

static void finish_episode(dexo_env* e, const dexo_params* p, const dexo_rollout_cfg* cfg,
                           int terminated, int64_t* cnt, double* rs) {
    const int success = cfg->success_is_terminated ? terminated : 0;
    const int la = dexo_classify_metrics(success, e->ep_steps, e->num_contacts, e->num_contacts,
                                         e->hist, e->ep_steps, cfg->loop_max_steps, p->success_threshold);
    const int lb = dexo_classify_taxonomy(success, e->ep_steps, e->num_contacts, e->num_contacts,
                                          e->hist, e->ep_steps, cfg->loop_max_steps, p->success_threshold, NULL);
    cnt[DEXO_CNT_EPISODES] += 1;
    cnt[DEXO_CNT_SUCCESSES] += success;
    cnt[DEXO_CNT_SUM_STEPS] += e->ep_steps;
    cnt[DEXO_CNT_SUM_STEPS_SQ] += (int64_t)e->ep_steps * e->ep_steps;
    cnt[DEXO_CNT_SUM_FINAL_CONTACTS] += e->num_contacts;
    if (la >= 0) cnt[DEXO_CNT_LABEL_METRICS + la] += 1;
    if (lb >= 0) cnt[DEXO_CNT_LABEL_TAXONOMY + lb] += 1;
    rs[0] += e->ep_return; rs[1] += e->ep_return * e->ep_return;
}

static void* rollout_worker(void* arg) {
    rollout_job* j = (rollout_job*)arg;
    const dexo_rollout_cfg* cfg = j->cfg;
    for (int64_t i = j->lo; i < j->hi; ++i) {
        dexo_env* e = &j->e[i];
        const uint32_t gid = (uint32_t)(cfg->env_gid0 + i);
        const int g = j->group_of_env ? j->group_of_env[i] : (int)(gid % (uint32_t)cfg->num_groups);
        const dexo_group* grp = &j->groups[g];
        int64_t* cnt = j->counters + (int64_t)g * DEXO_NCOUNTERS;   /* caller gives per-thread copies */
        double* rs = j->ret_sums + (int64_t)g * 2;
        for (int t = 0; t < cfg->k_steps; ++t) {
            float a[DEXO_NJ];
            const dexo_learner* L = j->learner;
            if (L) {                  /* SimpleLearner.select_action, policies/simple_learner.py:60-69 */
                const float* nz = L->act_noise + ((int64_t)t * j->n + i) * DEXO_NJ;
                for (int q = 0; q < DEXO_NJ; ++q) a[q] = clip_f32(L->mean[i * DEXO_NJ + q] + nz[q], -1.0f, 1.0f);
            }
            else if (cfg->policy_kind == 0) memcpy(a, j->actions + ((int64_t)t * j->n + i) * DEXO_NJ, sizeof a);
            else dexo_policy_action(cfg->seed, gid, e->episode, (uint32_t)e->step_count, cfg->policy_kind, a);
            const float* dn = j->dyn_noise ? j->dyn_noise + ((int64_t)t * j->n + i) * DEXO_NJ : NULL;
            dexo_reward r; int32_t te, tr;
            dexo_step_noisy(e, j->p, a, dn, NULL, NULL, &r, &te, &tr);
            if (L && r.total > L->best[i]) {                         /* SimpleLearner.update, :82-95 */
                const double* un = L->upd_noise + ((int64_t)t * j->n + i) * DEXO_NJ;
                for (int q = 0; q < DEXO_NJ; ++q) {
                    const float m = (float)((double)L->mean[i * DEXO_NJ + q] + un[q]);   /* float32 array += float64 array */
                    L->mean[i * DEXO_NJ + q] = clip_f32(m, -L->clip_range, L->clip_range);
                }
                L->best[i] = r.total;
            }
            e->ep_return += r.total;                                 /* evaluator.py:144 */
            if (e->ep_steps >= DEXO_HIST_MAX) { j->err = DEXO_E_HIST; return NULL; }   /* labels need every count */
            e->hist[e->ep_steps] = (uint8_t)e->num_contacts;
            e->ep_steps += 1;                                        /* evaluator.py:145 */
            if (te || tr || e->ep_steps >= cfg->loop_max_steps) {    /* evaluator.py:156, :135 */
                finish_episode(e, j->p, cfg, te, cnt, rs);
                if (L) L->best[i] = -INFINITY;                       /* policy.reset(), episode_utils.py:35-36 */
                e->episode += 1;
                float jp0[DEXO_NJ], pos[3]; double size, mass, fric;
                dexo_reset_draws(cfg->seed, gid, e->episode, grp, jp0, &size, &mass, &fric, pos);
                dexo_reset_predrawn(e, jp0, size, mass, fric, cfg->respawn ? pos : NULL);
            }
        }
    }
    return NULL;
}

static int32_t rollout_impl(dexo_env* e, int64_t n, const dexo_params* p, const dexo_group* groups,
                            const uint16_t* group_of_env, const dexo_rollout_cfg* cfg, const float* actions,
                            const float* dyn_noise, const dexo_learner* learner, int64_t* counters, double* ret_sums) {
    int threads = cfg->threads < 1 ? 1 : cfg->threads;
    if (threads > 256) threads = 256;
    if ((int64_t)threads > n) threads = (int)(n > 0 ? n : 1);
    const int G = cfg->num_groups;
    /* per-thread integer counters; the float64 return sums depend on the summation order, so
     * ret_sums is only bit-reproducible with threads == 1. */
    int64_t* tc = (int64_t*)calloc((size_t)threads * G * DEXO_NCOUNTERS, sizeof(int64_t));
    double* tr = (double*)calloc((size_t)threads * G * 2, sizeof(double));
    rollout_job jobs[256]; pthread_t tid[256];
    for (int t = 0; t < threads; ++t) {
        rollout_job j = {e, n * t / threads, n * (t + 1) / threads, n, p, groups, group_of_env, cfg,
                         actions, dyn_noise, tc + (size_t)t * G * DEXO_NCOUNTERS, tr + (size_t)t * G * 2, learner, 0};
        jobs[t] = j;
    }
    if (threads == 1) rollout_worker(&jobs[0]);
    else {
        for (int t = 0; t < threads; ++t) pthread_create(&tid[t], NULL, rollout_worker, &jobs[t]);
        for (int t = 0; t < threads; ++t) pthread_join(tid[t], NULL);
    }
    int32_t err = 0;
    for (int t = 0; t < threads; ++t) {
        for (int k = 0; k < G * DEXO_NCOUNTERS; ++k) counters[k] += tc[(size_t)t * G * DEXO_NCOUNTERS + k];
        for (int k = 0; k < G * 2; ++k) ret_sums[k] += tr[(size_t)t * G * 2 + k];
        if (jobs[t].err) err = jobs[t].err;
    }
    free(tc); free(tr);
    return err;
}

int32_t dexo_rollout(dexo_env* e, int64_t n, const dexo_params* p, const dexo_group* groups,
                     const uint16_t* group_of_env, const dexo_rollout_cfg* cfg, const float* actions,
                     const float* dyn_noise, int64_t* counters, double* ret_sums) {
    return rollout_impl(e, n, p, groups, group_of_env, cfg, actions, dyn_noise, NULL, counters, ret_sums);
}

int32_t dexo_rollout_learner(dexo_env* e, int64_t n, const dexo_params* p, const dexo_group* groups,
                             const uint16_t* group_of_env, const dexo_rollout_cfg* cfg, const dexo_learner* L,
                             int64_t* counters, double* ret_sums) {
    return rollout_impl(e, n, p, groups, group_of_env, cfg, NULL, NULL, L, counters, ret_sums);
}

int32_t dexo_sizeof_env(void) { return (int32_t)sizeof(dexo_env); }
int32_t dexo_sizeof_group(void) { return (int32_t)sizeof(dexo_group); }
