/*
 * dexsim_oracle.h -- CPU restatement of the reference's hot path.  TEST INFRASTRUCTURE ONLY.
 *
 * This is the parity oracle for the CUDA path in dexterous_rl_manipulation_b200/csrc/.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load it.  The product never links, imports or calls anything in this directory.
 *
 * PARITY PIN: the reference's own tests assert no observation / reward / flag values
 * (SURVEY.md section 4), so the restatement is pinned against outputs of the UNMODIFIED
 * reference executed in the build container (numpy 2.3.5, NEP 50 promotion) and committed
 * as tests/golden/ (npz files) by tests/golden/make_golden.py; and against the reference's asserted
 * failure-label known answers (tests/test_failure_taxonomy.py:73,106,142,176,212;
 * tests/test_evaluation_metrics.py:78,90,103).
 *
 * Every function cites the reference file:line (relative to the reference root) it follows.
 */
#ifndef DEXSIM_ORACLE_H
#define DEXSIM_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DEXO_NJ 15        /* num_fingers * joints_per_finger   envs/manipulation_env.py:52  */
#define DEXO_NF 5         /* num_fingers                        envs/manipulation_env.py:50  */
#define DEXO_JPF 3        /* joints_per_finger                  envs/manipulation_env.py:51  */
#define DEXO_OBS 45       /* 2*15 + 10 + 5                      envs/manipulation_env.py:96-106 */
/* per-step contact counts kept per env: the longest tracked episode the library accepts (5,242 steps, EPSTATS_MAX_STEPS
 * in dexterous_rl_manipulation_b200/csrc/dexsim_core.cuh) rounded up to a multiple of 8.  A longer episode is an error
 * of dexo_rollout, never a cut history. */
#define DEXO_HIST_MAX 5248

/* label codes: enum declaration order of FailureType (evaluation/metrics.py:15-22) and
 * FailureMode (evaluation/failure_taxonomy.py:14-26); -1 = success (classifier returns None) */
enum { DEXO_SLIPPAGE = 0, DEXO_UNSTABLE = 1, DEXO_MISALIGNED = 2, DEXO_TIMEOUT = 3,
       DEXO_DROPPED = 4, DEXO_INSUFFICIENT = 5, DEXO_NLABELS = 6 };

/* counters per group (same layout as include/dexsim.h) */
enum { DEXO_CNT_EPISODES = 0, DEXO_CNT_SUCCESSES = 1, DEXO_CNT_SUM_STEPS = 2,
       DEXO_CNT_SUM_FINAL_CONTACTS = 3, DEXO_CNT_LABEL_METRICS = 4, DEXO_CNT_LABEL_TAXONOMY = 10,
       DEXO_CNT_VAR_TIES = 16, DEXO_CNT_SUM_STEPS_SQ = 17, DEXO_NCOUNTERS = 18 };

typedef struct {
    /* RewardShaping weights, rewards/reward_shaping.py:20-39 */
    double w_distance, w_contact, w_closure, w_stability;
    int32_t reward_type;        /* 0 = sparse (rewards/reward_shaping.py:190), 1 = dense (:12) */
    int32_t max_episode_steps;  /* envs/manipulation_env.py:53 */
    int32_t success_threshold;  /* 3: envs/manipulation_env.py:336 */
    int32_t pad_;
} dexo_params;

/* One CurriculumConfig (experiments/config.py:17-42) plus the noise levels of one
 * robustness cell (evaluation/robustness_tests.py:145-164). */
typedef struct {
    double size, mass, friction;
    double size_lo, size_hi;   int32_t size_ranged;      int32_t pad0_;
    double mass_lo, mass_hi;   int32_t mass_ranged;      int32_t pad1_;
    double fric_lo, fric_hi;   int32_t fric_ranged;      int32_t pad2_;
    double spawn_lo[3], spawn_hi[3];
    float sigma_obs, sigma_dyn;
} dexo_group;

typedef struct {
    float   jp[DEXO_NJ];
    float   jv[DEXO_NJ];
    double  op[3];
    float   ov[3];
    float   c[DEXO_NF];
    float   prev_c[DEXO_NF];
    int32_t has_prev;           /* RewardShaping.prev_contacts is not None */
    int32_t step_count;
    int32_t op_is_f32;          /* object_position is still the float32 array made by reset() */
    int32_t num_contacts;
    double  size, mass, friction;
    /* episode record, evaluation/evaluator.py:118-173 */
    double  ep_return;
    int32_t ep_steps;
    uint32_t episode;           /* Philox episode counter */
    uint8_t hist[DEXO_HIST_MAX];/* per-step contact COUNTS (evaluator.py:148-150 count-encodes) */
} dexo_env;

typedef struct {
    double  total, distance, contact, closure, stability;
} dexo_reward;

/* ---- core path ---------------------------------------------------------------------- */
void dexo_default_params(dexo_params* p, int dense);
void dexo_reset_predrawn(dexo_env* e, const float* jp0, double size, double mass,
                         double friction, const float* pos /* NULL: keep position */);
void dexo_step(dexo_env* e, const dexo_params* p, const float* action,
               float* obs, dexo_reward* rew, int32_t* terminated, int32_t* truncated);
void dexo_step_noisy(dexo_env* e, const dexo_params* p, const float* action,
                     const float* dyn_noise /* [15] or NULL */, const float* obs_noise /* [45] or NULL */,
                     float* obs, dexo_reward* rew, int32_t* terminated, int32_t* truncated);
void dexo_observation(const dexo_env* e, float* obs);

/* batch wrappers (envs are independent; plain loops, optionally split over pthreads) */
void dexo_reset_predrawn_batch(dexo_env* e, int64_t n, const float* jp0 /* [n,15] */,
                               const double* size, const double* mass, const double* friction,
                               const float* pos /* [n,3] or NULL */);
void dexo_step_batch(dexo_env* e, int64_t n, const dexo_params* p, const float* action /* [n,15] */,
                     const float* dyn_noise /* [n,15] or NULL */, const float* obs_noise /* [n,45] or NULL */,
                     float* obs /* [n,45] */, double* reward /* [n] */, double* comps /* [n,4] or NULL */,
                     uint8_t* terminated, uint8_t* truncated, uint8_t* num_contacts, int32_t threads);

/* ---- failure labels ----------------------------------------------------------------- */
double dexo_np_var_counts(const uint8_t* counts, int64_t n);
int32_t dexo_classify_metrics(int32_t success, int32_t episode_steps, int32_t num_contacts,
                              int32_t final_contacts, const uint8_t* counts, int64_t len,
                              int32_t max_steps, int32_t success_threshold);
int32_t dexo_classify_taxonomy(int32_t success, int32_t episode_steps, int32_t num_contacts,
                               int32_t final_contacts, const uint8_t* counts, int64_t len,
                               int32_t max_steps, int32_t success_threshold, double* confidence);

/* ---- counter-based RNG spec (shared with the device by specification, not by code) ---- */
void dexo_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
void dexo_reset_draws(uint64_t seed, uint32_t env_gid, uint32_t episode, const dexo_group* g,
                      float* jp0 /* [15] */, double* size, double* mass, double* friction,
                      float* pos /* [3] */);
void dexo_policy_action(uint64_t seed, uint32_t env_gid, uint32_t episode, uint32_t step,
                        int32_t policy_kind /* 1 random, 2 heuristic */, float* action /* [15] */);
/* Box-Muller on Philox words in double precision (the spec the device's float32 draws approximate) */
void dexo_normal_pair_ref(const uint32_t* wa, const uint32_t* wb, int64_t n, double* z0 /* [n] */, double* z1 /* [n] */);
void dexo_normal_rows_ref(uint64_t seed, const uint32_t* env_gid, const uint32_t* episode, const uint32_t* step,
                          int64_t n /* envs */, uint32_t stream /* 2..5 */, int32_t rows, double sigma,
                          double* out /* [n, rows] */);

/* ---- fused rollout restatement (auto-reset, in-"kernel" policy, counters) -------------- */
typedef struct {
    uint64_t seed;
    int64_t  env_gid0;          /* global id of e[0] (shard offset) */
    int32_t  k_steps;
    int32_t  policy_kind;       /* 0 external, 1 random, 2 heuristic */
    int32_t  respawn;           /* 1: fresh-env reset (evaluator.py:91), 0: keep position (reused env) */
    int32_t  success_is_terminated; /* 1: evaluator.py:156-158, 0: episode_utils.py:52 (always False) */
    int32_t  loop_max_steps;    /* caller's loop bound, evaluator.py:135 / episode_utils.py:38 */
    int32_t  num_groups;
    int32_t  threads;
    int32_t  pad_;
} dexo_rollout_cfg;

/* Returns 0, or DEXO_E_HIST when an episode outgrew the history (DEXO_HIST_MAX steps); the envs are then left
 * mid-step and the call's outputs are meaningless. */
enum { DEXO_E_HIST = 1 };
int32_t dexo_rollout(dexo_env* e, int64_t n, const dexo_params* p, const dexo_group* groups,
                     const uint16_t* group_of_env /* [n] or NULL: gid % num_groups */,
                     const dexo_rollout_cfg* cfg,
                     const float* actions /* [k,n,15] for policy 0 */,
                     const float* dyn_noise /* [k,n,15] or NULL */,
                     int64_t* counters /* [num_groups, DEXO_NCOUNTERS] accumulated */,
                     double* ret_sums /* [num_groups, 2]: sum, sum of squares of episode returns */);

/* SimpleLearner (policies/simple_learner.py:13-95) as a per-env policy inside the rollout:
 * mean[n,15] float32 and best[n] float64 persist across calls; the normal draws of select_action
 * (:60-64, sigma = exploration noise, cast to float32) and update (:84-88, sigma = learning rate,
 * float64 like the reference's) are PRE-DRAWN by the caller. */
typedef struct {
    float*  mean;              /* [n, 15] in/out */
    double* best;              /* [n] in/out; -inf after policy.reset() */
    const float* act_noise;    /* [k, n, 15] already scaled by exploration_noise */
    const double* upd_noise;   /* [k, n, 15] float64, already scaled by learning_rate */
    float   clip_range;        /* action_clip_range, :90-94 */
    int32_t pad_;
} dexo_learner;

int32_t dexo_rollout_learner(dexo_env* e, int64_t n, const dexo_params* p, const dexo_group* groups,
                             const uint16_t* group_of_env, const dexo_rollout_cfg* cfg, const dexo_learner* L,
                             int64_t* counters, double* ret_sums);

int32_t dexo_sizeof_env(void);
int32_t dexo_sizeof_group(void);

#ifdef __cplusplus
}
#endif
#endif
