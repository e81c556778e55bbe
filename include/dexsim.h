/*
 * dexsim.h -- C ABI of the B200-native batched manipulation simulator (libdexsim_b200.so).
 *
 * The reference (I2S9/dexterous-rl-manipulation) has no FFI or plugin registry: the boundary
 * its callers use is the duck-typed Gymnasium env object (SURVEY.md 8b).  The Python class
 * dexterous_rl_manipulation_b200.BatchedManipulationEnv mirrors that object and calls the
 * entry points below through ctypes; INTEGRATION.md shows the binding.  Each entry point names
 * the reference interface it replaces (file:line relative to the reference root).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / C++ types.
 *   - Every pointer in DexsimState / DexsimStepIO is a DEVICE pointer owned by the caller
 *     (the Python side allocates them as torch tensors); the *_host entry points take HOST
 *     pointers (pinned for full speed) and are documented as such.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).  Calls are
 *     asynchronous on that stream unless stated; no allocation and no per-call global state
 *     (the only process-wide switches are dexsim_set_step_impl / dexsim_set_rollout_impl, for tests
 *     and profiling) => thread-safe per (device, stream).  dexsim_step_host forks onto a few internal
 *     streams per device, joins them into `stream` and (unless DEXSIM_HOST_ASYNC) synchronizes it before
 *     returning; concurrent callers on the SAME device are serialised while they enqueue.
 *   - Return value: 0 = ok; negative cudaError_t (-e) for CUDA failures; DEXSIM_E_* for
 *     argument errors.  No exceptions cross the boundary.  dexsim_error_string() explains.
 *   - Per-env arrays are structure-of-arrays with leading dimension `ld` (>= n, multiple of
 *     32 so every row starts 128-byte aligned): field f of env i lives at base[f * ld + i].
 *   - Only num_fingers = 5, joints_per_finger = 3 is built (the only geometry any reference
 *     config uses: experiments/experiment_config.py:32-33); other geometries are rejected by
 *     the Python face with DEXSIM_E_GEOMETRY semantics.
 */
#ifndef DEXSIM_H
#define DEXSIM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DEXSIM_ABI_VERSION 3
#define DEXSIM_NJ 15      /* joints            envs/manipulation_env.py:52 */
#define DEXSIM_NF 5       /* fingers           envs/manipulation_env.py:50 */
#define DEXSIM_OBS 45     /* observation width envs/manipulation_env.py:96-106 */

/* observation rows (envs/manipulation_env.py:254-264) */
#define DEXSIM_ROW_JP 0
#define DEXSIM_ROW_JV 15
#define DEXSIM_ROW_OP 30
#define DEXSIM_ROW_QUAT 33
#define DEXSIM_ROW_OV 37
#define DEXSIM_ROW_CONTACT 40

/* error codes */
#define DEXSIM_OK 0
#define DEXSIM_E_NULL (-1001)        /* required pointer is NULL */
#define DEXSIM_E_SIZE (-1002)        /* n < 0, ld < n, ld % 32 != 0, k_steps < 1 ... */
#define DEXSIM_E_ALIGN (-1003)       /* a row base is not 16-byte aligned */
#define DEXSIM_E_PARAM (-1004)       /* bad enum / flag / parameter value (e.g. tracked episodes longer than 5,242 steps) */
#define DEXSIM_E_GROUPS (-1005)      /* num_groups out of range [1, DEXSIM_MAX_GROUPS] */
#define DEXSIM_E_GEOMETRY (-1006)    /* unsupported num_fingers / joints_per_finger */

#define DEXSIM_MAX_GROUPS 256

/* policy kinds (policies/random_policy.py:40, policies/heuristic_policy.py:55-62) */
#define DEXSIM_POLICY_EXTERNAL 0
#define DEXSIM_POLICY_RANDOM 1
#define DEXSIM_POLICY_HEURISTIC 2
#define DEXSIM_POLICY_LEARNER 3      /* per-env SimpleLearner, policies/simple_learner.py:13-95 */

/* failure-label codes = enum declaration order of FailureType (evaluation/metrics.py:15-22)
 * and FailureMode (evaluation/failure_taxonomy.py:14-26) */
#define DEXSIM_LABEL_SLIPPAGE 0
#define DEXSIM_LABEL_UNSTABLE 1
#define DEXSIM_LABEL_MISALIGNED 2
#define DEXSIM_LABEL_TIMEOUT 3
#define DEXSIM_LABEL_DROPPED 4
#define DEXSIM_LABEL_INSUFFICIENT 5
#define DEXSIM_LABEL_NONE 255

/* per-group int64 counters written by rollouts / auto-reset (one row per group) */
#define DEXSIM_CNT_EPISODES 0
#define DEXSIM_CNT_SUCCESSES 1
#define DEXSIM_CNT_SUM_STEPS 2
#define DEXSIM_CNT_SUM_FINAL_CONTACTS 3
#define DEXSIM_CNT_LABEL_METRICS 4      /* +label code, 6 slots: evaluation/metrics.py:39-96 */
#define DEXSIM_CNT_LABEL_TAXONOMY 10    /* +label code, 6 slots: evaluation/failure_taxonomy.py:156-239 */
#define DEXSIM_CNT_VAR_TIES 16          /* episodes whose contact-count variance sat exactly on a threshold AND whose
                                         * history was not at hand to decide it the way np.var does (var_tie == 1) */
#define DEXSIM_CNT_SUM_STEPS_SQ 17
#define DEXSIM_NCOUNTERS 18

/*
 * Device-resident state of one shard of n envs.  `obs` doubles as the hot state: its rows ARE
 * the observation (quaternion rows are written once at reset), so stepping produces the
 * observation tensor for free.  The float64 object position and contact threshold exist
 * because the reference's contact test is (accidentally) float64 (SURVEY.md 8a-3/8a-4).
 */
typedef struct DexsimState {
    int64_t   n;           /* envs in this shard */
    int64_t   ld;          /* leading dimension of every per-env array */
    float*    obs;         /* [45, ld]  hot state == observation, envs/manipulation_env.py:254-264 */
    double*   op64;        /* [3, ld]   object_position in float64, :222-229 */
    double*   thr;         /* [ld]      object_size * 1.5 (float64), :293 */
    float*    damp;        /* [ld]      float32(1.0 - friction * 0.1 * dt), :215-216 */
    int32_t*  step_count;  /* [ld]      :173,247 */
    uint8_t*  cmask;       /* [ld]      bit f = finger f in contact after the last step (RewardShaping.prev_contacts) */
    double*   size;        /* [ld]      info["curriculum"]["object_size"], :273 */
    double*   mass;        /* [ld]      info["curriculum"]["object_mass"], :274 */
    double*   friction;    /* [ld]      info["curriculum"]["friction_coefficient"], :275 */
    uint32_t* episode;     /* [ld]      episodes finished by this env (Philox counter word) */
    double*   ep_return;   /* [ld]      running episode return (float64 like evaluator.py:144); NULL = not tracked */
    uint32_t* ep_stats;    /* [2, ld]   packed contact-count history summary; NULL = not tracked.  Holds episodes of up to
                            *           5,242 steps: calls that could run a tracked episode longer than that
                            *           (min(loop_max_steps, max_episode_steps + 1)) return DEXSIM_E_PARAM */
} DexsimState;

/* Scalars of one DexterousManipulationEnv construction + the batched env's own switches. */
typedef struct DexsimParams {
    double   w_distance, w_contact, w_closure, w_stability; /* rewards/reward_shaping.py:20-25 */
    int32_t  reward_type;            /* 0 sparse (rewards/reward_shaping.py:190), 1 dense (:12) */
    int32_t  max_episode_steps;      /* envs/manipulation_env.py:28 */
    int32_t  success_threshold;      /* 3, envs/manipulation_env.py:336 */
    int32_t  auto_reset;             /* 1: an env that finishes an episode is reset in the same launch */
    int32_t  respawn;                /* auto-reset mode: 1 fresh env (evaluator.py:91), 0 reused env keeps position (:160-161) */
    int32_t  success_is_terminated;  /* 1: evaluator.py:156-158; 0: episode_utils.py:52 (always False) */
    int32_t  loop_max_steps;         /* caller's loop bound (evaluator.py:135, episode_utils.py:38); <=0: none */
    int32_t  num_groups;             /* rows of the group table */
    uint64_t seed;                   /* Philox key */
    int64_t  env_gid0;               /* global id of env 0 of this shard (multi-GPU: rank offset) */
} DexsimParams;

/* One CurriculumConfig (experiments/config.py:17-42) + one robustness cell's noise levels
 * (evaluation/robustness_tests.py:145-164).  Staged in shared memory by the kernels. */
typedef struct DexsimGroup {
    double  size, mass, friction;
    double  size_lo, size_hi;  int32_t size_ranged;  int32_t pad0_;
    double  mass_lo, mass_hi;  int32_t mass_ranged;  int32_t pad1_;
    double  fric_lo, fric_hi;  int32_t fric_ranged;  int32_t pad2_;
    double  spawn_lo[3], spawn_hi[3];
    float   sigma_obs, sigma_dyn;
} DexsimGroup;

/* DexsimStepIO.flags: walk the batch from its last tile to its first.  A caller that steps the same state repeatedly
 * alternates this bit from call to call (the Python face does): what the previous step touched last is what is still in
 * the 126 MB L2 -- reads of those tiles hit, and their stores overwrite lines that are still dirty instead of costing a
 * write-back.  Results do not depend on it. */
#define DEXSIM_STEP_REVERSE_TILES 1
/* DexsimStepIO.flags, with host_static_rows set (pipelined kernel only; other configurations answer DEXSIM_E_PARAM):
 * write the observation into the host buffer as part of the step, not just rows 30/31/37/38 -- each tile's 30 joint
 * rows by a second bulk tensor store, object z (row 32) and its velocity (row 39) as two more row segments, and the
 * 1-byte contact masks into host_cmask (the five 0/1 contact rows 40-44 are NOT written: they follow from the mask,
 * dexsim_expand_contact_rows).  With the per-env outputs pointing at mapped host memory too, nothing is left to
 * download (dexsim_step_host: DEXSIM_HOST_ZERO_COPY). */
#define DEXSIM_STEP_HOST_ALL_ROWS 2

/* Inputs / outputs of one batched step (all device pointers, SoA with the state's ld). */
typedef struct DexsimStepIO {
    const float* action;        /* [15, ld] (layout 0) or [n, 15] (layout 1); required for dexsim_step.  A 16-byte aligned
                                 * base takes the vectorised / bulk-copy paths; any other alignment (e.g. an [n,15] slice
                                 * that starts at an odd env) is read with scalar loads by the register-resident kernel. */
    int32_t      action_layout; /* 0 = SoA [15, ld], 1 = AoS [n, 15] (the reference's per-env layout) */
    int32_t      flags;         /* DEXSIM_STEP_* bits */
    const float* dyn_noise;     /* [15, ld] pre-drawn float32 N(0, sigma_dyn) or NULL (robustness_tests.py:180-187) */
    const float* obs_noise;     /* [45, ld] pre-drawn float32 N(0, sigma_obs) or NULL (:204-205) */
    float*       noisy_obs;     /* [45, ld] out: obs + noise; required iff obs noise is on */
    float*       reward;        /* [ld] out, float32(total) */
    float*       reward_comps;  /* [4, ld] out (distance, contact, closure, stability) or NULL */
    uint8_t*     terminated;    /* [ld] out 0/1 */
    uint8_t*     truncated;     /* [ld] out 0/1 */
    uint8_t*     num_contacts;  /* [ld] out 0..5, info["num_contacts"] */
    uint8_t*     finished;      /* [ld] out 0/1: episode ended this step and the env was auto-reset; or NULL */
    int64_t*     counters;      /* [num_groups, DEXSIM_NCOUNTERS] accumulated; or NULL */
    double*      ret_sums;      /* [num_groups, 2] sum and sum of squares of episode returns; or NULL */
    double*      reward64;      /* [ld] out: the float64 total exactly as the reference returns it (Python float); or NULL.
                                 * Needed by callers that compare rewards (SimpleLearner.update); served by the
                                 * register-resident kernel. */
    /* Noise drawn INSIDE the step kernel (Philox normals, the streams dexsim_fill_normal exposes), used when the
     * corresponding pre-drawn pointer above is NULL:  > 0 = this standard deviation for every env,  < 0 = each env's
     * group value (DexsimGroup.sigma_dyn / sigma_obs; needs the group table),  0 = off.
     * sigma_dyn: a <- clip(a + N(0, sigma), -1, 1) keyed by (episode, step count BEFORE the step)
     * (robustness_tests.py:180-187);  sigma_obs: noisy_obs <- obs + N(0, sigma) for all 45 entries, keyed by
     * (episode, step count AFTER the step and a possible auto-reset) (:204-205); needs `noisy_obs`. */
    float        sigma_dyn;
    float        sigma_obs;
    /* Scratch of the pipelined step kernel's dynamic tile scheduler: DEXSIM_SCHED_WORDS zero-initialised device words,
     * or NULL = static round-robin tile assignment.  The kernel hands tiles to its CTAs from a counter kept here and
     * leaves the words zero again; one buffer per step that can be in flight at a time (calls on the same stream may
     * share it).  dexsim_step uses words 0-1, dexsim_step_host words 2c, 2c+1 for its chunk c. */
    uint32_t*    sched;
    /* Host mirror of the observation rows that only change when an episode is reset: object x, y (rows 30, 31) and
     * their velocities (rows 37, 38).  When set -- a pointer to the caller's HOST [45, ld] observation buffer in mapped
     * page-locked memory (any cudaHostAlloc / pinned allocation under unified addressing) -- every change of those four
     * entries is ALSO written there by the step kernel (a handful of 4-byte stores per reset), so a caller that downloads
     * the observation every step need not download these rows (dexsim_step_host: DEXSIM_HOST_STATIC_ROWS).  NULL = off. */
    float*       host_static_rows;
    /* With DEXSIM_STEP_HOST_ALL_ROWS in `flags` (pipelined kernel only): host copy of the 1-byte contact masks
     * (DexsimState.cmask), written every step; or NULL. */
    uint8_t*     host_cmask;
} DexsimStepIO;
#define DEXSIM_SCHED_WORDS 64

/* ---- library ---------------------------------------------------------------------------- */
int         dexsim_version(void);            /* DEXSIM_ABI_VERSION */
const char* dexsim_error_string(int code);
int         dexsim_sizeof_state(void);
int         dexsim_sizeof_params(void);
int         dexsim_sizeof_group(void);
int         dexsim_sizeof_step_io(void);
int         dexsim_sizeof_rollout_io(void);
int         dexsim_sizeof_episode_record(void);
/* SM count and max resident CTAs per SM of the step kernel on the current device */
int         dexsim_device_info(int* sm_count, int* step_ctas_per_sm, int* rollout_ctas_per_sm);
/* Which step kernel dexsim_step uses: 0 = auto (TMA/mbarrier pipeline when eligible, else the
 * register-resident kernel), 1 = register-resident only, 2 = TMA pipeline required (dexsim_step
 * returns DEXSIM_E_PARAM when a call is not eligible).  Both produce identical results; the switch
 * exists for tests and profiling.  Process-wide. */
int         dexsim_set_step_impl(int impl);
/* Tile width of the TMA pipeline: 0 = auto (by batch size), 1 = narrow tiles only (128 envs, 3 CTAs x 4 compute warps per
 * SM), 2 = wide tiles (224 envs, 2 CTAs x 7 compute warps per SM) wherever that instantiation exists (every step without
 * full per-env episode tracking).  Identical results; for tests and profiling.  Process-wide. */
int         dexsim_set_step_tile(int tile);
/* Which fused-rollout kernel dexsim_rollout uses: 0 = auto (the 5-lanes-per-env kernel for small batches with an
 * in-kernel policy and no dynamics noise, else one thread per env), 1 = one thread per env, 2 = 5 lanes per env
 * whenever eligible.  Identical results; for tests and profiling.  Process-wide. */
int         dexsim_set_rollout_impl(int impl);

/* ---- reset: replaces DexterousManipulationEnv.reset, envs/manipulation_env.py:124-182 ------ */
/* Host-sampled draws (exactly the reference's PCG64 draws when the Python face samples them):
 * jp0 [15, ld]; size/mass/friction [ld] float64; pos [3, ld] float32 or NULL = keep the current
 * position cast to float32 (:160-161).  mask [ld] 0/1 or NULL = all envs. */
int dexsim_reset_predrawn(const DexsimState* st, const DexsimParams* p, const uint8_t* mask,
                          const float* jp0, const double* size, const double* mass,
                          const double* friction, const float* pos, void* stream);
/* Device-sampled draws: Philox4x32-10 keyed by p->seed, counter (env gid, episode, 0, stream 0),
 * same draw order and distributions as :143-161 + experiments/config.py:44-113. */
int dexsim_reset_philox(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                        const uint16_t* group_of_env, const uint8_t* mask, int32_t respawn,
                        void* stream);

/* ---- step: replaces DexterousManipulationEnv.step, envs/manipulation_env.py:184-252,
 *      RewardShaping.compute / SparseReward.compute (rewards/reward_shaping.py:50-99,205-242)
 *      and CombinedNoiseWrapper.step (evaluation/robustness_tests.py:177-207) ---------------- */
int dexsim_step(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                const uint16_t* group_of_env, const DexsimStepIO* io, void* stream);

/* ---- fused rollout: replaces the caller loops training/episode_utils.py:42-53,
 *      evaluation/evaluator.py:135-158, evaluation/robustness_tests.py:292-304 with the policy
 *      (policies/random_policy.py:40 / policies/heuristic_policy.py:55-62) generated in-kernel.
 *      k_steps env-steps per env in ONE launch, state in registers, episodes auto-reset. ------ */

#define DEXSIM_ROLLOUT_NO_DYN_NOISE 1   /* caller asserts that no group has sigma_dyn > 0 (enables the small-batch kernel) */

/* One finished episode = the per-episode dict of evaluation/evaluator.py:163-173 (32 bytes). */
typedef struct DexsimEpisodeRecord {
    uint32_t env_gid;          /* global env id */
    uint32_t episode;          /* which episode of that env finished (0 = first after reset(seed)) */
    int32_t  steps;            /* "episode_steps" */
    uint8_t  success;          /* "success" (terminated, or 0 when success_is_terminated == 0) */
    uint8_t  final_contacts;   /* "num_contacts" == "final_contacts" */
    uint8_t  label_metrics;    /* evaluation/metrics.py label code or DEXSIM_LABEL_NONE */
    uint8_t  label_taxonomy;   /* evaluation/failure_taxonomy.py label code or DEXSIM_LABEL_NONE */
    double   episode_reward;   /* "episode_reward", float64 running sum */
    uint32_t t_end;            /* step_base + index of the step that ended the episode */
    uint32_t var_tie;          /* a variance threshold was hit exactly: 2 = decided by NumPy's np.var arithmetic on the recorded
                                * history (DexsimRolloutIO.hist), label exact; 1 = no history recorded, label resolved as in
                                * exact arithmetic -- re-label it with dexsim_classify_summary(counts) */
} DexsimEpisodeRecord;

typedef struct DexsimRolloutIO {
    const float* actions;      /* [k, 15, ld] for DEXSIM_POLICY_EXTERNAL, else NULL */
    const float* dyn_noise;    /* [k, 15, ld] pre-drawn, or NULL = Philox when the group's sigma_dyn > 0 */
    int64_t*     counters;     /* [num_groups, DEXSIM_NCOUNTERS] accumulated, or NULL */
    double*      ret_sums;     /* [num_groups, 2] or NULL */
    DexsimEpisodeRecord* ep_log;   /* [ep_log_capacity] or NULL */
    uint64_t*    ep_log_count; /* device scalar: records produced so far; records beyond capacity are dropped */
    int64_t      ep_log_capacity;
    uint8_t*     hist;         /* [hist_steps, ld] per-step contact counts (evaluator.py:148-150) or NULL */
    int64_t      hist_steps;   /* rows of hist; steps with step_base + t >= hist_steps are not recorded */
    int64_t      step_base;    /* index of this launch's first step (for t_end and hist rows) */
    int32_t      one_episode;  /* 1: an env stops at the end of its first episode of this launch and is NOT reset
                                * (run_episode / evaluate_episode semantics: the caller resets it) */
    int32_t      flags;        /* DEXSIM_ROLLOUT_* */
    /* DEXSIM_POLICY_LEARNER: one independent SimpleLearner per env (policies/simple_learner.py).
     * action = clip(mean + float32 N(0, exploration)) (:60-69); after every step, if reward > best:
     * mean = clip(float32(mean + float64 N(0, lr)), +-clip), best = reward (:82-95); best = -inf at
     * every episode start (policy.reset(), training/episode_utils.py:35-36). */
    float*       learner_mean;       /* [15, ld] float32 in/out */
    double*      learner_best;       /* [ld] float64 in/out */
    const float* learner_act_noise;  /* [k, 15, ld] pre-drawn (already scaled) or NULL = Philox stream 4 */
    const double* learner_upd_noise; /* [k, 15, ld] pre-drawn float64 (already scaled) or NULL = Philox stream 5 */
    float        learner_exploration, learner_lr, learner_clip;
    int32_t      pad2_;
} DexsimRolloutIO;

int dexsim_rollout(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                   const uint16_t* group_of_env, int32_t k_steps, int32_t policy_kind,
                   const DexsimRolloutIO* rio, void* stream);

/* ---- single-env read-back: everything the reference's step()/reset() return for env `index`, packed into
 *      64 float64 on the device (one launch + one small D2H instead of a dozen scalar reads):
 *      [0..44] obs (noisy_obs if given), 45 reward, 46 terminated, 47 truncated, 48 num_contacts, 49 step_count,
 *      50..52 object_position (float64), 53 size, 54 mass, 55 friction, 56..59 reward components, 60 finished.
 *      Serves the num_envs == 1 drop-in path (info dict of envs/manipulation_env.py:266-283). ------------------- */
int dexsim_pack_env(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset,
                    double* out64 /* device [64] */, void* stream);

/* Same, for a host that polls instead of synchronizing the stream: `out64` may be page-locked host memory that is
 * mapped into the device address space (cudaHostAlloc under unified addressing -- the kernel writes straight into
 * it, no copy); slot 63 receives `tag` AFTER slots 0..62 are visible system-wide, so a host thread that reads
 * out64[63] == tag may read the other slots.  Use a tag that differs from the previous call's.  `io->action` of the
 * preceding dexsim_step may likewise point to mapped page-locked host memory when n is small. */
int dexsim_pack_env_tagged(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset,
                           double* out64 /* device or mapped host [64] */, double tag, void* stream);

/* dexsim_step for a batch of ONE env (st->n == 1) with the tagged read-back of env 0 done by the same launch: what
 * DexterousManipulationEnv.step returns (envs/manipulation_env.py:184-283) in one kernel and no copy call when
 * `io->action` and `out64` are mapped page-locked host memory.  Same arguments as dexsim_step + dexsim_pack_env_tagged. */
int dexsim_step_single(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                       const uint16_t* group_of_env, const DexsimStepIO* io,
                       double* out64 /* device or mapped host [64] */, double tag, void* stream);

/* ---- RNG exposure (so tests can pre-draw exactly what the fused kernels draw) ---------------- */
int dexsim_fill_policy_actions(const DexsimState* st, const DexsimParams* p, int32_t policy_kind,
                               float* actions /* [15, ld] for each env's CURRENT (episode, step) */,
                               void* stream);
int dexsim_fill_normal(const DexsimState* st, const DexsimParams* p,
                       int32_t rng_stream /* 2 dyn, 3 obs, 4 learner exploration, 5 learner update */,
                       int32_t rows /* 15 or 45 */, float sigma, float* out /* [rows, ld] */, void* stream);

/* ---- failure labels from episode summaries: replaces EvaluationMetrics.classify_failure
 *      (evaluation/metrics.py:39-96) and FailureClassifier.classify
 *      (evaluation/failure_taxonomy.py:156-239).  HOST function (pure integer/IEEE arithmetic). -- */
typedef struct DexsimEpisodeSummary {
    int32_t success, episode_steps, num_contacts, final_contacts;
    int32_t hist_len;          /* len(contact_history) */
    int32_t max_count, sum_counts, sum_sq_counts;
    int32_t first5_sum, last5_sum;
} DexsimEpisodeSummary;
/* `counts`: the hist_len per-step contact counts (host pointer) or NULL.  Both classifiers threshold
 * np.var(contact_counts) (metrics.py:77-80, failure_taxonomy.py:189,219-230).  The summary decides every case except an
 * exact tie with a threshold, where NumPy's pairwise float64 sum can land on either side: with `counts` the tie is
 * decided by the same arithmetic np.var performs (*var_tie = 2, labels bit-exact); without it as in exact arithmetic
 * (*var_tie = 1, label unconfirmed).  *var_tie = 0: no tie, the labels are exact either way. */
int dexsim_classify_summary(const DexsimEpisodeSummary* s, const uint8_t* counts /* [hist_len] or NULL */,
                            int32_t max_steps, int32_t success_threshold,
                            int32_t* label_metrics, int32_t* label_taxonomy, int32_t* var_tie);

/* ---- host-buffer step (end-to-end path): actions in HOST memory -> device -> step ->
 *      obs / reward / flags back to HOST memory, synchronous on return unless DEXSIM_HOST_ASYNC.  Pinned buffers make
 *      the copies asynchronous DMA; pageable buffers work but stage through the driver.  With chunks > 1
 *      the envs are split into that many ranges whose H2D copy, kernel and D2H copies overlap on
 *      internal streams (created once per device, forked from / joined into `stream`).
 *      This is what a caller that keeps NumPy-side policies uses in place of
 *      `obs, r, term, trunc, info = env.step(action)` (envs/manipulation_env.py:184). ------------------ */
#define DEXSIM_HOST_SKIP_QUAT 1        /* do not copy obs rows 33-36 (constant quaternion, already in h_obs) */
#define DEXSIM_HOST_ASYNC 2            /* return without synchronizing: every copy is ordered before later work on `stream`;
                                        * the host buffers are valid once the caller has synchronized that stream (or an
                                        * event recorded on it).  Lets the upload of the next step (or of another env
                                        * group) overlap this step's download. */
#define DEXSIM_HOST_PACKED_CONTACTS 4  /* lossless narrower download: obs rows 40-44 (five 0/1 floats per env) stay on
                                        * the device and the 1-byte contact mask (bit f = finger f, DexsimState.cmask) is
                                        * copied to h_contact_mask instead (-19 bytes of 171 per env); the caller expands
                                        * the rows on the host if and when it needs them */
#define DEXSIM_HOST_STATIC_ROWS 16     /* h_obs is mapped page-locked memory whose rows 30, 31, 37, 38 are already current (a
                                        * previous dexsim_step_host call on the same buffer copied them and no other entry point has
                                        * touched the state since): do not download them -- the step kernel mirrors every change of
                                        * those entries straight into h_obs (DexsimStepIO.host_static_rows, set by this call).
                                        * Without the flag the rows are downloaded like the others (and the buffer becomes current). */
#define DEXSIM_HOST_ZERO_COPY 32       /* with PACKED_CONTACTS: every host output buffer of this call is mapped page-locked memory
                                        * and h_obs is current in the STATIC_ROWS sense: the step kernel writes the results
                                        * (joint rows, z, its velocity, contact masks, reward, flags) into the host buffers
                                        * itself, tile by tile, as part of the launch (DEXSIM_STEP_HOST_ALL_ROWS) -- no
                                        * device-to-host copies.  In this mode the per-env outputs exist ONLY in the host buffers
                                        * (io->reward / terminated / truncated / num_contacts on the device are not written).
                                        * Falls back to the copy transport when a buffer is not mapped, the batch is below one
                                        * tile or the pipelined kernel is not eligible. */
#define DEXSIM_HOST_EXPAND_CONTACTS 8  /* with PACKED_CONTACTS (and not ASYNC): the calling thread writes obs rows 40-44 of h_obs
                                        * from the masks while the other rows are still being downloaded, so h_obs is complete
                                        * on return although the five rows never crossed PCIe */
int dexsim_step_host(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                     const uint16_t* group_of_env, const DexsimStepIO* io /* device scratch */,
                     const float* h_action /* host [n, 15] (layout 1) or [15, ld] (layout 0) */,
                     float* h_obs /* host [45, ld] or NULL */, float* h_reward /* host [ld] */,
                     uint8_t* h_terminated, uint8_t* h_truncated, uint8_t* h_num_contacts /* host [ld] or NULL */,
                     uint8_t* h_contact_mask /* host [ld]: filled whenever given; required with DEXSIM_HOST_PACKED_CONTACTS */,
                     int32_t chunks, int32_t flags, void* stream);

/* Diagnostic: how many dexsim_step_host calls of this process were served by the DEXSIM_HOST_ZERO_COPY launch. */
int64_t dexsim_host_zero_copy_steps(void);

/* HOST function: observation rows 40-44 (the five 0/1 contact floats, envs/manipulation_env.py:262) of envs [0, n) of a
 * host [45, ld] observation buffer from their 1-byte contact masks -- what DEXSIM_HOST_EXPAND_CONTACTS does chunk by chunk
 * during the download, for callers that took DEXSIM_HOST_PACKED_CONTACTS and expand on demand.  AVX2 when available. */
int dexsim_expand_contact_rows(float* h_obs /* host [45, ld] */, const uint8_t* h_contact_mask /* host [ld] */,
                               int64_t n, int64_t ld);

#ifdef __cplusplus
}
#endif
#endif /* DEXSIM_H */
