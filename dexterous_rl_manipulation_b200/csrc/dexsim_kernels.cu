// dexsim_kernels.cu -- sm_100a kernels + C ABI (include/dexsim.h) of the batched simulator.
//
// Kernels
//   step_kernel      one env-step for every env: SoA state in HBM -> registers -> HBM.  Streaming,
//                    HBM-bound (DESIGN.md "Roofline"): every field is read and written at most once,
//                    coalesced 128-byte rows per warp, unchanged fields are not written back.
//   rollout_kernel   k env-steps per env in one launch with the policy drawn in-kernel (Philox),
//                    state in registers for the whole launch, episodes auto-reset, per-group
//                    counters aggregated in shared memory and flushed with one atomic per counter.
//   reset_*_kernel   episode (re)initialisation from pre-drawn or Philox draws.
//   finish_reset_kernel  the second launch of dexsim_step_final and dexsim_step_host_final: episode end + reset of
//                    the envs a step without auto-reset finished, after copying their terminal observation out.
// No CPU fallback exists: every entry point launches CUDA work or returns an error code.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <type_traits>

#include "dexsim_core.cuh"

namespace dexsim {

constexpr int STEP_MIN_BLOCKS = 2;
constexpr int STEP_THREADS = 256;

constexpr int SMEM_GROUPS_MAX = 64;     // group table + block counters are staged in smem up to this many groups

// ---- state <-> registers -----------------------------------------------------------------------
struct Hot {            // what a step needs beyond EnvRegs to decide which rows changed
    double op_old[3];
    float  ov_old[3];
    unsigned cmask_old;
};

__device__ __forceinline__ void load_env(const DexsimState& st, int64_t i, EnvRegs& e) {
    const int64_t ld = st.ld;
    const float* __restrict__ obs = st.obs;
#pragma unroll
    for (int j = 0; j < NJ; ++j) e.jp[j] = obs[(DEXSIM_ROW_JP + j) * ld + i];
#pragma unroll
    for (int j = 0; j < NJ; ++j) e.jv[j] = obs[(DEXSIM_ROW_JV + j) * ld + i];
#pragma unroll
    for (int k = 0; k < 3; ++k) e.ov[k] = obs[(DEXSIM_ROW_OV + k) * ld + i];
#pragma unroll
    for (int k = 0; k < 3; ++k) e.op[k] = st.op64[k * ld + i];
    e.thr = st.thr[i];
    e.damp = st.damp[i];
    e.sc = st.step_count[i];
    e.cmask = st.cmask[i];
}

// Full write-back (reset paths): every row including the constant quaternion.
// `host`: optional mirror of observation rows 30, 31, 37, 38 in mapped host memory (DexsimStepIO.host_static_rows)
__device__ __forceinline__ void mirror_static_rows(float* host, int64_t ld, int64_t i, const EnvRegs& e) {
    host[(DEXSIM_ROW_OP + 0) * ld + i] = (float)e.op[0];
    host[(DEXSIM_ROW_OP + 1) * ld + i] = (float)e.op[1];
    host[(DEXSIM_ROW_OV + 0) * ld + i] = e.ov[0];
    host[(DEXSIM_ROW_OV + 1) * ld + i] = e.ov[1];
}

__device__ __forceinline__ void store_env_full(const DexsimState& st, int64_t i, const EnvRegs& e, float* host = nullptr) {
    const int64_t ld = st.ld;
    float* __restrict__ obs = st.obs;
    if (host) mirror_static_rows(host, ld, i, e);
#pragma unroll
    for (int j = 0; j < NJ; ++j) obs[(DEXSIM_ROW_JP + j) * ld + i] = e.jp[j];
#pragma unroll
    for (int j = 0; j < NJ; ++j) obs[(DEXSIM_ROW_JV + j) * ld + i] = e.jv[j];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        obs[(DEXSIM_ROW_OP + k) * ld + i] = (float)e.op[k];
        obs[(DEXSIM_ROW_OV + k) * ld + i] = e.ov[k];
        st.op64[k * ld + i] = e.op[k];
    }
    obs[(DEXSIM_ROW_QUAT + 0) * ld + i] = 1.0f;          // envs/manipulation_env.py:164
    obs[(DEXSIM_ROW_QUAT + 1) * ld + i] = 0.0f;
    obs[(DEXSIM_ROW_QUAT + 2) * ld + i] = 0.0f;
    obs[(DEXSIM_ROW_QUAT + 3) * ld + i] = 0.0f;
#pragma unroll
    for (int f = 0; f < NF; ++f) obs[(DEXSIM_ROW_CONTACT + f) * ld + i] = ((e.cmask >> f) & 1u) ? 1.0f : 0.0f;
    st.thr[i] = e.thr;
    st.damp[i] = e.damp;
    st.step_count[i] = e.sc;
    st.cmask[i] = (uint8_t)e.cmask;
}

// Step write-back: joints always; object rows, contact rows and the mask only when they changed
// (x, y never move after the first step; z rests at 0 for most of a long episode; contact flags
// flip rarely).  The sector was read by this thread just before, so partial writes merge in L2.
__device__ __forceinline__ void store_env_step(const DexsimState& st, int64_t i, const EnvRegs& e, const Hot& h,
                                               float* host = nullptr) {
    const int64_t ld = st.ld;
    float* __restrict__ obs = st.obs;
#pragma unroll
    for (int j = 0; j < NJ; ++j) obs[(DEXSIM_ROW_JP + j) * ld + i] = e.jp[j];
#pragma unroll
    for (int j = 0; j < NJ; ++j) obs[(DEXSIM_ROW_JV + j) * ld + i] = e.jv[j];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (__double_as_longlong(e.op[k]) != __double_as_longlong(h.op_old[k])) {
            st.op64[k * ld + i] = e.op[k];
            obs[(DEXSIM_ROW_OP + k) * ld + i] = (float)e.op[k];
            if (host && k < 2) host[(DEXSIM_ROW_OP + k) * ld + i] = (float)e.op[k];
        }
        if (__float_as_uint(e.ov[k]) != __float_as_uint(h.ov_old[k])) {
            obs[(DEXSIM_ROW_OV + k) * ld + i] = e.ov[k];
            if (host && k < 2) host[(DEXSIM_ROW_OV + k) * ld + i] = e.ov[k];
        }
    }
    const unsigned flip = e.cmask ^ h.cmask_old;
    if (flip) {
#pragma unroll
        for (int f = 0; f < NF; ++f)
            if ((flip >> f) & 1u) obs[(DEXSIM_ROW_CONTACT + f) * ld + i] = ((e.cmask >> f) & 1u) ? 1.0f : 0.0f;
        st.cmask[i] = (uint8_t)e.cmask;
    }
    st.step_count[i] = e.sc;
}

__device__ __forceinline__ int group_index(const uint16_t* group_of_env, int64_t i, int64_t gid, int num_groups) {
    return group_of_env ? (int)group_of_env[i] : (int)((uint32_t)gid % (uint32_t)num_groups);
}

// One finished episode -> per-group counters (rows of DEXSIM_NCOUNTERS int64) + return sums.
__device__ __forceinline__ void record_episode(unsigned long long* cnt, double* rs, int success, int steps,
                                               int final_c, int la, int lb, int tie, double ret) {
    atomicAdd(&cnt[DEXSIM_CNT_EPISODES], 1ull);
    if (success) atomicAdd(&cnt[DEXSIM_CNT_SUCCESSES], 1ull);
    atomicAdd(&cnt[DEXSIM_CNT_SUM_STEPS], (unsigned long long)steps);
    atomicAdd(&cnt[DEXSIM_CNT_SUM_STEPS_SQ], (unsigned long long)steps * (unsigned long long)steps);
    if (final_c) atomicAdd(&cnt[DEXSIM_CNT_SUM_FINAL_CONTACTS], (unsigned long long)final_c);
    if (la != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_METRICS + la], 1ull);
    if (lb != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_TAXONOMY + lb], 1ull);
    if (tie == 1) atomicAdd(&cnt[DEXSIM_CNT_VAR_TIES], 1ull);       // 2 = decided by np.var on the history: not in doubt
    if (rs) { atomicAdd(&rs[0], ret); atomicAdd(&rs[1], __dmul_rn(ret, ret)); }
}

// Optional per-episode log of a launch (rollout kernel).
struct EpisodeLog {
    DexsimEpisodeRecord* rec = nullptr;
    unsigned long long* count = nullptr;
    long long capacity = 0;
    uint32_t t_end = 0;
};

// Episode end shared by the step kernel's auto-reset and the rollout kernel
// (loop shape of evaluation/evaluator.py:135-173 / training/episode_utils.py:42-55).
__device__ __forceinline__ void finish_episode(const EnvRegs& e, const DexsimParams& p, uint32_t gid, uint32_t episode,
                                               double ep_return, const EpStats& es, bool terminated, int n_c,
                                               unsigned long long* cnt, double* rs, const EpisodeLog* log,
                                               const bool classify = true) {
    if (!(cnt || (log && log->rec))) return;
    if (!classify) {            // counts-only tracking: no history summary, no return -> no labels, no return sums
        if (cnt) record_episode(cnt, nullptr, p.success_is_terminated ? (terminated ? 1 : 0) : 0, e.sc, n_c,
                                DEXSIM_LABEL_NONE, DEXSIM_LABEL_NONE, 0, 0.0);
        return;
    }
    DexsimEpisodeSummary s;
    s.success = p.success_is_terminated ? (terminated ? 1 : 0) : 0;
    s.episode_steps = e.sc; s.num_contacts = n_c; s.final_contacts = n_c; s.hist_len = e.sc;
    int sum, sq, f5, l5, mx;
    epstats_unpack(es, sum, sq, f5, l5, mx);
    s.max_count = mx; s.sum_counts = sum; s.sum_sq_counts = sq; s.first5_sum = f5; s.last5_sum = l5;
    int la, lb, tie;
    // an exact variance tie is only flagged here (tie == 1); when the launch records the history, resolve_ties_kernel
    // decides it afterwards with np.var's own arithmetic -- kept out of this kernel's registers and stack
    classify_summary(s, p.loop_max_steps > 0 ? p.loop_max_steps : p.max_episode_steps, p.success_threshold, la, lb, tie);
    if (cnt) record_episode(cnt, rs, s.success, e.sc, n_c, la, lb, tie, ep_return);
    if (log && log->rec) {
        const unsigned long long slot = atomicAdd(log->count, 1ull);
        if ((long long)slot < log->capacity) {
            DexsimEpisodeRecord r;
            r.env_gid = gid; r.episode = episode; r.steps = e.sc;
            r.success = (uint8_t)s.success; r.final_contacts = (uint8_t)n_c;
            r.label_metrics = (uint8_t)la; r.label_taxonomy = (uint8_t)lb;
            r.episode_reward = ep_return; r.t_end = log->t_end; r.var_tie = (uint32_t)tie;
            log->rec[slot] = r;
        }
    }
}

__device__ __forceinline__ void finish_and_reset(EnvRegs& e, const DexsimParams& p, const DexsimGroup& grp,
                                                 uint32_t gid, uint32_t& episode, double& ep_return, EpStats& es,
                                                 bool terminated, int n_c, unsigned long long* cnt, double* rs,
                                                 double& size, double& mass, double& friction,
                                                 const EpisodeLog* log = nullptr, const bool classify = true) {
    finish_episode(e, p, gid, episode, ep_return, es, terminated, n_c, cnt, rs, log, classify);
    episode += 1u;
    float jp0[NJ], pos[3];
    reset_draws(p.seed, gid, episode, grp, jp0, size, mass, friction, pos);
    env_reset(e, jp0, size, friction, pos, /*keep_pos=*/!p.respawn);
    ep_return = 0.0;
    es.w0 = 0u; es.w1 = 0u;
}

// ---- next-step auto-reset (dexsim_step_next_reset) -------------------------------------------------------------------
// An env has a pending reset when its stored state is what a step that ended its episode left behind: the step kernels'
// `done` evaluated on that state (terminated: the contact count of the stored mask; truncated: the step before the last
// one was at max_episode_steps; the loop bound).  Every reset leaves sc == 0, so a freshly reset env is never pending.
// Derived from the state alone, it survives state_dict() / load_state_dict() and needs no array of its own.
__device__ __forceinline__ bool pending_reset(const EnvRegs& e, const DexsimParams& p) {
    return e.sc > 0 && (__popc(e.cmask) >= p.success_threshold || e.sc > p.max_episode_steps ||
                        (p.loop_max_steps > 0 && e.sc >= p.loop_max_steps));
}

// The reset of a pending env, in place of its step: what finish_and_reset does after the episode end (counted by the step
// that ended it), and the outputs of a reset step -- reward 0, both flags 0, the contact count of the reset state.
__device__ __forceinline__ void next_step_reset(EnvRegs& e, const DexsimParams& p, const DexsimGroup& grp, uint32_t gid,
                                                uint32_t& episode, const DexsimState& st, int64_t i, StepResult& r) {
    double ep_return = 0.0, size, mass, friction;
    EpStats es{0u, 0u};
    finish_and_reset(e, p, grp, gid, episode, ep_return, es, false, 0, nullptr, nullptr, size, mass, friction);
    st.episode[i] = episode;
    st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
    r.total = r.distance = r.contact = r.closure = r.stability = 0.0;
    r.n_c = __popc(e.cmask);
    r.terminated = r.truncated = false;
}

// Observation entry `row` (envs/manipulation_env.py:254-264) of an env held in registers; `row` is a compile-time
// constant wherever this is called from an unrolled loop.
__device__ __forceinline__ float obs_entry(const EnvRegs& e, const int row) {
    if (row < DEXSIM_ROW_JV) return e.jp[row - DEXSIM_ROW_JP];
    if (row < DEXSIM_ROW_OP) return e.jv[row - DEXSIM_ROW_JV];
    if (row < DEXSIM_ROW_QUAT) return (float)e.op[row - DEXSIM_ROW_OP];
    if (row < DEXSIM_ROW_OV) return row == DEXSIM_ROW_QUAT ? 1.0f : 0.0f;
    if (row < DEXSIM_ROW_CONTACT) return e.ov[row - DEXSIM_ROW_OV];
    return ((e.cmask >> (row - DEXSIM_ROW_CONTACT)) & 1u) ? 1.0f : 0.0f;
}

}  // namespace dexsim

#include "dexsim_step_tma.cuh"
#include "dexsim_rollout_split.cuh"

namespace dexsim {

// ---- single-env read-back ------------------------------------------------------------------------------
// TAGGED: slot 63 = tag, written after every other slot is visible system-wide (host polling on mapped memory).
// Runs in the first 64 threads of a CTA.
template <bool TAGGED>
__device__ __forceinline__ void pack_env_body(const DexsimState& st, const DexsimStepIO& io, const int64_t i, const int after_reset,
                                              double* __restrict__ out) {
    const int t = threadIdx.x;
    const int64_t ld = st.ld;
    const bool noisy = io.noisy_obs && (io.obs_noise || io.sigma_obs != 0.0f);
    const float* obs = noisy ? io.noisy_obs : st.obs;
    if (t < NOBS) out[t] = (double)obs[t * ld + i];
    if (t == 45) out[45] = after_reset ? 0.0 : (io.reward64 ? io.reward64[i] : (double)io.reward[i]);
    if (t == 46) out[46] = after_reset ? 0.0 : (double)io.terminated[i];
    if (t == 47) out[47] = after_reset ? 0.0 : (double)io.truncated[i];
    if (t == 48) out[48] = (double)__popc((unsigned)st.cmask[i]);
    if (t == 49) out[49] = (double)st.step_count[i];
    if (t >= 50 && t < 53) out[t] = st.op64[(t - 50) * ld + i];
    if (t == 53) out[53] = st.size[i];
    if (t == 54) out[54] = st.mass[i];
    if (t == 55) out[55] = st.friction[i];
    if (t >= 56 && t < 60) out[t] = (io.reward_comps && !after_reset) ? (double)io.reward_comps[(t - 56) * ld + i] : 0.0;
    if (t == 60) out[60] = (io.finished && !after_reset) ? (double)io.finished[i] : 0.0;
    if (t > 60 && t < 63) out[t] = 0.0;
    if (!TAGGED) {
        if (t == 63) out[63] = 0.0;
    } else {
        __threadfence_system();         // the caller writes the tag after a block-wide barrier (pack_env_publish)
    }
}
// Every thread of the block must call this (it contains the barrier).
__device__ __forceinline__ void pack_env_publish(double* __restrict__ out, const double tag) {
    __syncthreads();
    if (threadIdx.x == 0) *reinterpret_cast<volatile double*>(out + 63) = tag;
}

template <bool TAGGED>
__global__ void pack_env_kernel(const DexsimState st, const DexsimStepIO io, const int64_t i, const int after_reset,
                                double* __restrict__ out, const double tag) {
    pack_env_body<TAGGED>(st, io, i, after_reset, out);
    if (TAGGED) pack_env_publish(out, tag);
}

// ---- step kernel -----------------------------------------------------------------------------------
// DENSE: reward type.  AOS: action is [n, 15] (reference layout) and is transposed through shared
// memory with coalesced float4 reads (15 is odd, so the per-thread reads are bank-conflict free).
// EXTRAS: noise, reward components, episode tracking, auto-reset -- the plain path carries none
// of their registers or branches.
// NEXT: next-step auto-reset (dexsim_step_next_reset, see pending_reset); only with EXTRAS.
template <bool DENSE, bool AOS, bool EXTRAS, bool NEXT>
__global__ void __launch_bounds__(STEP_THREADS, STEP_MIN_BLOCKS)
step_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
            const uint16_t* __restrict__ group_of_env, const DexsimStepIO io,
            double* __restrict__ pack_out = nullptr, const double pack_tag = 0.0) {
    static_assert(!NEXT || EXTRAS, "next-step auto-reset needs the auto-reset path");
    __shared__ __align__(16) float sh_act[AOS ? STEP_THREADS * NJ : 4];
    // Finished episodes are counted per CTA in shared memory and flushed with one global atomic per
    // non-zero counter at the end: thousands of episodes end per step and would otherwise serialise
    // on the same 18 L2 addresses.
    __shared__ unsigned long long sh_cnt[EXTRAS ? SMEM_GROUPS_MAX * DEXSIM_NCOUNTERS : 1];
    __shared__ double sh_rs[EXTRAS ? SMEM_GROUPS_MAX * 2 : 1];
    const bool count_episodes = EXTRAS && p.auto_reset && io.counters != nullptr;     // with or without per-env tracking arrays
    const bool staged = count_episodes && p.num_groups <= SMEM_GROUPS_MAX;
    if (EXTRAS && staged) {
        for (int w = threadIdx.x; w < p.num_groups * DEXSIM_NCOUNTERS; w += STEP_THREADS) sh_cnt[w] = 0ull;
        for (int w = threadIdx.x; w < p.num_groups * 2; w += STEP_THREADS) sh_rs[w] = 0.0;
        __syncthreads();
    }
    const int64_t n = st.n, ld = st.ld;
    for (int64_t base = (int64_t)blockIdx.x * STEP_THREADS; base < n; base += (int64_t)gridDim.x * STEP_THREADS) {
        const int64_t i = base + threadIdx.x;
        const bool active = i < n;
        float a[NJ];
        if (AOS) {
            // tile = envs [base, base + 256) -> 3840 contiguous floats starting 16-byte aligned
            const int64_t tile_floats = (((n - base) < STEP_THREADS) ? (n - base) : STEP_THREADS) * NJ;
            const float* __restrict__ src = io.action + base * NJ;
            __syncthreads();                         // previous tile fully consumed
            // float4 reads need a 16-byte aligned base (a tile starts 256 * 60 bytes further, still aligned); any
            // other base (e.g. an [n,15] slice starting at an odd env) takes the scalar loop below for the whole tile
            const int64_t nvec = (reinterpret_cast<uintptr_t>(io.action) & 15u) ? 0 : (tile_floats >> 2);
            for (int64_t v = threadIdx.x; v < nvec; v += STEP_THREADS)
                reinterpret_cast<float4*>(sh_act)[v] = __ldg(reinterpret_cast<const float4*>(src) + v);
            for (int64_t r = (nvec << 2) + threadIdx.x; r < tile_floats; r += STEP_THREADS) sh_act[r] = __ldg(src + r);
            __syncthreads();
            if (active) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = sh_act[threadIdx.x * NJ + j];
            }
        } else if (active) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) a[j] = __ldg(io.action + j * ld + i);
        }
        if (!active) continue;

        EnvRegs e;
        load_env(st, i, e);
        Hot h;
#pragma unroll
        for (int k = 0; k < 3; ++k) { h.op_old[k] = e.op[k]; h.ov_old[k] = e.ov[k]; }
        h.cmask_old = e.cmask;
        bool pending = false;
        if constexpr (NEXT) pending = pending_reset(e, p);

        // in-kernel Philox noise (DexsimStepIO.sigma_*): needs the env's identity before the step
        const bool fused_dyn = EXTRAS && !io.dyn_noise && io.sigma_dyn != 0.0f;
        const bool fused_obs = EXTRAS && !io.obs_noise && io.noisy_obs && io.sigma_obs != 0.0f;
        const int64_t gid = p.env_gid0 + i;
        uint32_t episode = 0u;
        int g = 0;
        if (EXTRAS && (fused_dyn || fused_obs)) {
            episode = st.episode[i];
            if (io.sigma_dyn < 0.0f || io.sigma_obs < 0.0f) g = group_index(group_of_env, i, gid, p.num_groups);
        }
        if (EXTRAS && io.dyn_noise) {                // evaluation/robustness_tests.py:180-187
#pragma unroll
            for (int j = 0; j < NJ; ++j)
                a[j] = clip_f32(__fadd_rn(a[j], __ldg(io.dyn_noise + j * ld + i)), -1.0f, 1.0f);
        } else if (fused_dyn && !pending) {
            const float sigma = io.sigma_dyn > 0.0f ? io.sigma_dyn : groups[g].sigma_dyn;
            if (sigma > 0.0f) {
                float nz[NJ];
                normal_rows<NJ>(p.seed, (uint32_t)gid, episode, (uint32_t)e.sc, STREAM_DYN, sigma, nz);
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(__fadd_rn(a[j], nz[j]), -1.0f, 1.0f);
            }
        }

        StepResult r;
        if constexpr (NEXT) {
            if (pending) {          // the reset the previous step left for this env, instead of a step: the action is ignored
                g = group_index(group_of_env, i, gid, p.num_groups);
                episode = st.episode[i];
                next_step_reset(e, p, groups[g], (uint32_t)gid, episode, st, i, r);
            } else {
                env_step<DENSE>(e, a, p, r);
            }
        } else {
            env_step<DENSE>(e, a, p, r);
        }

        io.reward[i] = (float)r.total;
        io.terminated[i] = r.terminated ? 1 : 0;
        io.truncated[i] = r.truncated ? 1 : 0;
        io.num_contacts[i] = (uint8_t)r.n_c;

        if (!EXTRAS) {
            store_env_step(st, i, e, h);
            continue;
        }

        if (io.reward64) io.reward64[i] = r.total;
        if (io.reward_comps) {
            io.reward_comps[0 * ld + i] = (float)r.distance;
            io.reward_comps[1 * ld + i] = (float)r.contact;
            io.reward_comps[2 * ld + i] = (float)r.closure;
            io.reward_comps[3 * ld + i] = (float)r.stability;
        }
        const bool tracking = st.ep_return != nullptr && st.ep_stats != nullptr;
        double ep_return = 0.0;
        EpStats es{0u, 0u};
        if (tracking && !pending) {                                    // a pending env's episode starts now: both stay 0
            ep_return = __dadd_rn(st.ep_return[i], r.total);           // evaluator.py:144
            es.w0 = st.ep_stats[i]; es.w1 = st.ep_stats[ld + i];
            epstats_push(es, e.sc - 1, r.n_c);                         // evaluator.py:148-150
        }
        // (never true for a pending env: its reset left step count 0 and both flags 0)
        const bool done = r.terminated || r.truncated || (p.loop_max_steps > 0 && e.sc >= p.loop_max_steps);
        bool finished = false;
        if (p.auto_reset && done) {
            finished = true;
            g = group_index(group_of_env, i, gid, p.num_groups);
            episode = st.episode[i];
            double size, mass, friction;
            unsigned long long* cnt = nullptr;
            double* rs = nullptr;
            if (count_episodes) {
                cnt = (staged ? sh_cnt : reinterpret_cast<unsigned long long*>(io.counters)) + (int64_t)g * DEXSIM_NCOUNTERS;
                if (io.ret_sums) rs = (staged ? sh_rs : io.ret_sums) + 2 * g;
            }
            if constexpr (NEXT) {   // counted and flagged now, reset by the env's next step
                finish_episode(e, p, (uint32_t)gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs, nullptr,
                               /*classify=*/tracking);
                store_env_step(st, i, e, h, io.host_static_rows);
            } else {
                finish_and_reset(e, p, groups[g], (uint32_t)gid, episode, ep_return, es, r.terminated, r.n_c,
                                 cnt, rs, size, mass, friction, nullptr, /*classify=*/tracking);
                st.episode[i] = episode;
                st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
                store_env_full(st, i, e, io.host_static_rows);
            }
        } else if (pending) {
            store_env_full(st, i, e, io.host_static_rows);
        } else {
            store_env_step(st, i, e, h, io.host_static_rows);
        }
        if (tracking) {
            st.ep_return[i] = ep_return;
            st.ep_stats[i] = es.w0; st.ep_stats[ld + i] = es.w1;
        }
        if (io.finished) io.finished[i] = finished ? 1 : 0;
        if (io.noisy_obs && io.obs_noise) {          // evaluation/robustness_tests.py:204-205, all 45 entries
            const float* __restrict__ nz = io.obs_noise;
            float* __restrict__ out = io.noisy_obs;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                out[(DEXSIM_ROW_JP + j) * ld + i] = __fadd_rn(e.jp[j], __ldg(nz + (DEXSIM_ROW_JP + j) * ld + i));
                out[(DEXSIM_ROW_JV + j) * ld + i] = __fadd_rn(e.jv[j], __ldg(nz + (DEXSIM_ROW_JV + j) * ld + i));
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                out[(DEXSIM_ROW_OP + k) * ld + i] = __fadd_rn((float)e.op[k], __ldg(nz + (DEXSIM_ROW_OP + k) * ld + i));
                out[(DEXSIM_ROW_OV + k) * ld + i] = __fadd_rn(e.ov[k], __ldg(nz + (DEXSIM_ROW_OV + k) * ld + i));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)
                out[(DEXSIM_ROW_QUAT + k) * ld + i] = __fadd_rn(k == 0 ? 1.0f : 0.0f, __ldg(nz + (DEXSIM_ROW_QUAT + k) * ld + i));
#pragma unroll
            for (int f = 0; f < NF; ++f)
                out[(DEXSIM_ROW_CONTACT + f) * ld + i] =
                    __fadd_rn(((e.cmask >> f) & 1u) ? 1.0f : 0.0f, __ldg(nz + (DEXSIM_ROW_CONTACT + f) * ld + i));
        } else if (fused_obs) {
            // the same 45 normals dexsim_fill_normal(STREAM_OBS) would produce for the env's state AFTER this step
            // (and after an auto-reset): one Philox block = four observation rows, written as they are drawn
            const float sigma = io.sigma_obs > 0.0f ? io.sigma_obs : groups[g].sigma_obs;
            float* __restrict__ out = io.noisy_obs;
#pragma unroll
            for (int b = 0; b < (NOBS + 3) / 4; ++b) {
                const U4 o = rng_block(p.seed, (uint32_t)gid, episode, (uint32_t)e.sc, STREAM_OBS, (uint32_t)b);
                float z[4];
                normal_pair(o.x, o.y, z[0], z[1]);
                normal_pair(o.z, o.w, z[2], z[3]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int row = 4 * b + k;
                    if (row < NOBS) out[row * ld + i] = __fadd_rn(obs_entry(e, row), __fmul_rn(sigma, z[k]));
                }
            }
        }
    }
    if (EXTRAS && staged) {
        __syncthreads();
        unsigned long long* gc = reinterpret_cast<unsigned long long*>(io.counters);
        for (int w = threadIdx.x; w < p.num_groups * DEXSIM_NCOUNTERS; w += STEP_THREADS)
            if (sh_cnt[w]) atomicAdd(&gc[w], sh_cnt[w]);
        if (io.ret_sums)
            for (int w = threadIdx.x; w < p.num_groups * 2; w += STEP_THREADS)
                if (sh_rs[w] != 0.0) atomicAdd(&io.ret_sums[w], sh_rs[w]);
    }
    // dexsim_step_single (one env, one CTA): pack what step() returns in the same launch; the 64 packing threads
    // read what thread 0 just stored, hence the block-wide barrier
    if (EXTRAS && pack_out) {
        __syncthreads();
        if (threadIdx.x < 64) pack_env_body<true>(st, io, 0, 0, pack_out);
        pack_env_publish(pack_out, pack_tag);
    }
}

// ---- reset kernels --------------------------------------------------------------------------------
__global__ void __launch_bounds__(STEP_THREADS)
reset_predrawn_kernel(const DexsimState st, const uint8_t* __restrict__ mask, const float* __restrict__ jp0,
                      const double* __restrict__ size, const double* __restrict__ mass,
                      const double* __restrict__ friction, const float* __restrict__ pos) {
    const int64_t n = st.n, ld = st.ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[i]) continue;
        EnvRegs e;
        float j0[NJ], ps[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int j = 0; j < NJ; ++j) j0[j] = jp0[j * ld + i];
        if (pos) {
#pragma unroll
            for (int k = 0; k < 3; ++k) ps[k] = pos[k * ld + i];
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) e.op[k] = st.op64[k * ld + i];
        }
        env_reset(e, j0, size[i], friction[i], ps, pos == nullptr);
        store_env_full(st, i, e);
        st.size[i] = size[i]; st.mass[i] = mass[i]; st.friction[i] = friction[i];
        if (st.ep_return) st.ep_return[i] = 0.0;
        if (st.ep_stats) { st.ep_stats[i] = 0u; st.ep_stats[ld + i] = 0u; }
    }
}

__global__ void __launch_bounds__(STEP_THREADS)
reset_philox_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
                    const uint16_t* __restrict__ group_of_env, const uint8_t* __restrict__ mask, int respawn) {
    const int64_t n = st.n, ld = st.ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (mask && !mask[i]) continue;
        const int64_t gid = p.env_gid0 + i;
        const int g = group_index(group_of_env, i, gid, p.num_groups);
        EnvRegs e;
        if (!respawn) {
#pragma unroll
            for (int k = 0; k < 3; ++k) e.op[k] = st.op64[k * ld + i];
        }
        float j0[NJ], ps[3];
        double size, mass, friction;
        reset_draws(p.seed, (uint32_t)gid, st.episode[i], groups[g], j0, size, mass, friction, ps);
        env_reset(e, j0, size, friction, ps, !respawn);
        store_env_full(st, i, e);
        st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
        if (st.ep_return) st.ep_return[i] = 0.0;
        if (st.ep_stats) { st.ep_stats[i] = 0u; st.ep_stats[ld + i] = 0u; }
    }
}

// ---- finish-and-reset pass (dexsim_step_final) ----------------------------------------------------------
// Runs after a step launched with auto_reset = 0 and no finished / counters / ret_sums outputs, and does what the step
// kernels' in-kernel auto-reset does, from the arrays that step left behind: `done` from the flags and the step count,
// `finished`, the episode end (counters staged per CTA as in step_kernel, labels when tracking), the reset through
// load_env -> finish_and_reset -> store_env_full, and the reset observation's noise.  Before the reset, the column the
// step returned (noisy_obs when observation noise is on, obs otherwise) is copied into `final_obs`; columns of envs
// that did not finish are not written.  One thread per env of a grid-stride loop: a warp without a finished lane moves
// on after one ballot.  `pdl`: launched as a programmatic dependent of the step (see step_then_finish_reset).
//
// HOST (dexsim_step_host_final): the outputs of `hf` instead of `final_obs`, all of them device aliases of the caller's
// mapped page-locked buffers, offset to the chunk.
struct FinishHost {
    float* final_obs;       // [n, 45] batch-first: row i <- the returned observation of env i, finished envs only
    float* obs;             // the host observation [45, ld] or NULL: rows 30, 31, 37, 38 of a reset env (the static-row
                            // mirror); with `zero_copy` also every other row the zero-copy step writes (0-32, 37-39)
    uint8_t* cmask;         // zero_copy: the host contact masks (of reset envs)
    uint8_t* terminated;    // zero_copy: the flags of every env, which the step left on the device for this pass
    uint8_t* truncated;
    uint8_t* num_contacts;  // (NULL: the caller has no buffer for them)
    uint8_t* finished;
    int zero_copy;
};
constexpr int FINISH_HOST_SMEM = STEP_THREADS * NOBS * 4;      // one [32 envs, 45] record block per warp

template <bool HOST>
__global__ void __launch_bounds__(STEP_THREADS)
finish_reset_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
                    const uint16_t* __restrict__ group_of_env, const DexsimStepIO io, float* __restrict__ final_obs,
                    const int pdl, const FinishHost hf) {
    __shared__ unsigned long long sh_cnt[SMEM_GROUPS_MAX * DEXSIM_NCOUNTERS];
    __shared__ double sh_rs[SMEM_GROUPS_MAX * 2];
    const bool count_episodes = io.counters != nullptr;
    const bool staged = count_episodes && p.num_groups <= SMEM_GROUPS_MAX;
    if (staged) {
        for (int w = threadIdx.x; w < p.num_groups * DEXSIM_NCOUNTERS; w += STEP_THREADS) sh_cnt[w] = 0ull;
        for (int w = threadIdx.x; w < p.num_groups * 2; w += STEP_THREADS) sh_rs[w] = 0.0;
        __syncthreads();
    }
    // every global access below comes after the step grid has completed and flushed
    if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
    const int64_t n = st.n, ld = st.ld;
    const bool tracking = st.ep_return != nullptr && st.ep_stats != nullptr;
    const bool noisy = io.noisy_obs && (io.obs_noise || io.sigma_obs != 0.0f);
    const bool fused_obs = !io.obs_noise && io.noisy_obs && io.sigma_obs != 0.0f;
    const float* __restrict__ returned = noisy ? io.noisy_obs : st.obs;
    for (int64_t base = (int64_t)blockIdx.x * STEP_THREADS; base < n; base += (int64_t)gridDim.x * STEP_THREADS) {
        const int64_t i = base + threadIdx.x;
        bool done = false;
        if (i < n) {
            const int sc = st.step_count[i];
            done = io.terminated[i] || io.truncated[i] || (p.loop_max_steps > 0 && sc >= p.loop_max_steps);
            io.finished[i] = done ? 1 : 0;
            if (HOST && hf.zero_copy) {              // consecutive lanes, consecutive bytes: one PCIe write per warp and vector
                hf.terminated[i] = io.terminated[i];
                hf.truncated[i] = io.truncated[i];
                if (hf.num_contacts) hf.num_contacts[i] = io.num_contacts[i];
                hf.finished[i] = done ? 1 : 0;
            }
        }
        const unsigned fin = __ballot_sync(0xffffffffu, done);
        if (fin == 0u) continue;
        if (HOST) {
            // Records leave from consecutive lanes: 4-byte writes scattered over host memory would cost a PCIe transaction
            // each.  The finished lanes stage their columns in the warp's block of shared memory; the warp then writes
            // each record as 45 contiguous floats (two stores), or, when every lane finished, 32 x 45 contiguous floats.
            extern __shared__ float sh_rec[];
            const int lane = threadIdx.x & 31;
            float* rec = sh_rec + (threadIdx.x - lane) * NOBS;
            if (done) {
#pragma unroll
                for (int row = 0; row < NOBS; ++row) rec[lane * NOBS + row] = returned[row * ld + i];
            }
            __syncwarp();
            float* dst = hf.final_obs + (i - lane) * NOBS;
            if (fin == 0xffffffffu) {
#pragma unroll
                for (int k = 0; k < NOBS; ++k) dst[k * 32 + lane] = rec[k * 32 + lane];
            } else {
                for (unsigned m = fin; m; m &= m - 1u) {
                    const int j = __ffs(m) - 1;
                    dst[j * NOBS + lane] = rec[j * NOBS + lane];
                    if (lane < NOBS - 32) dst[j * NOBS + 32 + lane] = rec[j * NOBS + 32 + lane];
                }
            }
            __syncwarp();
        }
        if (!done) continue;

        if (!HOST) {
#pragma unroll
            for (int row = 0; row < NOBS; ++row) final_obs[row * ld + i] = returned[row * ld + i];
        }

        EnvRegs e;
        load_env(st, i, e);
        const int64_t gid = p.env_gid0 + i;
        const int g = group_index(group_of_env, i, gid, p.num_groups);
        uint32_t episode = st.episode[i];
        double ep_return = 0.0;
        EpStats es{0u, 0u};
        if (tracking) { ep_return = st.ep_return[i]; es.w0 = st.ep_stats[i]; es.w1 = st.ep_stats[ld + i]; }
        unsigned long long* cnt = nullptr;
        double* rs = nullptr;
        if (count_episodes) {
            cnt = (staged ? sh_cnt : reinterpret_cast<unsigned long long*>(io.counters)) + (int64_t)g * DEXSIM_NCOUNTERS;
            if (io.ret_sums) rs = (staged ? sh_rs : io.ret_sums) + 2 * g;
        }
        double size, mass, friction;
        finish_and_reset(e, p, groups[g], (uint32_t)gid, episode, ep_return, es, io.terminated[i] != 0, (int)io.num_contacts[i],
                         cnt, rs, size, mass, friction, nullptr, /*classify=*/tracking);
        st.episode[i] = episode;
        st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
        store_env_full(st, i, e, HOST ? hf.obs : nullptr);
        if (HOST && hf.zero_copy) {
            // the zero-copy step sent this env's pre-reset rows and mask to the host: overwrite them with the reset state
            float* __restrict__ h = hf.obs;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                h[(DEXSIM_ROW_JP + j) * ld + i] = e.jp[j];
                h[(DEXSIM_ROW_JV + j) * ld + i] = e.jv[j];
            }
            h[(DEXSIM_ROW_OP + 2) * ld + i] = (float)e.op[2];
            h[(DEXSIM_ROW_OV + 2) * ld + i] = e.ov[2];
            hf.cmask[i] = (uint8_t)e.cmask;
        }
        if (tracking) {
            st.ep_return[i] = ep_return;
            st.ep_stats[i] = es.w0; st.ep_stats[ld + i] = es.w1;
        }
        // the observation noise of the reset state, as the in-kernel reset draws it
        float* __restrict__ out = io.noisy_obs;
        if (io.noisy_obs && io.obs_noise) {
#pragma unroll
            for (int row = 0; row < NOBS; ++row) out[row * ld + i] = __fadd_rn(obs_entry(e, row), __ldg(io.obs_noise + row * ld + i));
        } else if (fused_obs) {
            const float sigma = io.sigma_obs > 0.0f ? io.sigma_obs : groups[g].sigma_obs;
#pragma unroll
            for (int b = 0; b < (NOBS + 3) / 4; ++b) {
                const U4 o = rng_block(p.seed, (uint32_t)gid, episode, (uint32_t)e.sc, STREAM_OBS, (uint32_t)b);
                float z[4];
                normal_pair(o.x, o.y, z[0], z[1]);
                normal_pair(o.z, o.w, z[2], z[3]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int row = 4 * b + k;
                    if (row < NOBS) out[row * ld + i] = __fadd_rn(obs_entry(e, row), __fmul_rn(sigma, z[k]));
                }
            }
        }
    }
    if (staged) {
        __syncthreads();
        unsigned long long* gc = reinterpret_cast<unsigned long long*>(io.counters);
        for (int w = threadIdx.x; w < p.num_groups * DEXSIM_NCOUNTERS; w += STEP_THREADS)
            if (sh_cnt[w]) atomicAdd(&gc[w], sh_cnt[w]);
        if (io.ret_sums)
            for (int w = threadIdx.x; w < p.num_groups * 2; w += STEP_THREADS)
                if (sh_rs[w] != 0.0) atomicAdd(&io.ret_sums[w], sh_rs[w]);
    }
}

// ---- fused rollout ------------------------------------------------------------------------------------
// Row t of a recorded rollout (DexsimTrajectory), stored from registers in three parts so that nothing of it stays live
// across the step: the action as the policy produced it, the step's outcome, and the observation once the step and a
// possible reset are done.  Every store of a warp is one 128-byte line of one row.
__device__ __forceinline__ void record_action(const DexsimTrajectory& tr, int64_t ld, int t, int64_t i, const float* a) {
    if (!tr.action) return;
    float* out = tr.action + (int64_t)t * NJ * ld + i;
#pragma unroll
    for (int j = 0; j < NJ; ++j) out[j * ld] = a[j];
}

__device__ __forceinline__ void record_outcome(const DexsimTrajectory& tr, int64_t ld, int t, int64_t i, const StepResult& r,
                                               bool done) {
    const int64_t at = (int64_t)t * ld + i;
    tr.reward[at] = (float)r.total;
    tr.terminated[at] = r.terminated ? 1 : 0;
    tr.truncated[at] = r.truncated ? 1 : 0;
    tr.finished[at] = done ? 1 : 0;
}

__device__ __forceinline__ void record_obs(const DexsimTrajectory& tr, int64_t ld, int t, int64_t i, const EnvRegs& e) {
    float* out = tr.obs + (int64_t)t * DEXSIM_OBS * ld + i;
#pragma unroll
    for (int row = 0; row < DEXSIM_OBS; ++row) out[row * ld] = obs_entry(e, row);
}

// A recording that also keeps the terminal observation of every episode it ends (dexsim_rollout_record_final):
// `final_obs` [capacity, 45, ld] like tr.obs.  A distinct type, so that it instantiates rollout_kernel anew and the
// DexsimTrajectory instantiations keep their code: for them record_final_obs is empty.
struct TrajectoryFinal {
    DexsimTrajectory tr;
    float* final_obs;
};

__device__ __forceinline__ void record_action(const TrajectoryFinal& f, int64_t ld, int t, int64_t i, const float* a) {
    record_action(f.tr, ld, t, i, a);
}

__device__ __forceinline__ void record_outcome(const TrajectoryFinal& f, int64_t ld, int t, int64_t i, const StepResult& r,
                                               bool done) {
    record_outcome(f.tr, ld, t, i, r, done);
}

__device__ __forceinline__ void record_obs(const TrajectoryFinal& f, int64_t ld, int t, int64_t i, const EnvRegs& e) {
    record_obs(f.tr, ld, t, i, e);
}

__device__ __forceinline__ void record_final_obs(const DexsimTrajectory&, int64_t, int, int64_t, const EnvRegs&) {}

// Called where the episode has ended and `e` still holds the state after the step, before any reset: the observation
// dexsim_step_final returns in final_obs.  Only finished lanes store, so a warp's store covers its finished lanes.
__device__ __forceinline__ void record_final_obs(const TrajectoryFinal& f, int64_t ld, int t, int64_t i, const EnvRegs& e) {
    float* out = f.final_obs + (int64_t)t * DEXSIM_OBS * ld + i;
#pragma unroll
    for (int row = 0; row < DEXSIM_OBS; ++row) out[row * ld] = obs_entry(e, row);
}

// ---- MLP policy (dexsim_rollout_mlp, dexsim_mlp_policy_mean) -------------------------------------------------------
// The packed torch-layout parameters are staged once per CTA into shared memory, transposed and zero-padded so that the
// weights of 16 consecutive neurons for one input are four warp-uniform (broadcast) 128-bit loads:
//   W1T [45][h1p]  b1 [h1p]  (W2T [h1][h2p]  b2 [h2p])  W3T [h_last][16]  b3 [16]  std [16]      (hNp = hN rounded up to 16)
// A thread keeps 16 accumulators and walks the inputs in ascending order, so every neuron's FMA chain is the one
// include/dexsim.h specifies.  The first layer reads its inputs from registers (the env state, plus regenerated noise);
// the last hidden layer feeds each finished block of 16 straight into the 15 output accumulators.  Only a second hidden
// layer needs per-thread scratch for the first layer's outputs: h1 floats per thread, in shared memory, thread-major.
constexpr int MLP_BLOCK = 16;
constexpr int DEXSIM_POLICY_MLP_KIND = 4;        // policy_kind the MLP instantiations receive (dexsim_rollout rejects it)

struct MlpArgs {             // validated DexsimMlpPolicy + the shared-memory layout (offsets in floats)
    const float* params;
    const float* action_std;
    int32_t nh, h1, h2, act;
    int32_t h1p, h2p, o_b1, o_w2, o_b2, o_w3, o_b3, o_std, words;
    int32_t scratch_off;     // float offset of the per-thread scratch (second hidden layer only)
};

__device__ __forceinline__ float mlp_act(float y, int act) {
    if (act == DEXSIM_ACT_TANH) return tanhf(y);
    return (y > 0.0f || y != y) ? y : 0.0f;
}

// Cooperative copy of the packed parameters into the padded transposed layout; every thread of the CTA calls it.
__device__ __forceinline__ void mlp_stage(const MlpArgs& m, float* sw) {
    const int hl = m.nh == 2 ? m.h2 : m.h1;
    // packed offsets (torch layout)
    const int p_b1 = m.h1 * NOBS, p_w2 = p_b1 + m.h1;
    const int p_b2 = p_w2 + (m.nh == 2 ? m.h2 * m.h1 : 0), p_w3 = p_b2 + (m.nh == 2 ? m.h2 : 0);
    const int p_b3 = p_w3 + NJ * hl;
    for (int w = threadIdx.x; w < m.words; w += blockDim.x) {
        float v = 0.0f;
        if (w < m.o_b1) {                                  // W1T[i][j] = W1[j][i]
            const int i = w / m.h1p, j = w % m.h1p;
            if (j < m.h1) v = m.params[j * NOBS + i];
        } else if (w < m.o_w2) {
            const int j = w - m.o_b1;
            if (j < m.h1) v = m.params[p_b1 + j];
        } else if (w < m.o_b2) {                           // W2T[i][j] = W2[j][i]
            const int i = (w - m.o_w2) / m.h2p, j = (w - m.o_w2) % m.h2p;
            if (j < m.h2) v = m.params[p_w2 + j * m.h1 + i];
        } else if (w < m.o_w3) {
            const int j = w - m.o_b2;
            if (j < m.h2) v = m.params[p_b2 + j];
        } else if (w < m.o_b3) {                           // W3T[i][j] = W3[j][i]
            const int i = (w - m.o_w3) / MLP_BLOCK, j = (w - m.o_w3) % MLP_BLOCK;
            if (j < NJ) v = m.params[p_w3 + j * hl + i];
        } else if (w < m.o_std) {
            const int j = w - m.o_b3;
            if (j < NJ) v = m.params[p_b3 + j];
        } else {
            const int j = w - m.o_std;
            if (j < NJ && m.action_std) v = m.action_std[j];
        }
        sw[w] = v;
    }
}

// acc[k] = fmaf(w[k], x, acc[k]) for the 16 weights at `w` (16-byte aligned shared memory, the same for the whole warp)
__device__ __forceinline__ void mlp_fma16(const float* w, const float x, float* acc) {
#pragma unroll
    for (int q = 0; q < MLP_BLOCK / 4; ++q) {
        const float4 v = reinterpret_cast<const float4*>(w)[q];
        acc[4 * q + 0] = __fmaf_rn(v.x, x, acc[4 * q + 0]);
        acc[4 * q + 1] = __fmaf_rn(v.y, x, acc[4 * q + 1]);
        acc[4 * q + 2] = __fmaf_rn(v.z, x, acc[4 * q + 2]);
        acc[4 * q + 3] = __fmaf_rn(v.w, x, acc[4 * q + 3]);
    }
}

// A finished block of the last hidden layer, acc[k] = pre-activation of neuron jb + k, into the output accumulators.
__device__ __forceinline__ void mlp_block_out(const MlpArgs& m, const float* sw, const float* b, int jb, int h, float* acc,
                                              float* o) {
#pragma unroll
    for (int k = 0; k < MLP_BLOCK; ++k) {
        if (jb + k < h) mlp_fma16(sw + m.o_w3 + (jb + k) * MLP_BLOCK, mlp_act(__fadd_rn(acc[k], b[jb + k]), m.act), o);
    }
}

// The network's mean for one env.  `X` provides the 45 inputs in chunks of four: X::chunk(b, x) fills x[0..3] with
// inputs 4b .. 4b+3 (b = 0..11; the last chunk has one).  `scr`: this thread's scratch, stride `ss` floats.
template <typename X>
__device__ __forceinline__ void mlp_mean(const MlpArgs& m, const float* sw, float* scr, int ss, const X& xin, float* mean) {
    float o[MLP_BLOCK];
#pragma unroll
    for (int j = 0; j < MLP_BLOCK; ++j) o[j] = 0.0f;
    for (int jb = 0; jb < m.h1p; jb += MLP_BLOCK) {
        float acc[MLP_BLOCK];
#pragma unroll
        for (int k = 0; k < MLP_BLOCK; ++k) acc[k] = 0.0f;
#pragma unroll
        for (int b = 0; b < (NOBS + 3) / 4; ++b) {
            float x[4];
            xin.chunk(b, x);
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * b + k < NOBS) mlp_fma16(sw + (4 * b + k) * m.h1p + jb, x[k], acc);
        }
        if (m.nh == 1) {
            mlp_block_out(m, sw, sw + m.o_b1, jb, m.h1, acc, o);
        } else {
#pragma unroll
            for (int k = 0; k < MLP_BLOCK; ++k)
                if (jb + k < m.h1) scr[(jb + k) * ss] = mlp_act(__fadd_rn(acc[k], sw[m.o_b1 + jb + k]), m.act);
        }
    }
    if (m.nh == 2) {
        for (int jb = 0; jb < m.h2p; jb += MLP_BLOCK) {
            float acc[MLP_BLOCK];
#pragma unroll
            for (int k = 0; k < MLP_BLOCK; ++k) acc[k] = 0.0f;
#pragma unroll 4
            for (int i = 0; i < m.h1; ++i) mlp_fma16(sw + m.o_w2 + i * m.h2p + jb, scr[i * ss], acc);
            mlp_block_out(m, sw, sw + m.o_b2, jb, m.h2, acc, o);
        }
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) mean[j] = __fadd_rn(o[j], sw[m.o_b3 + j]);
}

// Inputs of the rollout: the observation of the env's registers, plus the stream-3 noise of its current state where
// sigma > 0 -- what the step kernel writes to noisy_obs (one Philox block = four observation rows).
struct MlpEnvInput {
    const EnvRegs& e;
    uint64_t seed;
    uint32_t gid, episode;
    float sigma;
    __device__ __forceinline__ void chunk(const int b, float* x) const {
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = 4 * b + k < NOBS ? obs_entry(e, 4 * b + k) : 0.0f;
        if (sigma > 0.0f) {
            const U4 o = rng_block(seed, gid, episode, (uint32_t)e.sc, STREAM_OBS, (uint32_t)b);
            float z[4];
            normal_pair(o.x, o.y, z[0], z[1]);
            normal_pair(o.z, o.w, z[2], z[3]);
#pragma unroll
            for (int k = 0; k < 4; ++k) x[k] = __fadd_rn(x[k], __fmul_rn(sigma, z[k]));
        }
    }
};

// Inputs of dexsim_mlp_policy_mean: column i of an [45, ld] array
struct MlpColumnInput {
    const float* obs;
    int64_t ld, i;
    __device__ __forceinline__ void chunk(const int b, float* x) const {
#pragma unroll
        for (int k = 0; k < 4; ++k) x[k] = 4 * b + k < NOBS ? obs[(4 * b + k) * ld + i] : 0.0f;
    }
};

__global__ void __launch_bounds__(256)
mlp_mean_kernel(const MlpArgs m, const float* __restrict__ obs, const int64_t n, const int64_t ld, float* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float* sw = reinterpret_cast<float*>(smem_raw);
    mlp_stage(m, sw);
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float mean[NJ];
    mlp_mean(m, sw, sw + m.scratch_off + threadIdx.x, (int)blockDim.x, MlpColumnInput{obs, ld, i}, mean);
#pragma unroll
    for (int j = 0; j < NJ; ++j) out[j * ld + i] = mean[j];
}

// The rollout kernel receives the policy as the first element of its trailing pack: (MlpArgs) or (MlpArgs, trajectory).
// The record_* calls forward past it.
template <typename Tr> __device__ __forceinline__ void record_action(const MlpArgs&, const Tr& tr, int64_t ld, int t, int64_t i,
                                                                     const float* a) { record_action(tr, ld, t, i, a); }
template <typename Tr> __device__ __forceinline__ void record_outcome(const MlpArgs&, const Tr& tr, int64_t ld, int t, int64_t i,
                                                                      const StepResult& r, bool done) {
    record_outcome(tr, ld, t, i, r, done);
}
template <typename Tr> __device__ __forceinline__ void record_obs(const MlpArgs&, const Tr& tr, int64_t ld, int t, int64_t i,
                                                                  const EnvRegs& e) { record_obs(tr, ld, t, i, e); }
template <typename Tr> __device__ __forceinline__ void record_final_obs(const MlpArgs&, const Tr& tr, int64_t ld, int t,
                                                                        int64_t i, const EnvRegs& e) {
    record_final_obs(tr, ld, t, i, e);
}

template <typename... T> struct first_is_mlp : std::false_type {};
template <typename... T> struct first_is_mlp<MlpArgs, T...> : std::true_type {};
template <typename... T> __device__ __forceinline__ const MlpArgs& mlp_of(const MlpArgs& m, const T&...) { return m; }

constexpr int ROLLOUT_MIN_BLOCKS = 2;
constexpr int ROLLOUT_THREADS = 256;      // CTA shape of the fused rollout for large batches (x MIN_BLOCKS resident CTAs per SM)
// REC: record every step into the trajectory (dexsim_rollout_record), passed as the one element of `traj`: a
// DexsimTrajectory, or a TrajectoryFinal that also records terminal observations (dexsim_rollout_record_final).  The REC =
// false instantiations take no trajectory at all, so their parameter list -- and their code -- is what it was before
// recording existed.  The MLP policy (dexsim_rollout_mlp) comes first in the pack when present: (MlpArgs[, trajectory]).
template <bool DENSE, bool LEARNER, bool REC, typename... Traj>
__global__ void __launch_bounds__(ROLLOUT_THREADS, ROLLOUT_MIN_BLOCKS)
rollout_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
               const uint16_t* __restrict__ group_of_env, const int k_steps, const int policy_kind,
               const DexsimRolloutIO rio, const Traj... traj) {
    constexpr bool MLP = first_is_mlp<Traj...>::value;
    static_assert(sizeof...(Traj) == (REC ? 1 : 0) + (MLP ? 1 : 0), "a recording rollout takes one trajectory");
    static_assert(!(MLP && LEARNER), "the MLP and the learner never share a launch");
    const float* __restrict__ actions = rio.actions;
    const float* __restrict__ dyn_noise = rio.dyn_noise;
    int64_t* __restrict__ counters = rio.counters;
    double* __restrict__ ret_sums = rio.ret_sums;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int G = p.num_groups;
    const bool staged = G <= SMEM_GROUPS_MAX;
    DexsimGroup* sh_groups = reinterpret_cast<DexsimGroup*>(smem_raw);
    unsigned long long* sh_cnt = reinterpret_cast<unsigned long long*>(sh_groups + (staged ? G : 0));
    double* sh_rs = reinterpret_cast<double*>(sh_cnt + (staged ? G * DEXSIM_NCOUNTERS : 0));
    if (staged) {
        // per-env object / curriculum parameters are read from shared memory at every reset
        const int words = G * (int)(sizeof(DexsimGroup) / 4);
        for (int w = threadIdx.x; w < words; w += blockDim.x)
            reinterpret_cast<uint32_t*>(sh_groups)[w] = reinterpret_cast<const uint32_t*>(groups)[w];
        for (int w = threadIdx.x; w < G * DEXSIM_NCOUNTERS; w += blockDim.x) sh_cnt[w] = 0ull;
        for (int w = threadIdx.x; w < G * 2; w += blockDim.x) sh_rs[w] = 0.0;
        __syncthreads();
    }
    float* sh_mlp = nullptr;                      // the MLP's weights, after the group table (16-byte aligned)
    if constexpr (MLP) {
        const size_t groups_bytes = staged ? (size_t)G * (sizeof(DexsimGroup) + DEXSIM_NCOUNTERS * 8 + 16) : 0;
        sh_mlp = reinterpret_cast<float*>(smem_raw + ((groups_bytes + 15) & ~(size_t)15));
        mlp_stage(mlp_of(traj...), sh_mlp);
        __syncthreads();
    }
    const DexsimGroup* gtab = staged ? sh_groups : groups;
    unsigned long long* cnt_base = staged ? sh_cnt : reinterpret_cast<unsigned long long*>(counters);
    double* rs_base = staged ? sh_rs : ret_sums;

    const int64_t n = st.n, ld = st.ld;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const int64_t gid64 = p.env_gid0 + i;
        const uint32_t gid = (uint32_t)gid64;
        const int g = group_index(group_of_env, i, gid64, G);
        const DexsimGroup& grp = gtab[g];
        unsigned long long* cnt = counters ? cnt_base + (int64_t)g * DEXSIM_NCOUNTERS : nullptr;
        double* rs = (ret_sums && counters) ? rs_base + 2 * g : nullptr;
        const float sigma_dyn = grp.sigma_dyn;

        EnvRegs e;
        load_env(st, i, e);
        uint32_t episode = st.episode[i];
        const bool tracking = st.ep_return != nullptr && st.ep_stats != nullptr;
        double ep_return = tracking ? st.ep_return[i] : 0.0;
        EpStats es{0u, 0u};
        if (tracking) { es.w0 = st.ep_stats[i]; es.w1 = st.ep_stats[ld + i]; }
        double size = st.size[i], mass = st.mass[i], friction = st.friction[i];
        bool params_dirty = false;
        float lmean[LEARNER ? NJ : 1];
        double lbest = 0.0;
        if (LEARNER) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) lmean[j] = rio.learner_mean[j * ld + i];
            lbest = rio.learner_best[i];
        }

        for (int t = 0; t < k_steps; ++t) {
            float a[NJ];
            if constexpr (MLP) {                           // dexsim_rollout_mlp: the observation this state returns from step()
                const MlpArgs& m = mlp_of(traj...);
                mlp_mean(m, sh_mlp, sh_mlp + m.scratch_off + threadIdx.x, (int)blockDim.x,
                         MlpEnvInput{e, p.seed, gid, episode, grp.sigma_obs}, a);
                if (m.action_std) {
                    float z[NJ];
                    normal_rows<NJ>(p.seed, gid, episode, (uint32_t)e.sc, STREAM_LEARNER_ACT, 1.0f, z);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) a[j] = __fadd_rn(a[j], __fmul_rn(sh_mlp[m.o_std + j], z[j]));
                }
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(a[j], -1.0f, 1.0f);
            } else if (LEARNER) {                          // SimpleLearner.select_action, policies/simple_learner.py:60-69
                float nz[NJ];
                if (rio.learner_act_noise) {
#pragma unroll
                    for (int j = 0; j < NJ; ++j) nz[j] = __ldg(rio.learner_act_noise + ((int64_t)t * NJ + j) * ld + i);
                } else {
                    normal_rows<NJ>(p.seed, gid, episode, (uint32_t)e.sc, STREAM_LEARNER_ACT, rio.learner_exploration, nz);
                }
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(__fadd_rn(lmean[j], nz[j]), -1.0f, 1.0f);
            } else if (policy_kind == DEXSIM_POLICY_EXTERNAL) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = __ldg(actions + ((int64_t)t * NJ + j) * ld + i);
            } else {
                policy_action(p.seed, gid, episode, (uint32_t)e.sc, policy_kind, a);
            }
            if constexpr (REC) record_action(traj..., ld, t, i, a);     // the policy's action, before dynamics noise
            if (dyn_noise) {                               // pre-drawn, already scaled by sigma
#pragma unroll
                for (int j = 0; j < NJ; ++j)
                    a[j] = clip_f32(__fadd_rn(a[j], __ldg(dyn_noise + ((int64_t)t * NJ + j) * ld + i)), -1.0f, 1.0f);
            } else if (sigma_dyn > 0.0f) {                 // evaluation/robustness_tests.py:180-187
                float nz[NJ];
                normal_rows<NJ>(p.seed, gid, episode, (uint32_t)e.sc, STREAM_DYN, sigma_dyn, nz);
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(__fadd_rn(a[j], nz[j]), -1.0f, 1.0f);
            }
            StepResult r;
            const uint32_t step_idx = (uint32_t)e.sc;
            // every action reaching this point is already inside [-1, 1] unless it came from an external tensor:
            // Philox policies are in range by construction, the noise and learner paths clip after adding
            if (policy_kind == DEXSIM_POLICY_EXTERNAL && !dyn_noise && !(sigma_dyn > 0.0f)) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(a[j], -1.0f, 1.0f);
            }
            env_step<DENSE, false>(e, a, p, r);
            if (LEARNER && r.total > lbest) {              // SimpleLearner.update, policies/simple_learner.py:82-95
                if (rio.learner_upd_noise) {
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const double adj = __ldg(rio.learner_upd_noise + ((int64_t)t * NJ + j) * ld + i);
                        lmean[j] = clip_f32((float)__dadd_rn((double)lmean[j], adj), -rio.learner_clip, rio.learner_clip);
                    }
                } else {
                    float nz[NJ];
                    normal_rows<NJ>(p.seed, gid, episode, step_idx, STREAM_LEARNER_UPD, rio.learner_lr, nz);
#pragma unroll
                    for (int j = 0; j < NJ; ++j)
                        lmean[j] = clip_f32((float)__dadd_rn((double)lmean[j], (double)nz[j]), -rio.learner_clip, rio.learner_clip);
                }
                lbest = r.total;
            }
            ep_return = __dadd_rn(ep_return, r.total);
            epstats_push(es, e.sc - 1, r.n_c);
            if (rio.hist && rio.step_base + t < rio.hist_steps) rio.hist[(rio.step_base + t) * ld + i] = (uint8_t)r.n_c;
            const bool done = r.terminated || r.truncated || (p.loop_max_steps > 0 && e.sc >= p.loop_max_steps);
            if constexpr (REC) record_outcome(traj..., ld, t, i, r, done);
            if (done) {
                if (LEARNER) lbest = -INFINITY;              // policy.reset() before the next episode
                EpisodeLog log;
                log.rec = rio.ep_log; log.count = reinterpret_cast<unsigned long long*>(rio.ep_log_count);
                log.capacity = rio.ep_log_capacity; log.t_end = (uint32_t)(rio.step_base + t);
                if (rio.one_episode) {          // run_episode semantics: stop here, the caller resets
                    finish_episode(e, p, gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs, &log);
                    if constexpr (REC) record_obs(traj..., ld, t, i, e);   // the terminal observation
                    if constexpr (REC) record_final_obs(traj..., ld, t, i, e);
                    break;
                }
                if constexpr (REC) record_final_obs(traj..., ld, t, i, e); // the terminal observation, before the reset
                finish_and_reset(e, p, grp, gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs,
                                 size, mass, friction, &log);
                params_dirty = true;
            }
            if constexpr (REC) record_obs(traj..., ld, t, i, e);       // after the auto-reset, as step() returns it
        }
        store_env_full(st, i, e);
        st.episode[i] = episode;
        if (tracking) {
            st.ep_return[i] = ep_return;
            st.ep_stats[i] = es.w0; st.ep_stats[ld + i] = es.w1;
        }
        if (params_dirty) { st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction; }
        if (LEARNER) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) rio.learner_mean[j * ld + i] = lmean[j];
            rio.learner_best[i] = lbest;
        }
    }
    if (staged && counters) {
        __syncthreads();
        unsigned long long* gc = reinterpret_cast<unsigned long long*>(counters);
        for (int w = threadIdx.x; w < G * DEXSIM_NCOUNTERS; w += blockDim.x)
            if (sh_cnt[w]) atomicAdd(&gc[w], sh_cnt[w]);
        if (ret_sums)
            for (int w = threadIdx.x; w < G * 2; w += blockDim.x)
                if (sh_rs[w] != 0.0) atomicAdd(&ret_sums[w], sh_rs[w]);
    }
}

// ---- exact variance ties -----------------------------------------------------------------------------------
// Runs after a rollout launch that recorded both the episode log and the per-step contact-count history: every
// logged episode whose label met an exact variance tie (var_tie == 1, decided in exact arithmetic by the rollout
// kernel) is classified again with np.var's own pairwise float64 arithmetic on its history (classify_summary with
// counts), the record and the per-group label counters are corrected and var_tie becomes 2.  Idempotent; ties are
// rare (no shipped config produces one), so this is a scan of the log and nothing else.
__global__ void resolve_ties_kernel(const DexsimParams p, const uint16_t* __restrict__ group_of_env, const DexsimRolloutIO rio,
                                    const int64_t n, const int64_t ld) {
    const unsigned long long produced = *reinterpret_cast<const unsigned long long*>(rio.ep_log_count);
    const long long kept = produced < (unsigned long long)rio.ep_log_capacity ? (long long)produced : rio.ep_log_capacity;
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < kept; q += (long long)gridDim.x * blockDim.x) {
        DexsimEpisodeRecord rec = rio.ep_log[q];
        if (rec.var_tie != 1u) continue;
        const int64_t i = (int64_t)(uint32_t)(rec.env_gid - (uint32_t)p.env_gid0);   // gids wrap at 2^32 like the Philox counter word
        const int64_t first = (int64_t)rec.t_end + 1 - rec.steps;                     // history row of the episode's first step
        if (i >= n || first < 0 || (int64_t)rec.t_end >= rio.hist_steps) continue;
        const CountsView cv{rio.hist + first * ld + i, ld};
        DexsimEpisodeSummary s;
        s.success = rec.success; s.episode_steps = rec.steps; s.num_contacts = rec.final_contacts;
        s.final_contacts = rec.final_contacts; s.hist_len = rec.steps;
        int sum = 0, sq = 0, mx = 0, f5 = 0, l5 = 0;
        for (int t = 0; t < rec.steps; ++t) {
            const int c = cv.base[(int64_t)t * ld];
            sum += c; sq += c * c; mx = c > mx ? c : mx;
            if (t < 5) f5 += c;
            if (t >= rec.steps - 5) l5 += c;
        }
        s.sum_counts = sum; s.sum_sq_counts = sq; s.max_count = mx; s.first5_sum = f5; s.last5_sum = l5;
        int la, lb, tie;
        classify_summary(s, p.loop_max_steps > 0 ? p.loop_max_steps : p.max_episode_steps, p.success_threshold, la, lb, tie, &cv);
        if (rio.counters) {
            const int g = group_of_env ? (int)group_of_env[i] : (int)(rec.env_gid % (uint32_t)p.num_groups);
            unsigned long long* cnt = reinterpret_cast<unsigned long long*>(rio.counters) + (int64_t)g * DEXSIM_NCOUNTERS;
            if (la != rec.label_metrics) {
                if (rec.label_metrics != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_METRICS + rec.label_metrics], ~0ull);
                if (la != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_METRICS + la], 1ull);
            }
            if (lb != rec.label_taxonomy) {
                if (rec.label_taxonomy != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_TAXONOMY + rec.label_taxonomy], ~0ull);
                if (lb != DEXSIM_LABEL_NONE) atomicAdd(&cnt[DEXSIM_CNT_LABEL_TAXONOMY + lb], 1ull);
            }
            atomicAdd(&cnt[DEXSIM_CNT_VAR_TIES], ~0ull);                  // no longer in doubt
        }
        rec.label_metrics = (uint8_t)la; rec.label_taxonomy = (uint8_t)lb; rec.var_tie = 2u;
        rio.ep_log[q] = rec;
    }
}

// ---- single-env read-back ------------------------------------------------------------------------------
// ---- RNG exposure ------------------------------------------------------------------------------------
__global__ void fill_policy_kernel(const DexsimState st, const DexsimParams p, int policy_kind, float* __restrict__ out) {
    const int64_t n = st.n, ld = st.ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float a[NJ];
        policy_action(p.seed, (uint32_t)(p.env_gid0 + i), st.episode[i], (uint32_t)st.step_count[i], policy_kind, a);
#pragma unroll
        for (int j = 0; j < NJ; ++j) out[j * ld + i] = a[j];
    }
}

template <int ROWS>
__global__ void fill_normal_kernel(const DexsimState st, const DexsimParams p, uint32_t stream, float sigma,
                                   float* __restrict__ out) {
    const int64_t n = st.n, ld = st.ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float z[ROWS];
        normal_rows<ROWS>(p.seed, (uint32_t)(p.env_gid0 + i), st.episode[i], (uint32_t)st.step_count[i], stream, sigma, z);
#pragma unroll
        for (int j = 0; j < ROWS; ++j) out[j * ld + i] = z[j];
    }
}

// ---- host side -----------------------------------------------------------------------------------------
struct DeviceInfo { int sm_count = 0; int step_ctas = 0; int rollout_ctas = 0; bool valid = false; };

static int query_device(DeviceInfo& d) {
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return -(int)err;
    err = cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
    if (err != cudaSuccess) return -(int)err;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d.step_ctas, step_kernel<true, false, false, false>, STEP_THREADS, 0);
    if (err != cudaSuccess) return -(int)err;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d.rollout_ctas, rollout_kernel<true, false, false>, ROLLOUT_THREADS, 0);
    if (err != cudaSuccess) return -(int)err;
    d.valid = true;
    return 0;
}

static int device_info_cached(DeviceInfo& out) {
    static thread_local DeviceInfo cache[64];
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return -(int)err;
    if (dev < 0 || dev >= 64) { return query_device(out); }
    if (!cache[dev].valid) {
        const int rc = query_device(cache[dev]);
        if (rc) return rc;
    }
    out = cache[dev];
    return 0;
}

static int check_state(const DexsimState* st) {
    if (!st) return DEXSIM_E_NULL;
    if (st->n < 0 || st->ld < st->n || (st->ld % 32) != 0) return DEXSIM_E_SIZE;
    if (!st->obs || !st->op64 || !st->thr || !st->damp || !st->step_count || !st->cmask || !st->size ||
        !st->mass || !st->friction || !st->episode)
        return DEXSIM_E_NULL;
    if ((reinterpret_cast<uintptr_t>(st->obs) & 15u) || (reinterpret_cast<uintptr_t>(st->op64) & 15u)) return DEXSIM_E_ALIGN;
    if ((st->ep_return == nullptr) != (st->ep_stats == nullptr)) return DEXSIM_E_NULL;
    return 0;
}

static int check_params(const DexsimParams* p, bool need_groups, const DexsimGroup* groups, bool tracked = false) {
    if (!p) return DEXSIM_E_NULL;
    if (p->reward_type != 0 && p->reward_type != 1) return DEXSIM_E_PARAM;
    if (p->max_episode_steps < 0 || p->success_threshold < 0) return DEXSIM_E_PARAM;
    if (tracked) {
        // the packed per-env history summary (EpStats) holds episodes of up to EPSTATS_MAX_STEPS steps; an episode
        // ends at the caller's loop bound or one step after max_episode_steps (truncation is reported one step late)
        const int64_t longest = (p->loop_max_steps > 0 && p->loop_max_steps <= p->max_episode_steps)
                                    ? p->loop_max_steps : (int64_t)p->max_episode_steps + 1;
        if (longest > EPSTATS_MAX_STEPS) return DEXSIM_E_PARAM;
    }
    if (need_groups) {
        if (p->num_groups < 1 || p->num_groups > DEXSIM_MAX_GROUPS) return DEXSIM_E_GROUPS;
        if (!groups) return DEXSIM_E_NULL;
    }
    return 0;
}

static int grid_for(int64_t n, int threads, int ctas_per_sm, int sm_count) {
    int64_t blocks = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)sm_count * (ctas_per_sm > 0 ? ctas_per_sm : 1);   // one full resident wave
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

static inline int cuda_rc(cudaError_t e) { return e == cudaSuccess ? 0 : -(int)e; }

template <bool DENSE, bool AOS>
static void launch_step_variant(bool extras, bool next, int grid, cudaStream_t s, const DexsimState& st, const DexsimParams& p,
                                const DexsimGroup* groups, const uint16_t* goe, const DexsimStepIO& io,
                                double* pack_out, double pack_tag) {
    if (next)        step_kernel<DENSE, AOS, true, true><<<grid, STEP_THREADS, 0, s>>>(st, p, groups, goe, io, pack_out, pack_tag);
    else if (extras) step_kernel<DENSE, AOS, true, false><<<grid, STEP_THREADS, 0, s>>>(st, p, groups, goe, io, pack_out, pack_tag);
    else             step_kernel<DENSE, AOS, false, false><<<grid, STEP_THREADS, 0, s>>>(st, p, groups, goe, io);
}

// Launches KERNEL with programmatic dependent launch, eagerly and inside captured graphs: its grid may start while the
// previous grid on `s` drains and blocks in griddepcontrol.wait until that grid has completed -- stream order is
// preserved for every access.  `grid_of(CTAs per SM)` must stay within one resident wave (SMs x CTAs per SM), so that
// all CTAs of a launch are resident at once and a waiting grid can never keep its predecessor's CTAs off the SMs.
template <auto KERNEL, typename GridOf, typename... Args>
static int launch_pdl(int threads, size_t smem, GridOf grid_of, cudaStream_t s, const Args&... args) {
    // per kernel and per device: the shared-memory opt-in is a per-device function attribute
    static thread_local int occupancy[64] = {0};
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return -(int)err;
    int uncached = 0;
    int& ctas_per_sm = (dev >= 0 && dev < 64) ? occupancy[dev] : uncached;
    if (ctas_per_sm == 0) {
        if (smem) {
            err = cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (err != cudaSuccess) return -(int)err;
        }
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, KERNEL, threads, smem);
        if (err != cudaSuccess) return -(int)err;
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid_of(ctas_per_sm)); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    return cuda_rc(cudaLaunchKernelEx(&cfg, KERNEL, args...));
}

template <bool DENSE, bool AOS, int TRACK, bool EXTRA, int STAGES, int TILE_, bool NEXT>
static int launch_tma_variant(int sm_count, cudaStream_t s, const DexsimState& st, const DexsimParams& p,
                              const DexsimGroup* groups, const uint16_t* goe, const DexsimStepIO& io,
                              const StepMaps& maps, int num_tiles) {
    constexpr int TMA_THREADS = TILE_ + 32;            // one compute thread per env of a tile + the producer warp
    const size_t smem = (size_t)STAGES * StageLayout<TILE_>::stage_bytes(TRACK) + 2 * STAGES * (sizeof(uint64_t) + sizeof(int)) +
                        (TRACK ? TMA_GROUPS_MAX * (DEXSIM_NCOUNTERS * sizeof(unsigned long long) + 2 * sizeof(double)) : 0);
    // Programmatic dependent launch lets this grid start (barrier init, counter staging) while the previous step's grid
    // drains.  Measured on B200, us per step with / without:
    // eager (tools/time_small.py) 131,072 envs 12.1 / 14.3, 1 Mi 67.7 / 70.0; replayed from capture_step(steps=8)
    // (tools/time_graph.py) 65,536 envs 9.4 / 10.6, 131,072 12.6 / 13.6, 1 Mi 69.2 / 70.0.  Eager stepping with PDL
    // (9.3 / 12.1 / 67.1) is as fast as a graph replay once the GPU, not the host, is the bound (>= 65,536 envs); at
    // 4,096 envs the replay wins (6.5 vs 7.5, the eager loop runs at the host's issue rate).
    return launch_pdl<step_tma_kernel<DENSE, AOS, TRACK, EXTRA, STAGES, TILE_, NEXT>>(
        TMA_THREADS, smem, [&](int ctas_per_sm) { return sm_count * ctas_per_sm < num_tiles ? sm_count * ctas_per_sm : num_tiles; }, s,
        st, p, groups, goe, io, maps, num_tiles, /*pdl=*/1);
}

// Step kernel (dexsim_set_step_impl): 0 = auto (TMA pipeline when eligible), 1 = register-resident kernel only,
// 2 = TMA pipeline required.
static int g_rollout_impl = 0;
static int g_step_impl = 0;

// Tile width of the pipelined kernel (dexsim_set_step_tile): 0 = auto, 1 = narrow (128 envs, three CTAs of four compute
// warps per SM) only, 2 = wide (224 envs, two CTAs of seven compute warps per SM) wherever it exists.  Identical results
// either way.
static int g_step_tile = 0;

static bool aligned16(const void* ptr) { return !(reinterpret_cast<uintptr_t>(ptr) & 15u); }

// What a step call asks of the kernel beyond the plain step.  track: 0 = plain step, 1 = full episode tracking (returns
// + history summaries -> labels), 2 = counts only.  extra: noise, reward components or the float64 reward.
static int step_track(const DexsimState& st, const DexsimParams& p, const DexsimStepIO& io) {
    if (!p.auto_reset && st.ep_return == nullptr && io.finished == nullptr) return 0;
    return st.ep_return != nullptr ? 1 : 2;
}
static bool step_extra_io(const DexsimStepIO& io) {
    return io.dyn_noise || io.obs_noise || io.reward_comps || io.reward64 || io.sigma_dyn != 0.0f || io.sigma_obs != 0.0f;
}

// Whether the pipelined kernel takes a step call (`single`: dexsim_step_single, which packs its env in the same launch).
// It needs 16-byte aligned bases for everything its bulk copies touch; noise / reward-component / float64-reward calls
// ride it too (their rows are accessed directly) when the actions are [n,15].  Every batch of at least one tile takes
// it: measured on B200 (tools/time_small.py, us per step, register-resident kernel vs pipeline, hard curriculum,
// 400 steps), without programmatic dependent launch the register-resident kernel won below ~80k envs (65,536 envs,
// counts: 10.2 vs 11.4) -- with it the pipeline's prologue overlaps the previous step's tail:
//   counts:  4,096 envs 7.6 vs 6.3;  16,384 8.4 vs 7.0;  65,536 10.2 vs 9.3;  131,072 15.1 vs 12.0;  196,608 20.2 vs 14.4
//   tracked: 4,096 8.7 vs 7.1;  65,536 11.1 vs 10.7;  131,072 16.8 vs 14.2;  196,608 22.5 vs 17.2
//   plain:   16,384 6.2 vs 4.9;  65,536 6.2 vs 7.0 (both at the ~5 us host issue rate);  131,072 10.3 vs 9.0
static bool pipeline_eligible(const DexsimState& st, const DexsimStepIO& io, int track, bool extra_io, bool single) {
    return (!extra_io || io.action_layout == 1) && !single && st.n >= TILE && st.n < (int64_t)0x7FFFFF00 &&
           aligned16(io.action) && aligned16(io.reward) && aligned16(st.thr) && aligned16(st.damp) &&
           aligned16(st.step_count) && aligned16(st.cmask) && aligned16(io.terminated) && aligned16(io.truncated) &&
           aligned16(io.num_contacts) && aligned16(st.episode) && aligned16(io.finished) &&
           (track != 1 || (aligned16(st.ep_return) && aligned16(st.ep_stats))) &&
           g_step_impl != 1 && get_encode_fn() != nullptr;
}

// A step of a batch whose state sits in L2 (below ~256 Ki envs) is bound by how many env-warps an SM can run side by side
// and how many of them each compute warp has to run one after the other: ceil(tiles / resident CTAs) tiles per CTA.  The
// wide tile has 14 instead of 12 compute warps per SM; it is taken when that makes the chain of tiles per CTA shorter.
// Measured (tools/time_tile.py, profiles/r02_time_tile.txt, us per step narrow / wide, counts-only): 65,536 envs 9.4 / 9.8
// (plain 7.4 / 6.5), 98,304 9.9 / 10.4, 131,072 11.7 / 10.7 (plain 9.2 / 8.9), 163,840 12.6 / 13.3, 196,608 14.1 / 13.8,
// 229,376 15.2 / 15.7, 262,144 16.9 / 16.7, 1 Mi 57.9 / 57.8 --
// HBM-bound batches gain nothing, so they stay on the narrow tile (more CTAs for the dynamic tile hand-out to balance).
static bool use_wide_tile(int64_t n, int track, int sm_count) {
    if (track == 1 || n < TILE_WIDE || TILE != 128) return false;       // full tracking: its stages only fit the narrow tile
    if (g_step_tile) return g_step_tile == 2;
    if (n >= (int64_t)1 << 18) return false;
    // tiles per resident CTA, rounded up -- a handful of CTAs with one tile more (5 % of a round) do not count as a round:
    // the dynamic hand-out spreads them over the SMs
    auto depth = [](int64_t tiles, int64_t ctas) { return (int64_t)ceil((double)tiles / (double)ctas - 0.05); };
    const int64_t depth_narrow = depth((n + TILE - 1) / TILE, 3 * (int64_t)sm_count);
    const int64_t depth_wide = depth((n + TILE_WIDE - 1) / TILE_WIDE, 2 * (int64_t)sm_count);
    return depth_wide < depth_narrow;
}

static int launch_step_tma(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups, const uint16_t* goe,
                           const DexsimStepIO* io, cudaStream_t s, int track, bool extra, bool next, int sm_count) {
    // Tensor maps are pure functions of (base pointers, n, ld): a stepping loop re-encodes nothing.  One cached set
    // per host thread; the SoA action map is keyed by the action pointer too (AoS actions use 1-D bulk copies).
    struct MapCache { const void* obs; const void* op64; const void* act; const void* host; int64_t n, ld; int tile; bool valid; StepMaps maps; };
    static thread_local MapCache cache = {nullptr, nullptr, nullptr, nullptr, 0, 0, 0, false, {}};
    const bool aos = io->action_layout == 1;
    const bool wide = use_wide_tile(st->n, track, sm_count);
    const int tile = wide ? TILE_WIDE : TILE;
    const void* act_key = aos ? nullptr : (const void*)io->action;
    // zero-copy host step: one more map, over the caller's mapped host observation (device alias of the host pointer)
    const void* host_key = (io->flags & DEXSIM_STEP_HOST_ALL_ROWS) ? (const void*)io->host_static_rows : nullptr;
    if (!(cache.valid && cache.obs == st->obs && cache.op64 == st->op64 && cache.act == act_key && cache.host == host_key &&
          cache.n == st->n && cache.ld == st->ld && cache.tile == tile)) {
        cache.valid = false;
        memset(&cache.maps, 0, sizeof(cache.maps));
        bool ok = make_map_2d(&cache.maps.obs_jpjv, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, st->obs, st->n, st->ld, DEXSIM_OBS, 30, tile) &&
                  make_map_2d(&cache.maps.obs_ov, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, st->obs, st->n, st->ld, DEXSIM_OBS, 3, tile) &&
                  make_map_2d(&cache.maps.op64, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 8, st->op64, st->n, st->ld, 3, 3, tile);
        if (ok && !aos)
            ok = make_map_2d(&cache.maps.act_soa, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(io->action), st->n,
                             st->ld, NJ, NJ, tile);
        if (ok && host_key)
            ok = make_map_2d(&cache.maps.host_jpjv, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(host_key), st->n, st->ld,
                             DEXSIM_OBS, 30, tile);
        if (!ok) return 1;                           // caller falls back to the register-resident kernel
        cache.obs = st->obs; cache.op64 = st->op64; cache.act = act_key; cache.host = host_key; cache.n = st->n; cache.ld = st->ld; cache.tile = tile;
        cache.valid = true;
    }
    const StepMaps& maps = cache.maps;
    const int num_tiles = (int)((st->n + tile - 1) / tile);
    // runtime (dense, aos, track, extra, next) -> template arguments: each call hands its value on as a std::integral_constant
    const auto as_bool = [](bool b, auto&& f) { return b ? f(std::true_type{}) : f(std::false_type{}); };
    const auto as_track = [](int t, auto&& f) {
        using std::integral_constant;
        return t == 1 ? f(integral_constant<int, 1>{}) : t == 2 ? f(integral_constant<int, 2>{}) : f(integral_constant<int, 0>{});
    };
    return as_bool(p->reward_type == 1, [&](auto dense) {
        return as_bool(aos, [&](auto aos_) {
            return as_track(track, [&](auto track_) {
                return as_bool(extra, [&](auto extra_) {
                    return as_bool(next, [&](auto next_) -> int {
                        constexpr bool DENSE = decltype(dense)::value, AOS = decltype(aos_)::value, EXTRA = decltype(extra_)::value;
                        constexpr int TRACK = decltype(track_)::value;
                        constexpr bool NEXT = decltype(next_)::value;
                        // The instantiations: noise / reward components only with the reference's [n,15] action layout
                        // (SoA callers take the register kernel), the wide tile only without full tracking (its stages
                        // have no room for the per-env return / history arrays), and next-step auto-reset only with the
                        // episode bookkeeping (an auto-reset call always has TRACK 1 or 2).
                        if constexpr ((EXTRA && !AOS) || (NEXT && TRACK == 0)) {
                            return 1;
                        } else {
                            if constexpr (TRACK != 1) {
                                if (wide)
                                    return launch_tma_variant<DENSE, AOS, TRACK, EXTRA, 2, TILE_WIDE, NEXT>(sm_count, s, *st, *p,
                                                                                                            groups, goe, *io, maps,
                                                                                                            num_tiles);
                            }
                            return launch_tma_variant<DENSE, AOS, TRACK, EXTRA, DEXSIM_TMA_STAGES, TILE, NEXT>(sm_count, s, *st, *p,
                                                                                                               groups, goe, *io,
                                                                                                               maps, num_tiles);
                        }
                    });
                });
            });
        });
    });
}

// next: next-step auto-reset (dexsim_step_next_reset; the caller has checked its arguments).
static int launch_step(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                       const uint16_t* goe, const DexsimStepIO* io, cudaStream_t s,
                       double* pack_out = nullptr, double pack_tag = 0.0, bool next = false) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!io || !io->action || !io->reward || !io->terminated || !io->truncated || !io->num_contacts) return DEXSIM_E_NULL;
    if (io->action_layout != 0 && io->action_layout != 1) return DEXSIM_E_PARAM;
    const bool fused_dyn = !io->dyn_noise && io->sigma_dyn != 0.0f;
    const bool fused_obs = !io->obs_noise && io->sigma_obs != 0.0f;
    if ((io->obs_noise != nullptr || fused_obs) != (io->noisy_obs != nullptr)) return DEXSIM_E_NULL;
    if (pack_out && st->n != 1) return DEXSIM_E_SIZE;
    const bool extras = io->dyn_noise || io->obs_noise || io->reward_comps || io->reward64 || io->finished || io->host_static_rows ||
                        (p && p->auto_reset) || st->ep_return != nullptr || fused_dyn || fused_obs || pack_out != nullptr;
    const bool group_sigma = (fused_dyn && io->sigma_dyn < 0.0f) || (fused_obs && io->sigma_obs < 0.0f);
    rc = check_params(p, p && (p->auto_reset || group_sigma), groups, st->ep_return != nullptr && p && p->auto_reset);
    if (rc) return rc;
    if (st->n == 0) return 0;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    const int track = step_track(*st, *p, *io);
    const bool extra_io = step_extra_io(*io);
    if (pipeline_eligible(*st, *io, track, extra_io, pack_out != nullptr)) {
        rc = launch_step_tma(st, p, groups, goe, io, s, track, extra_io, next, di.sm_count);
        if (rc <= 0) return rc;                      // launched (0) or CUDA error (< 0); 1 = a tensor map was rejected
    }
    if (g_step_impl == 2) return DEXSIM_E_PARAM;     // TMA pipeline was demanded but is not eligible
    if (io->flags & DEXSIM_STEP_HOST_ALL_ROWS) return DEXSIM_E_PARAM;   // only the pipelined kernel mirrors every row
    const int grid = grid_for(st->n, STEP_THREADS, di.step_ctas, di.sm_count);
    const bool dense = p->reward_type == 1, aos = io->action_layout == 1;
    if (dense) { if (aos) launch_step_variant<true, true>(extras, next, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag);
                 else     launch_step_variant<true, false>(extras, next, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag); }
    else       { if (aos) launch_step_variant<false, true>(extras, next, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag);
                 else     launch_step_variant<false, false>(extras, next, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag); }
    return cuda_rc(cudaGetLastError());
}

// dexsim_step_final (HOST: one chunk of dexsim_step_host_final, outputs in `hf`): the step without the reset, which leaves
// the observation of the step that ended an episode in obs / noisy_obs and writes neither `finished` nor the counters,
// then the finish-and-reset pass, which resets, counts and writes them.  The pass is one resident wave of CTAs, launched
// as a programmatic dependent of the step, so that its launch and counter staging overlap the step's tail.
template <bool HOST>
static int step_then_finish_reset(const DexsimState& st, const DexsimParams& p, const DexsimGroup* groups, const uint16_t* goe,
                                  const DexsimStepIO& io, float* final_obs, const FinishHost& hf, cudaStream_t s) {
    DexsimParams sp = p;
    sp.auto_reset = 0;
    DexsimStepIO sio = io;
    sio.finished = nullptr; sio.counters = nullptr; sio.ret_sums = nullptr;
    int rc = launch_step(&st, &sp, groups, goe, &sio, s);
    if (rc || st.n == 0) return rc;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    // HOST: the record blocks and the static counter arrays together exceed the default 48 KB of shared memory
    return launch_pdl<finish_reset_kernel<HOST>>(
        STEP_THREADS, HOST ? FINISH_HOST_SMEM : 0,
        [&](int ctas_per_sm) { return grid_for(st.n, STEP_THREADS, ctas_per_sm, di.sm_count); }, s,
        st, p, groups, goe, io, final_obs, /*pdl=*/1, hf);
}

// The arguments every auto-reset entry point checks first, in this order: p and io, auto-reset on, then its outputs
// (`outputs`: whether the entry point's own outputs are present; io->finished is one of every such entry point).
static int check_auto_reset(const DexsimParams* p, const DexsimStepIO* io, bool outputs) {
    if (!p || !io) return DEXSIM_E_NULL;
    if (!p->auto_reset) return DEXSIM_E_PARAM;
    if (!outputs || !io->finished) return DEXSIM_E_NULL;
    return 0;
}

// ... and, of the entry points that run the step without the reset (step_then_finish_reset), the state and the limits of
// an auto-reset call, which that step does not check.
static int check_finish_reset(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups, const DexsimStepIO* io,
                              bool outputs) {
    int rc = check_auto_reset(p, io, outputs);
    if (rc) return rc;
    rc = check_state(st);
    if (rc) return rc;
    return check_params(p, true, groups, st->ep_return != nullptr);
}

}  // namespace dexsim

namespace dexsim {
// csrc/dexsim_host_expand.cpp: observation rows 40-44 of envs [lo, hi) from their 1-byte contact masks (host code)
void expand_contact_rows_range(float* h_obs, const uint8_t* mask, int64_t lo, int64_t hi, int64_t ld);
}  // namespace dexsim

using namespace dexsim;

template <bool TAGGED>
static int pack_env(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset, double* out64,
                    double tag, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!io || !out64 || !io->reward || !io->terminated || !io->truncated) return DEXSIM_E_NULL;
    if (index < 0 || index >= st->n) return DEXSIM_E_SIZE;
    pack_env_kernel<TAGGED><<<1, 64, 0, (cudaStream_t)stream>>>(*st, *io, index, after_reset ? 1 : 0, out64, tag);
    return cuda_rc(cudaGetLastError());
}

static std::atomic<int64_t> g_zero_copy_steps{0};    // dexsim_step_host calls served by the single-launch transport

extern "C" {

int dexsim_version(void) { return DEXSIM_ABI_VERSION; }

const char* dexsim_error_string(int code) {
    switch (code) {
        case DEXSIM_OK: return "ok";
        case DEXSIM_E_NULL: return "dexsim: required pointer is NULL";
        case DEXSIM_E_SIZE: return "dexsim: bad size (need n >= 0, ld >= n, ld % 32 == 0, k_steps >= 1)";
        case DEXSIM_E_ALIGN: return "dexsim: array base not 16-byte aligned";
        case DEXSIM_E_PARAM: return "dexsim: bad enum, flag or parameter value (tracked episodes hold at most 5,242 steps)";
        case DEXSIM_E_GROUPS: return "dexsim: num_groups out of range";
        case DEXSIM_E_GEOMETRY: return "dexsim: only num_fingers=5, joints_per_finger=3 is supported";
        default: break;
    }
    if (code < 0 && code > -1000) return cudaGetErrorString((cudaError_t)(-code));
    return "dexsim: unknown error code";
}

int dexsim_set_step_impl(int impl) {
    if (impl < 0 || impl > 2) return DEXSIM_E_PARAM;
    g_step_impl = impl;
    return 0;
}

int dexsim_set_step_tile(int tile) {
    if (tile < 0 || tile > 2) return DEXSIM_E_PARAM;
    g_step_tile = tile;
    return 0;
}

int dexsim_set_rollout_impl(int impl) {
    if (impl < 0 || impl > 2) return DEXSIM_E_PARAM;
    g_rollout_impl = impl;
    return 0;
}

int dexsim_sizeof_state(void) { return (int)sizeof(DexsimState); }
int dexsim_sizeof_params(void) { return (int)sizeof(DexsimParams); }
int dexsim_sizeof_group(void) { return (int)sizeof(DexsimGroup); }
int dexsim_sizeof_step_io(void) { return (int)sizeof(DexsimStepIO); }
int dexsim_sizeof_rollout_io(void) { return (int)sizeof(DexsimRolloutIO); }
int dexsim_sizeof_episode_record(void) { return (int)sizeof(DexsimEpisodeRecord); }
int dexsim_sizeof_trajectory(void) { return (int)sizeof(DexsimTrajectory); }

int dexsim_device_info(int* sm_count, int* step_ctas_per_sm, int* rollout_ctas_per_sm) {
    DeviceInfo di;
    const int rc = device_info_cached(di);
    if (rc) return rc;
    if (sm_count) *sm_count = di.sm_count;
    if (step_ctas_per_sm) *step_ctas_per_sm = di.step_ctas;
    if (rollout_ctas_per_sm) *rollout_ctas_per_sm = di.rollout_ctas;
    return 0;
}

int dexsim_reset_predrawn(const DexsimState* st, const DexsimParams* p, const uint8_t* mask, const float* jp0,
                          const double* size, const double* mass, const double* friction, const float* pos,
                          void* stream) {
    (void)p;
    int rc = check_state(st);
    if (rc) return rc;
    if (!jp0 || !size || !mass || !friction) return DEXSIM_E_NULL;
    if (st->n == 0) return 0;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    const int grid = grid_for(st->n, STEP_THREADS, 4, di.sm_count);
    reset_predrawn_kernel<<<grid, STEP_THREADS, 0, (cudaStream_t)stream>>>(*st, mask, jp0, size, mass, friction, pos);
    return cuda_rc(cudaGetLastError());
}

int dexsim_reset_philox(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                        const uint16_t* group_of_env, const uint8_t* mask, int32_t respawn, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    rc = check_params(p, true, groups);
    if (rc) return rc;
    if (st->n == 0) return 0;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    const int grid = grid_for(st->n, STEP_THREADS, 4, di.sm_count);
    reset_philox_kernel<<<grid, STEP_THREADS, 0, (cudaStream_t)stream>>>(*st, *p, groups, group_of_env, mask, respawn ? 1 : 0);
    return cuda_rc(cudaGetLastError());
}

int dexsim_step(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                const uint16_t* group_of_env, const DexsimStepIO* io, void* stream) {
    if (!p) return DEXSIM_E_NULL;
    return launch_step(st, p, groups, group_of_env, io, (cudaStream_t)stream);
}

int dexsim_step_single(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                       const uint16_t* group_of_env, const DexsimStepIO* io, double* out64, double tag, void* stream) {
    if (!p || !out64) return DEXSIM_E_NULL;
    return launch_step(st, p, groups, group_of_env, io, (cudaStream_t)stream, out64, tag);
}

int dexsim_step_final(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                      const uint16_t* group_of_env, const DexsimStepIO* io, float* final_obs, void* stream) {
    // the host mirrors are dexsim_step_host's (a NULL p or io is check_auto_reset's error)
    if (p && io && (io->host_static_rows || (io->flags & DEXSIM_STEP_HOST_ALL_ROWS))) return DEXSIM_E_PARAM;
    const int rc = check_finish_reset(st, p, groups, io, final_obs != nullptr);
    if (rc) return rc;
    return step_then_finish_reset<false>(*st, *p, groups, group_of_env, *io, final_obs, FinishHost{}, (cudaStream_t)stream);
}

int dexsim_step_next_reset(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                           const uint16_t* group_of_env, const DexsimStepIO* io, void* stream) {
    // the host mirrors are dexsim_step_host's (a NULL p or io is check_auto_reset's error)
    if (p && io && (io->host_static_rows || (io->flags & DEXSIM_STEP_HOST_ALL_ROWS))) return DEXSIM_E_PARAM;
    const int rc = check_auto_reset(p, io, true);
    if (rc) return rc;
    return launch_step(st, p, groups, group_of_env, io, (cudaStream_t)stream, nullptr, 0.0, /*next=*/true);
}

// DexsimMlpPolicy -> MlpArgs (shape checks and the shared-memory layout of mlp_stage); no device call
static int mlp_args(const DexsimMlpPolicy* pol, MlpArgs& m) {
    if (!pol || !pol->params) return DEXSIM_E_NULL;
    if (pol->num_hidden != 1 && pol->num_hidden != 2) return DEXSIM_E_PARAM;
    for (int l = 0; l < pol->num_hidden; ++l)
        if (pol->hidden[l] < 1 || pol->hidden[l] > DEXSIM_MLP_MAX_WIDTH) return DEXSIM_E_PARAM;
    if (pol->activation != DEXSIM_ACT_RELU && pol->activation != DEXSIM_ACT_TANH) return DEXSIM_E_PARAM;
    if (!aligned16(pol->params) || !aligned16(pol->action_std)) return DEXSIM_E_ALIGN;
    const auto pad = [](int h) { return (h + MLP_BLOCK - 1) / MLP_BLOCK * MLP_BLOCK; };
    m.params = pol->params; m.action_std = pol->action_std;
    m.nh = pol->num_hidden; m.h1 = pol->hidden[0]; m.h2 = m.nh == 2 ? pol->hidden[1] : 0; m.act = pol->activation;
    m.h1p = pad(m.h1); m.h2p = m.nh == 2 ? pad(m.h2) : 0;
    m.o_b1 = NOBS * m.h1p;
    m.o_w2 = m.o_b1 + m.h1p;
    m.o_b2 = m.o_w2 + m.h1 * m.h2p;
    m.o_w3 = m.o_b2 + m.h2p;
    m.o_b3 = m.o_w3 + (m.nh == 2 ? m.h2 : m.h1) * MLP_BLOCK;
    m.o_std = m.o_b3 + MLP_BLOCK;
    m.words = m.o_std + MLP_BLOCK;
    m.scratch_off = m.words;
    return 0;
}

// bytes of shared memory the MLP needs behind `base` bytes: weights + one scratch float per first-layer unit and thread
static size_t mlp_smem(const MlpArgs& m, size_t base, int threads) {
    return ((base + 15) & ~(size_t)15) + (size_t)m.words * 4 + (m.nh == 2 ? (size_t)m.h1 * threads * 4 : 0);
}

// dexsim_rollout (traj == NULL), dexsim_rollout_record (final_obs == NULL) and dexsim_rollout_record_final; with `mlp`
// dexsim_rollout_mlp (policy_kind == DEXSIM_POLICY_MLP_KIND)
static int rollout_launch(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups, const uint16_t* group_of_env,
                          int32_t k_steps, int32_t policy_kind, const DexsimRolloutIO* rio, const DexsimTrajectory* traj,
                          float* final_obs, void* stream, const MlpArgs* mlp = nullptr) {
    int rc = check_state(st);
    if (rc) return rc;
    rc = check_params(p, true, groups, st->ep_return != nullptr);
    if (rc) return rc;
    if (!rio) return DEXSIM_E_NULL;
    if (k_steps < 1) return DEXSIM_E_SIZE;
    if ((policy_kind < DEXSIM_POLICY_EXTERNAL || policy_kind > DEXSIM_POLICY_LEARNER) &&
        !(mlp && policy_kind == DEXSIM_POLICY_MLP_KIND))
        return DEXSIM_E_PARAM;
    if (policy_kind == DEXSIM_POLICY_EXTERNAL && !rio->actions) return DEXSIM_E_NULL;
    if (policy_kind == DEXSIM_POLICY_LEARNER && (!rio->learner_mean || !rio->learner_best)) return DEXSIM_E_NULL;
    if (rio->ret_sums && !rio->counters) return DEXSIM_E_NULL;
    if ((rio->counters || rio->ep_log) && !st->ep_return) return DEXSIM_E_NULL;   // labels need the per-env history summary
    if (rio->ep_log && (!rio->ep_log_count || rio->ep_log_capacity < 0)) return DEXSIM_E_NULL;
    if (rio->hist && rio->hist_steps < 0) return DEXSIM_E_SIZE;
    // small batches with an in-kernel policy: 5 lanes per env (dexsim_rollout_split.cuh); the crossover with the
    // one-thread-per-env kernel was measured between 4k and 16k envs on B200 (DESIGN.md 5.2).  Only the one-thread-per-env
    // kernel records a trajectory.
    const bool split_ok = (rio->flags & DEXSIM_ROLLOUT_NO_DYN_NOISE) && !rio->dyn_noise && st->ep_return != nullptr &&
                          (policy_kind == DEXSIM_POLICY_RANDOM || policy_kind == DEXSIM_POLICY_HEURISTIC);
    if (traj) {
        if (!traj->obs || !traj->reward || !traj->terminated || !traj->truncated || !traj->finished ||
            (!traj->action && policy_kind != DEXSIM_POLICY_EXTERNAL))
            return DEXSIM_E_NULL;
        if (k_steps > traj->capacity) return DEXSIM_E_SIZE;
        if (!aligned16(traj->obs) || !aligned16(traj->action) || !aligned16(traj->reward) || !aligned16(traj->terminated) ||
            !aligned16(traj->truncated) || !aligned16(traj->finished) || !aligned16(final_obs))
            return DEXSIM_E_ALIGN;
        if (split_ok && g_rollout_impl == 2) return DEXSIM_E_PARAM;
    }
    if (st->n == 0) return 0;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    // Small batches are latency-bound: spread warps over as many SM sub-partitions as possible
    // (4 per SM) by shrinking the CTA; large batches use full 256-thread CTAs.
    const int64_t warps = (st->n + 31) / 32;
    int threads = ROLLOUT_THREADS;
    while (threads > 32 && warps * 32 / threads < (int64_t)di.sm_count * 4) threads = (threads / 2 + 31) / 32 * 32;
    const int64_t blocks = (st->n + threads - 1) / threads;
    if (blocks > 0x7FFFFFFFll) return DEXSIM_E_SIZE;
    const int G = p->num_groups;
    const size_t smem = G <= SMEM_GROUPS_MAX
        ? (size_t)G * (sizeof(DexsimGroup) + DEXSIM_NCOUNTERS * sizeof(unsigned long long) + 2 * sizeof(double)) : 0;
    cudaStream_t s = (cudaStream_t)stream;
    const bool dense = p->reward_type == 1, learner = policy_kind == DEXSIM_POLICY_LEARNER;
    // the one-thread-per-env kernel, recording (one trailing DexsimTrajectory or TrajectoryFinal) or not (none)
    auto launch_thread_kernel = [&](const auto&... tr) {
        constexpr bool REC = sizeof...(tr) == 1;
        if (dense && learner) rollout_kernel<true, true, REC><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio, tr...);
        else if (dense) rollout_kernel<true, false, REC><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio, tr...);
        else if (learner) rollout_kernel<false, true, REC><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio, tr...);
        else rollout_kernel<false, false, REC><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio, tr...);
    };
    // the MLP policy: the one-thread-per-env kernel with the weights (and the second layer's scratch) in shared memory
    auto launch_mlp_kernel = [&](const auto&... tr) {
        constexpr bool REC = sizeof...(tr) == 1;
        const auto kernel = dense ? rollout_kernel<true, false, REC, MlpArgs, std::decay_t<decltype(tr)>...>
                                  : rollout_kernel<false, false, REC, MlpArgs, std::decay_t<decltype(tr)>...>;
        const size_t msmem = mlp_smem(*mlp, smem, threads);
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)msmem);
        if (e != cudaSuccess) return cuda_rc(e);
        kernel<<<(int)blocks, threads, msmem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio, *mlp, tr...);
        return 0;
    };
    if (mlp) {
        rc = traj && final_obs ? launch_mlp_kernel(TrajectoryFinal{*traj, final_obs})
           : traj              ? launch_mlp_kernel(*traj)
                               : launch_mlp_kernel();
        if (rc) return rc;
    } else if (split_ok && !traj && g_rollout_impl != 1 && (g_rollout_impl == 2 || st->n <= 8192)) {
        const int64_t warps_needed = (st->n + SPLIT_ENVS_PER_WARP - 1) / SPLIT_ENVS_PER_WARP;
        const int64_t sblocks = (warps_needed * 32 + SPLIT_THREADS - 1) / SPLIT_THREADS;
        if (sblocks > 0x7FFFFFFFll) return DEXSIM_E_SIZE;
        if (dense) rollout_split_kernel<true><<<(int)sblocks, SPLIT_THREADS, 0, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
        else rollout_split_kernel<false><<<(int)sblocks, SPLIT_THREADS, 0, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
    } else if (traj && final_obs) {
        launch_thread_kernel(TrajectoryFinal{*traj, final_obs});
    } else if (traj) {
        launch_thread_kernel(*traj);
    } else {
        launch_thread_kernel();
    }
    rc = cuda_rc(cudaGetLastError());
    if (rc) return rc;
    if (rio->ep_log && rio->hist && rio->ep_log_capacity > 0) {
        // exact variance ties flagged by the launch above are decided with np.var's arithmetic on the recorded history
        const long long rblocks = (rio->ep_log_capacity + 255) / 256;
        resolve_ties_kernel<<<(int)(rblocks > 4096 ? 4096 : rblocks), 256, 0, s>>>(*p, group_of_env, *rio, st->n, st->ld);
        rc = cuda_rc(cudaGetLastError());
    }
    return rc;
}

int dexsim_rollout(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                   const uint16_t* group_of_env, int32_t k_steps, int32_t policy_kind, const DexsimRolloutIO* rio,
                   void* stream) {
    return rollout_launch(st, p, groups, group_of_env, k_steps, policy_kind, rio, nullptr, nullptr, stream);
}

int dexsim_rollout_record(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                          const uint16_t* group_of_env, int32_t k_steps, int32_t policy_kind, const DexsimRolloutIO* rio,
                          const DexsimTrajectory* traj, void* stream) {
    if (!traj) return DEXSIM_E_NULL;
    return rollout_launch(st, p, groups, group_of_env, k_steps, policy_kind, rio, traj, nullptr, stream);
}

int dexsim_rollout_record_final(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                                const uint16_t* group_of_env, int32_t k_steps, int32_t policy_kind, const DexsimRolloutIO* rio,
                                const DexsimTrajectory* traj, float* final_obs, void* stream) {
    if (!traj || !final_obs) return DEXSIM_E_NULL;
    return rollout_launch(st, p, groups, group_of_env, k_steps, policy_kind, rio, traj, final_obs, stream);
}

int dexsim_sizeof_mlp_policy(void) { return (int)sizeof(DexsimMlpPolicy); }

int dexsim_rollout_mlp(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                       const uint16_t* group_of_env, int32_t k_steps, const DexsimRolloutIO* rio,
                       const DexsimMlpPolicy* policy, const DexsimTrajectory* traj, float* final_obs, void* stream) {
    MlpArgs m;
    const int rc = mlp_args(policy, m);
    if (rc) return rc;
    if (final_obs && !traj) return DEXSIM_E_NULL;
    if (rio && (rio->actions || rio->learner_mean || rio->learner_best || rio->learner_act_noise || rio->learner_upd_noise))
        return DEXSIM_E_PARAM;
    return rollout_launch(st, p, groups, group_of_env, k_steps, DEXSIM_POLICY_MLP_KIND, rio, traj, final_obs, stream, &m);
}

int dexsim_mlp_policy_mean(const DexsimMlpPolicy* policy, const float* obs, int64_t n, int64_t ld, float* out, void* stream) {
    MlpArgs m;
    const int rc = mlp_args(policy, m);
    if (rc) return rc;
    if (n < 0 || ld < n || ld % 32 != 0) return DEXSIM_E_SIZE;
    if (n == 0) return 0;
    if (!obs || !out) return DEXSIM_E_NULL;
    const int64_t blocks = (n + 255) / 256;
    if (blocks > 0x7FFFFFFFll) return DEXSIM_E_SIZE;
    const size_t smem = mlp_smem(m, 0, 256);
    cudaError_t e = cudaFuncSetAttribute(mlp_mean_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_rc(e);
    mlp_mean_kernel<<<(int)blocks, 256, smem, (cudaStream_t)stream>>>(m, obs, n, ld, out);
    return cuda_rc(cudaGetLastError());
}

int dexsim_pack_env(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset, double* out64,
                    void* stream) {
    return pack_env<false>(st, io, index, after_reset, out64, 0.0, stream);
}

int dexsim_pack_env_tagged(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset, double* out64,
                           double tag, void* stream) {
    return pack_env<true>(st, io, index, after_reset, out64, tag, stream);
}

int dexsim_fill_policy_actions(const DexsimState* st, const DexsimParams* p, int32_t policy_kind, float* actions,
                               void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p || !actions) return DEXSIM_E_NULL;
    if (policy_kind != DEXSIM_POLICY_RANDOM && policy_kind != DEXSIM_POLICY_HEURISTIC) return DEXSIM_E_PARAM;
    if (st->n == 0) return 0;
    const int grid = (int)((st->n + 255) / 256 > 65535 ? 65535 : (st->n + 255) / 256);
    fill_policy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*st, *p, policy_kind, actions);
    return cuda_rc(cudaGetLastError());
}

int dexsim_fill_normal(const DexsimState* st, const DexsimParams* p, int32_t rng_stream, int32_t rows, float sigma,
                       float* out, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p || !out) return DEXSIM_E_NULL;
    if (rng_stream < (int)STREAM_DYN || rng_stream > (int)STREAM_LEARNER_UPD) return DEXSIM_E_PARAM;
    if (rows != NJ && rows != NOBS) return DEXSIM_E_PARAM;
    if (st->n == 0) return 0;
    const int grid = (int)((st->n + 255) / 256 > 65535 ? 65535 : (st->n + 255) / 256);
    if (rows == NJ) fill_normal_kernel<NJ><<<grid, 256, 0, (cudaStream_t)stream>>>(*st, *p, (uint32_t)rng_stream, sigma, out);
    else fill_normal_kernel<NOBS><<<grid, 256, 0, (cudaStream_t)stream>>>(*st, *p, (uint32_t)rng_stream, sigma, out);
    return cuda_rc(cudaGetLastError());
}

int dexsim_classify_summary(const DexsimEpisodeSummary* s, const uint8_t* counts, int32_t max_steps,
                            int32_t success_threshold, int32_t* label_metrics, int32_t* label_taxonomy, int32_t* var_tie) {
    if (!s || !label_metrics || !label_taxonomy) return DEXSIM_E_NULL;
    if (s->hist_len < 0) return DEXSIM_E_SIZE;
    int la, lb, tie;
    const CountsView cv{counts, 1};
    classify_summary(*s, max_steps, success_threshold, la, lb, tie, &cv);
    *label_metrics = la; *label_taxonomy = lb;
    if (var_tie) *var_tie = tie;
    return 0;
}

// ---- host-buffer step: chunked so that H2D of chunk c+1, the kernel of chunk c and D2H of chunk c-1
//      overlap (separate copy engines per direction).  Internal streams/events are created once per
//      device and fork from / join into the caller's stream, so the call stays stream-ordered. ----------
namespace {
constexpr int HOST_STREAMS = 3;        // chunk c: upload, kernel and observation download on stream c % 3
constexpr int HOST_MAX_CHUNKS = 32;
struct HostPipe {
    bool ready = false;
    cudaStream_t streams[HOST_STREAMS];
    cudaStream_t small;                // per-env vectors (reward, flags) of the WHOLE batch: a few large copies instead of
                                       // one small copy per vector per chunk
    cudaEvent_t fork_ev;
    cudaEvent_t join_ev[HOST_STREAMS + 1];
    cudaEvent_t kdone[HOST_MAX_CHUNKS];
};
HostPipe g_pipes[64];
std::mutex g_pipes_mutex;      // first use from several host threads at once
std::mutex g_enqueue_mutex[64];   // per device: the fork / join events of a device's pipe are reused by every call on it

int get_pipe(HostPipe** out) {
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return -(int)err;
    if (dev < 0 || dev >= 64) return DEXSIM_E_PARAM;
    HostPipe& hp = g_pipes[dev];
    std::lock_guard<std::mutex> lock(g_pipes_mutex);
    if (!hp.ready) {
        for (int k = 0; k < HOST_STREAMS; ++k) {
            err = cudaStreamCreateWithFlags(&hp.streams[k], cudaStreamNonBlocking);
            if (err != cudaSuccess) return -(int)err;
        }
        err = cudaStreamCreateWithFlags(&hp.small, cudaStreamNonBlocking);
        if (err != cudaSuccess) return -(int)err;
        for (int k = 0; k < HOST_STREAMS + 1; ++k) {
            err = cudaEventCreateWithFlags(&hp.join_ev[k], cudaEventDisableTiming);
            if (err != cudaSuccess) return -(int)err;
        }
        for (int k = 0; k < HOST_MAX_CHUNKS; ++k) {
            err = cudaEventCreateWithFlags(&hp.kdone[k], cudaEventDisableTiming);
            if (err != cudaSuccess) return -(int)err;
        }
        err = cudaEventCreateWithFlags(&hp.fork_ev, cudaEventDisableTiming);
        if (err != cudaSuccess) return -(int)err;
        hp.ready = true;
    }
    *out = &hp;
    return 0;
}
}  // namespace

// DEXSIM_HOST_TRACE=1: device-side timeline of every tenth chunked dexsim_step_host call on stderr (experiments): when each
// chunk's upload, kernel and row download finished, relative to the call's fork point (profiles/r02_host_step_timeline.txt).
static bool host_trace() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DEXSIM_HOST_TRACE");
        v = (e && atoi(e)) ? 1 : 0;
    }
    return v == 1;
}
struct HostTrace {               // one set of timing events, owned by the first device (and thread) that traces
    cudaEvent_t t0, up[HOST_MAX_CHUNKS], k[HOST_MAX_CHUNKS], down[HOST_MAX_CHUNKS], small;
    int dev = -1;
    bool make(int device) {
        if (dev >= 0) return dev == device;
        bool ok = cudaEventCreate(&t0) == cudaSuccess && cudaEventCreate(&small) == cudaSuccess;
        for (int i = 0; ok && i < HOST_MAX_CHUNKS; ++i)
            ok = cudaEventCreate(&up[i]) == cudaSuccess && cudaEventCreate(&k[i]) == cudaSuccess && cudaEventCreate(&down[i]) == cudaSuccess;
        if (!ok) { (void)cudaGetLastError(); return false; }
        dev = device;
        return true;
    }
};
static HostTrace g_trace;
static std::atomic<int> g_trace_calls{0};

int dexsim_expand_contact_rows(float* h_obs, const uint8_t* h_contact_mask, int64_t n, int64_t ld) {
    if (!h_obs || !h_contact_mask) return DEXSIM_E_NULL;
    if (n < 0 || ld < n) return DEXSIM_E_SIZE;
    expand_contact_rows_range(h_obs, h_contact_mask, 0, n, ld);
    return 0;
}

int64_t dexsim_host_zero_copy_steps(void) { return g_zero_copy_steps.load(std::memory_order_relaxed); }

static void* mapped_alias(const void* h) {       // device alias of mapped page-locked host memory, else NULL
    if (!h) return nullptr;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, h) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
        return attr.devicePointer;
    (void)cudaGetLastError();
    return nullptr;
}

// dexsim_step_host and, with final outputs (h_final_obs != NULL, argument checks done by the caller),
// dexsim_step_host_final: per chunk, the step without the reset and then the finish-and-reset pass, after which
// everything that chunk moves to the host is enqueued.
static int step_host_impl(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                          const uint16_t* group_of_env, const DexsimStepIO* io, const float* h_action, float* h_obs,
                          float* h_reward, uint8_t* h_terminated, uint8_t* h_truncated, uint8_t* h_num_contacts,
                          uint8_t* h_contact_mask, uint8_t* h_finished, float* h_final_obs, int32_t chunks, int32_t flags,
                          void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p || !io || !io->action || !h_action || !h_reward || !h_terminated || !h_truncated) return DEXSIM_E_NULL;
    if ((flags & DEXSIM_HOST_PACKED_CONTACTS) && !h_contact_mask) return DEXSIM_E_NULL;
    if (io->dyn_noise || io->obs_noise || io->noisy_obs || io->sigma_dyn != 0.0f || io->sigma_obs != 0.0f)
        return DEXSIM_E_PARAM;   // noise: use dexsim_step
    const bool final = h_final_obs != nullptr;
    float* d_final = nullptr;                    // device alias of h_final_obs
    if (final) {
        d_final = static_cast<float*>(mapped_alias(h_final_obs));
        if (!d_final) return DEXSIM_E_PARAM;
    }
    cudaStream_t user = (cudaStream_t)stream;
    const int64_t n = st->n, ld = st->ld;
    if (n == 0) return 0;
    const bool aos = io->action_layout == 1;
    // Zero-copy transport (DEXSIM_HOST_ZERO_COPY): the pipelined kernel itself writes every result into the caller's mapped
    // page-locked buffers -- the joint rows as a second bulk tensor store per tile, object z, its velocity and the contact
    // mask as three more bulk rows, x / y and their velocities when a reset changes them (h_obs must be current, as for
    // DEXSIM_HOST_STATIC_ROWS) -- so nothing is downloaded by the copy engine: no per-copy hand-over times, no pipeline
    // fill, and the download of a tile starts the moment it is computed.  The contact rows follow from the mask
    // (PACKED_CONTACTS semantics; EXPAND_CONTACTS as below).  The actions come up chunk by chunk on the copy engine: uploads
    // of chunk k+1 overlap the PCIe writes of chunk k's kernel.  The transport is decided here, once, for the whole batch:
    // chunk offsets are multiples of 1,024 envs, so every chunk keeps the batch's alignment, and the fold rule below keeps
    // every chunk at one tile or more.  Not eligible (a buffer that is not mapped, fewer envs than a tile, the register
    // kernel selected): the copy transport below runs instead.
    // With final outputs the step leaves its flags on the device, where the pass reads them; the pass writes them, and
    // `finished`, to the host (zflags).
    DexsimStepIO zio = *io;
    bool zc = false;
    FinishHost zflags = {};
    if ((flags & DEXSIM_HOST_ZERO_COPY) && (flags & DEXSIM_HOST_PACKED_CONTACTS) && h_obs) {
        zio.host_static_rows = static_cast<float*>(mapped_alias(h_obs));
        zio.reward = static_cast<float*>(mapped_alias(h_reward));
        zflags.terminated = static_cast<uint8_t*>(mapped_alias(h_terminated));
        zflags.truncated = static_cast<uint8_t*>(mapped_alias(h_truncated));
        zflags.num_contacts = h_num_contacts ? static_cast<uint8_t*>(mapped_alias(h_num_contacts)) : nullptr;
        zio.host_cmask = static_cast<uint8_t*>(mapped_alias(h_contact_mask));
        zio.flags |= DEXSIM_STEP_HOST_ALL_ROWS;
        if (final) {
            zflags.finished = static_cast<uint8_t*>(mapped_alias(h_finished));
        } else {
            zio.terminated = zflags.terminated; zio.truncated = zflags.truncated;
            if (h_num_contacts) zio.num_contacts = zflags.num_contacts;
        }
        zc = zio.host_static_rows && zio.reward && zflags.terminated && zflags.truncated &&
             (h_num_contacts ? zflags.num_contacts : io->num_contacts) && zio.host_cmask && (!final || zflags.finished) &&
             pipeline_eligible(*st, zio, step_track(*st, *p, zio), step_extra_io(zio), /*single=*/false);
    }
    // chunk boundaries are multiples of 1024 envs (tile- and alignment-friendly)
    if (chunks > HOST_MAX_CHUNKS) chunks = HOST_MAX_CHUNKS;
    int64_t per = ((n + (chunks > 0 ? chunks : 1) - 1) / (chunks > 0 ? chunks : 1) + 1023) / 1024 * 1024;
    int nchunks = (int)((n + per - 1) / per);
    // a last chunk below one tile would not run on the pipelined kernel: the zero-copy transport folds it into its neighbour
    if (zc && nchunks > 1 && n - (int64_t)(nchunks - 1) * per < TILE) nchunks -= 1;
    auto chunk_hi = [&](int c) -> int64_t { return c == nchunks - 1 ? n : (int64_t)(c + 1) * per; };
    HostPipe* hp = nullptr;
    int dev = 0;
    bool tracing = host_trace() && nchunks > 1 && !zc && h_obs && !(flags & DEXSIM_HOST_ASYNC) &&
                   (g_trace_calls.fetch_add(1, std::memory_order_relaxed) % 10 == 9);
    if (tracing) {
        int tdev = -1;
        tracing = cudaGetDevice(&tdev) == cudaSuccess && g_trace.make(tdev);
    }
    // A device's internal streams and events are shared by every caller on that device: enqueue one step at a time
    // per device (callers driving different GPUs from different host threads do not wait for each other).
    std::unique_lock<std::mutex> enqueue_lock;
    if (nchunks > 1) {
        rc = get_pipe(&hp);
        if (rc) return rc;
        cudaError_t err = cudaGetDevice(&dev);
        if (err != cudaSuccess) return -(int)err;
        enqueue_lock = std::unique_lock<std::mutex>(g_enqueue_mutex[dev & 63]);
        err = cudaEventRecord(hp->fork_ev, user);
        if (err != cudaSuccess) return -(int)err;
        if (tracing) cudaEventRecord(g_trace.t0, user);
        for (int k = 0; k < HOST_STREAMS && k < nchunks; ++k) {
            err = cudaStreamWaitEvent(hp->streams[k], hp->fork_ev, 0);
            if (err != cudaSuccess) return -(int)err;
        }
    }
    // observation rows that travel: all 45, or without the constant quaternion rows 33-36 (SKIP_QUAT), and without the
    // five 0/1 contact rows 40-44 when the 1-byte contact mask is sent instead (PACKED_CONTACTS)
    const int rows_hi = (flags & DEXSIM_HOST_PACKED_CONTACTS) ? DEXSIM_ROW_CONTACT : DEXSIM_OBS;
    bool expand_on_host = (flags & DEXSIM_HOST_EXPAND_CONTACTS) && (flags & DEXSIM_HOST_PACKED_CONTACTS) &&
                          !(flags & DEXSIM_HOST_ASYNC) && h_obs != nullptr;
    // Rows 30, 31, 37, 38 (object x, y and their velocities) only change when an episode is reset.  When h_obs is mapped
    // page-locked memory the step kernel mirrors every such change straight into it (DexsimStepIO.host_static_rows), and a
    // caller whose buffer is already current (DEXSIM_HOST_STATIC_ROWS) does not download those rows at all.
    float* mirror = io->host_static_rows ? nullptr : static_cast<float*>(mapped_alias(h_obs));
    const bool skip_static = (flags & DEXSIM_HOST_STATIC_ROWS) && mirror != nullptr && (flags & DEXSIM_HOST_SKIP_QUAT);
    // Whatever happens while enqueueing, the caller's stream is joined with the internal ones before returning,
    // so that no copy is still in flight on a stream the caller cannot see.
    auto copy_vectors = [&](cudaStream_t s, int64_t lo, int64_t m) -> int {
        cudaError_t err = cudaMemcpyAsync(h_reward + lo, io->reward + lo, (size_t)m * sizeof(float), cudaMemcpyDeviceToHost, s);
        if (err != cudaSuccess) return -(int)err;
        err = cudaMemcpyAsync(h_terminated + lo, io->terminated + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
        if (err != cudaSuccess) return -(int)err;
        err = cudaMemcpyAsync(h_truncated + lo, io->truncated + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
        if (err != cudaSuccess) return -(int)err;
        if (h_num_contacts) {
            err = cudaMemcpyAsync(h_num_contacts + lo, io->num_contacts + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
            if (err != cudaSuccess) return -(int)err;
        }
        if (h_contact_mask && !(expand_on_host && nchunks > 1)) {        // (1 byte per env: sent whenever the caller has room for it)
            err = cudaMemcpyAsync(h_contact_mask + lo, st->cmask + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
            if (err != cudaSuccess) return -(int)err;
        }
        if (final) {
            err = cudaMemcpyAsync(h_finished + lo, io->finished + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
            if (err != cudaSuccess) return -(int)err;
        }
        return 0;
    };
    for (int c = 0; c < nchunks && rc == 0; ++c) {
        const int64_t lo = (int64_t)c * per, hi = chunk_hi(c), m = hi - lo;
        cudaStream_t s = nchunks > 1 ? hp->streams[c % HOST_STREAMS] : user;
        DexsimState sub = *st;
        sub.n = m;
        sub.obs += lo; sub.op64 += lo; sub.thr += lo; sub.damp += lo; sub.step_count += lo; sub.cmask += lo;
        sub.size += lo; sub.mass += lo; sub.friction += lo; sub.episode += lo;
        if (sub.ep_return) sub.ep_return += lo;
        if (sub.ep_stats) sub.ep_stats += lo;
        DexsimParams sp = *p;
        sp.env_gid0 = p->env_gid0 + lo;
        DexsimStepIO sio = zc ? zio : *io;
        float* d_action = const_cast<float*>(io->action) + (aos ? lo * NJ : lo);
        sio.action = d_action;
        sio.reward += lo; sio.terminated += lo; sio.truncated += lo; sio.num_contacts += lo;
        if (sio.reward_comps) sio.reward_comps += lo;
        if (sio.reward64) sio.reward64 += lo;
        if (sio.finished) sio.finished += lo;
        if (sio.sched) sio.sched = (2 * (c + 1) + 1 < DEXSIM_SCHED_WORDS) ? io->sched + 2 * (c + 1) : nullptr;   // chunks run concurrently
        if (zc) { sio.host_static_rows = zio.host_static_rows + lo; if (sio.host_cmask) sio.host_cmask += lo; }
        else if (mirror) sio.host_static_rows = mirror + lo;
        cudaError_t err;
        if (aos) err = cudaMemcpyAsync(d_action, h_action + lo * NJ, (size_t)m * NJ * sizeof(float), cudaMemcpyHostToDevice, s);
        else err = cudaMemcpy2DAsync(d_action, (size_t)ld * 4, h_action + lo, (size_t)ld * 4, (size_t)m * 4, NJ, cudaMemcpyHostToDevice, s);
        if (err != cudaSuccess) { rc = -(int)err; break; }
        if (tracing) cudaEventRecord(g_trace.up[c], s);
        const uint16_t* goe = group_of_env ? group_of_env + lo : nullptr;
        if (!final) {
            rc = launch_step(&sub, &sp, groups, goe, &sio, s);
        } else {
            FinishHost hf = {};
            hf.final_obs = d_final + lo * NOBS;
            hf.obs = sio.host_static_rows;
            if (zc) {
                hf.zero_copy = 1;
                hf.cmask = sio.host_cmask;
                hf.terminated = zflags.terminated + lo; hf.truncated = zflags.truncated + lo; hf.finished = zflags.finished + lo;
                hf.num_contacts = zflags.num_contacts ? zflags.num_contacts + lo : nullptr;
            }
            rc = step_then_finish_reset<true>(sub, sp, groups, goe, sio, nullptr, hf, s);
        }
        if (rc) break;
        if (tracing) cudaEventRecord(g_trace.k[c], s);
        if (zc) {                                        // every result is already on its way to the host buffers
            if (nchunks > 1) rc = cuda_rc(cudaEventRecord(hp->kdone[c], s));
            continue;
        }
        if (nchunks > 1) {
            if (expand_on_host) {                        // the chunk's contact masks first: the host expands them while its rows travel
                err = cudaMemcpyAsync(h_contact_mask + lo, st->cmask + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
                if (err != cudaSuccess) { rc = -(int)err; break; }
            }
            err = cudaEventRecord(hp->kdone[c], s);      // this chunk's kernel has run: its per-env vectors are final
            if (err != cudaSuccess) { rc = -(int)err; break; }
        }
        if (h_obs) {
            auto rows = [&](int r0, int r1) -> cudaError_t {       // observation rows [r0, r1) of this chunk
                return cudaMemcpy2DAsync(h_obs + (size_t)r0 * ld + lo, (size_t)ld * 4, st->obs + (size_t)r0 * ld + lo, (size_t)ld * 4,
                                         (size_t)m * 4, r1 - r0, cudaMemcpyDeviceToHost, s);
            };
            if (skip_static) {                       // joints, z, vz (+ contacts): x, y, vx, vy are mirrored by the kernel
                err = rows(0, DEXSIM_ROW_OP);
                if (err == cudaSuccess && rows_hi == DEXSIM_ROW_CONTACT) {
                    // object z (row 32) and its velocity (row 39) in ONE pitched copy: both sit 7 rows apart on either side
                    // (every copy costs the DMA engine a fixed hand-over time, so fewer copies per chunk matter)
                    constexpr int zr = DEXSIM_ROW_OP + 2, gap = (DEXSIM_ROW_OV + 2) - (DEXSIM_ROW_OP + 2);
                    err = cudaMemcpy2DAsync(h_obs + (size_t)zr * ld + lo, (size_t)gap * ld * 4, st->obs + (size_t)zr * ld + lo,
                                            (size_t)gap * ld * 4, (size_t)m * 4, 2, cudaMemcpyDeviceToHost, s);
                } else {
                    if (err == cudaSuccess) err = rows(DEXSIM_ROW_OP + 2, DEXSIM_ROW_QUAT);
                    if (err == cudaSuccess) err = rows(DEXSIM_ROW_OV + 2, rows_hi);
                }
            } else if (flags & DEXSIM_HOST_SKIP_QUAT) {     // rows 33-36 are the constant (1,0,0,0): caller keeps them
                err = rows(0, DEXSIM_ROW_QUAT);
                if (err == cudaSuccess) err = rows(DEXSIM_ROW_OV, rows_hi);
            } else {
                err = cudaMemcpy2DAsync(h_obs + lo, (size_t)ld * 4, st->obs + lo, (size_t)ld * 4, (size_t)m * 4, rows_hi,
                                        cudaMemcpyDeviceToHost, s);
            }
            if (err != cudaSuccess) { rc = -(int)err; break; }
            if (tracing) cudaEventRecord(g_trace.down[c], s);
        }
        if (nchunks == 1) rc = copy_vectors(s, 0, n);
    }
    if (rc == 0 && nchunks > 1 && !zc) {
        // reward / flags of the whole batch in one copy per vector (5 copies instead of 5 per chunk: every copy costs
        // the DMA engine a few microseconds whatever its size), on their own stream once every chunk's kernel has run --
        // the kernels finish long before the observation downloads do, so these ride along with them
        for (int c = 0; c < nchunks && rc == 0; ++c) rc = cuda_rc(cudaStreamWaitEvent(hp->small, hp->kdone[c], 0));
        if (rc == 0) rc = copy_vectors(hp->small, 0, n);
        if (rc == 0 && tracing) cudaEventRecord(g_trace.small, hp->small);
    }
    if (zc && rc == 0) g_zero_copy_steps.fetch_add(1, std::memory_order_relaxed);
    if (nchunks > 1) {
        for (int k = 0; k < HOST_STREAMS && k < nchunks; ++k) {
            cudaError_t err = cudaEventRecord(hp->join_ev[k], hp->streams[k]);
            if (err == cudaSuccess) err = cudaStreamWaitEvent(user, hp->join_ev[k], 0);
            if (err != cudaSuccess && rc == 0) rc = -(int)err;
        }
        cudaError_t err = cudaEventRecord(hp->join_ev[HOST_STREAMS], hp->small);
        if (err == cudaSuccess) err = cudaStreamWaitEvent(user, hp->join_ev[HOST_STREAMS], 0);
        if (err != cudaSuccess && rc == 0) rc = -(int)err;
        enqueue_lock.unlock();
    }
    if ((flags & DEXSIM_HOST_ASYNC) && rc == 0) return 0;          // the caller synchronizes `stream` before reading
    if (rc == 0 && expand_on_host) {
        // A chunk's 1-byte contact masks reach the host right after its kernel, before its observation rows: this thread
        // writes the five 0/1 contact rows chunk by chunk while the DMA engine is still downloading the other 36 rows --
        // 20 of 171 bytes per env never cross PCIe and the observation is complete on return.
        for (int c = 0; c < nchunks && rc == 0; ++c) {
            const int64_t lo = (int64_t)c * per, hi = chunk_hi(c);
            const cudaError_t err = nchunks > 1 ? cudaEventSynchronize(hp->kdone[c]) : cudaStreamSynchronize(user);
            if (err == cudaSuccess) expand_contact_rows_range(h_obs, h_contact_mask, lo, hi, ld);
            else rc = -(int)err;
        }
    }
    const int sync_rc = cuda_rc(cudaStreamSynchronize(user));
    if (tracing && rc == 0 && sync_rc == 0) {
        fprintf(stderr, "dexsim_step_host trace (us after fork; n %lld, %d chunks):\n", (long long)n, nchunks);
        for (int c = 0; c < nchunks; ++c) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, g_trace.t0, g_trace.up[c]); cudaEventElapsedTime(&b, g_trace.t0, g_trace.k[c]);
            cudaEventElapsedTime(&d, g_trace.t0, g_trace.down[c]);
            fprintf(stderr, "  chunk %2d [%8lld, %8lld): upload done %8.1f  kernel done %8.1f  rows down %8.1f\n", c,
                    (long long)((int64_t)c * per), (long long)chunk_hi(c), a * 1e3, b * 1e3, d * 1e3);
        }
        float v = 0;
        cudaEventElapsedTime(&v, g_trace.t0, g_trace.small);
        fprintf(stderr, "  per-env vectors down %8.1f\n", v * 1e3);
    }
    return rc ? rc : sync_rc;
}

int dexsim_step_host(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                     const uint16_t* group_of_env, const DexsimStepIO* io, const float* h_action, float* h_obs,
                     float* h_reward, uint8_t* h_terminated, uint8_t* h_truncated, uint8_t* h_num_contacts,
                     uint8_t* h_contact_mask, int32_t chunks, int32_t flags, void* stream) {
    return step_host_impl(st, p, groups, group_of_env, io, h_action, h_obs, h_reward, h_terminated, h_truncated,
                          h_num_contacts, h_contact_mask, nullptr, nullptr, chunks, flags, stream);
}

int dexsim_step_host_final(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                           const uint16_t* group_of_env, const DexsimStepIO* io, const float* h_action, float* h_obs,
                           float* h_reward, uint8_t* h_terminated, uint8_t* h_truncated, uint8_t* h_num_contacts,
                           uint8_t* h_contact_mask, uint8_t* h_finished, float* h_final_obs, int32_t chunks, int32_t flags,
                           void* stream) {
    const int rc = check_finish_reset(st, p, groups, io, h_finished && h_final_obs);
    if (rc) return rc;
    return step_host_impl(st, p, groups, group_of_env, io, h_action, h_obs, h_reward, h_terminated, h_truncated,
                          h_num_contacts, h_contact_mask, h_finished, h_final_obs, chunks, flags, stream);
}

}  // extern "C"
