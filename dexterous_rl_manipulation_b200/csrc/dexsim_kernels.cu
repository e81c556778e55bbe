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
// No CPU fallback exists: every entry point launches CUDA work or returns an error code.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>

#include "dexsim_core.cuh"

namespace dexsim {

#ifndef DEXSIM_STEP_MIN_BLOCKS
#define DEXSIM_STEP_MIN_BLOCKS 2
#endif
constexpr int STEP_THREADS = 256;
#ifndef DEXSIM_PDL_DEFAULT
#define DEXSIM_PDL_DEFAULT(n) 1      // measured on B200 (tools/time_small.py): 14.3 -> 12.1 us at 131,072 envs, 70.0 -> 67.7 us at 1 Mi
#endif

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
template <bool DENSE, bool AOS, bool EXTRAS>
__global__ void __launch_bounds__(STEP_THREADS, DEXSIM_STEP_MIN_BLOCKS)
step_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
            const uint16_t* __restrict__ group_of_env, const DexsimStepIO io,
            double* __restrict__ pack_out = nullptr, const double pack_tag = 0.0) {
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
        } else if (fused_dyn) {
            const float sigma = io.sigma_dyn > 0.0f ? io.sigma_dyn : groups[g].sigma_dyn;
            if (sigma > 0.0f) {
                float nz[NJ];
                normal_rows<NJ>(p.seed, (uint32_t)gid, episode, (uint32_t)e.sc, STREAM_DYN, sigma, nz);
#pragma unroll
                for (int j = 0; j < NJ; ++j) a[j] = clip_f32(__fadd_rn(a[j], nz[j]), -1.0f, 1.0f);
            }
        }

        StepResult r;
        env_step<DENSE>(e, a, p, r);

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
        if (tracking) {
            ep_return = __dadd_rn(st.ep_return[i], r.total);           // evaluator.py:144
            es.w0 = st.ep_stats[i]; es.w1 = st.ep_stats[ld + i];
            epstats_push(es, e.sc - 1, r.n_c);                         // evaluator.py:148-150
        }
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
            finish_and_reset(e, p, groups[g], (uint32_t)gid, episode, ep_return, es, r.terminated, r.n_c,
                             cnt, rs, size, mass, friction, nullptr, /*classify=*/tracking);
            st.episode[i] = episode;
            st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
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

// ---- fused rollout ------------------------------------------------------------------------------------
#ifndef DEXSIM_ROLLOUT_MIN_BLOCKS
#define DEXSIM_ROLLOUT_MIN_BLOCKS 2
#endif
#ifndef DEXSIM_ROLLOUT_THREADS
#define DEXSIM_ROLLOUT_THREADS 256      // CTA shape of the fused rollout for large batches (x MIN_BLOCKS resident CTAs per SM)
#endif
template <bool DENSE, bool LEARNER>
__global__ void __launch_bounds__(DEXSIM_ROLLOUT_THREADS, DEXSIM_ROLLOUT_MIN_BLOCKS)
rollout_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
               const uint16_t* __restrict__ group_of_env, const int k_steps, const int policy_kind,
               const DexsimRolloutIO rio) {
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
            if (LEARNER) {                                 // SimpleLearner.select_action, policies/simple_learner.py:60-69
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
            if (done) {
                if (LEARNER) lbest = -INFINITY;              // policy.reset() before the next episode
                EpisodeLog log;
                log.rec = rio.ep_log; log.count = reinterpret_cast<unsigned long long*>(rio.ep_log_count);
                log.capacity = rio.ep_log_capacity; log.t_end = (uint32_t)(rio.step_base + t);
                if (rio.one_episode) {          // run_episode semantics: stop here, the caller resets
                    finish_episode(e, p, gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs, &log);
                    break;
                }
                finish_and_reset(e, p, grp, gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs,
                                 size, mass, friction, &log);
                params_dirty = true;
            }
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
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d.step_ctas, step_kernel<true, false, false>, STEP_THREADS, 0);
    if (err != cudaSuccess) return -(int)err;
    err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&d.rollout_ctas, rollout_kernel<true, false>, DEXSIM_ROLLOUT_THREADS, 0);
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
static void launch_step_variant(bool extras, int grid, cudaStream_t s, const DexsimState& st, const DexsimParams& p,
                                const DexsimGroup* groups, const uint16_t* goe, const DexsimStepIO& io,
                                double* pack_out, double pack_tag) {
    if (extras) step_kernel<DENSE, AOS, true><<<grid, STEP_THREADS, 0, s>>>(st, p, groups, goe, io, pack_out, pack_tag);
    else        step_kernel<DENSE, AOS, false><<<grid, STEP_THREADS, 0, s>>>(st, p, groups, goe, io);
}

// Programmatic dependent launch of the pipelined step kernel: DEXSIM_PDL=0 never, =1 always, unset = default policy.
static int pdl_choice(int64_t n) {
    static int forced = -2;
    if (forced == -2) {
        const char* e = getenv("DEXSIM_PDL");
        forced = e ? atoi(e) : -1;
    }
    if (forced >= 0) return forced ? 1 : 0;
    return DEXSIM_PDL_DEFAULT(n);
}

// The programmatic edge is kept inside captured graphs as well (DEXSIM_PDL_GRAPH=0 drops it, for experiments): measured on
// B200 with capture_step(steps=8), us per step with / without: 65,536 envs 9.4 / 10.6, 131,072 12.6 / 13.6, 1 Mi 69.2 / 70.0.
// Eager stepping with PDL (9.3 / 12.1 / 67.1) is as fast as a graph replay once the GPU, not the host, is the bound
// (>= 65,536 envs); at 4,096 envs the replay wins (6.5 vs 7.5, the eager loop runs at the host's issue rate).
static bool pdl_in_graphs() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DEXSIM_PDL_GRAPH");
        v = (e && !atoi(e)) ? 0 : 1;
    }
    return v == 1;
}

template <bool DENSE, bool AOS, int TRACK, bool EXTRA, int STAGES, int TILE_>
static int launch_tma_variant(int sm_count, cudaStream_t s, const DexsimState& st, const DexsimParams& p,
                              const DexsimGroup* groups, const uint16_t* goe, const DexsimStepIO& io,
                              const StepMaps& maps, int num_tiles) {
    auto kern = step_tma_kernel<DENSE, AOS, TRACK, EXTRA, STAGES, TILE_>;
    constexpr int TMA_THREADS = TILE_ + 32;            // one compute thread per env of a tile + the producer warp
    const size_t smem = (size_t)STAGES * StageLayout<TILE_>::stage_bytes(TRACK) + 2 * STAGES * (sizeof(uint64_t) + sizeof(int)) +
                        (TRACK ? TMA_GROUPS_MAX * (DEXSIM_NCOUNTERS * sizeof(unsigned long long) + 2 * sizeof(double)) : 0);
    // per template instantiation and per device: the shared-memory opt-in is a per-device function attribute
    static thread_local int occupancy[64] = {0};
    int dev = 0;
    cudaError_t err = cudaGetDevice(&dev);
    if (err != cudaSuccess) return -(int)err;
    int uncached = 0;
    int& ctas_per_sm = (dev >= 0 && dev < 64) ? occupancy[dev] : uncached;
    if (ctas_per_sm == 0) {
        err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return -(int)err;
        err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, kern, TMA_THREADS, smem);
        if (err != cudaSuccess) return -(int)err;
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    int grid = sm_count * ctas_per_sm;
    if (grid > num_tiles) grid = num_tiles;
    // Programmatic dependent launch for back-to-back steps of batches whose step is launch-latency bound: this grid may
    // start (barrier init, counter staging) while the previous step's grid drains and blocks in griddepcontrol.wait
    // until that grid has completed -- stream order is preserved for every access.  All CTAs of a launch are resident
    // at once (grid <= SMs x CTAs per SM), so a waiting grid can never keep its predecessor's CTAs off the SMs.
    int pdl = pdl_choice(st.n);
    if (pdl && !pdl_in_graphs()) {
        // inside a stream capture the kernel nodes of consecutive steps already launch back to back
        cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
        if (cudaStreamIsCapturing(s, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) pdl = 0;
    }
    if (pdl) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(TMA_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        return cuda_rc(cudaLaunchKernelEx(&cfg, kern, st, p, groups, goe, io, maps, num_tiles, pdl));
    }
    kern<<<grid, TMA_THREADS, smem, s>>>(st, p, groups, goe, io, maps, num_tiles, 0);
    return cuda_rc(cudaGetLastError());
}

// 0 = auto (TMA pipeline when eligible), 1 = register-resident kernel only, 2 = TMA pipeline required.
// Initialised from DEXSIM_STEP_IMPL (v1 | v2), changeable at run time with dexsim_set_step_impl().
static int g_rollout_impl = 0;
static int g_step_impl = -1;
static int step_impl_choice() {
    if (g_step_impl < 0) {
        const char* e = getenv("DEXSIM_STEP_IMPL");
        g_step_impl = (e && !strcmp(e, "v1")) ? 1 : (e && !strcmp(e, "v2")) ? 2 : 0;
    }
    return g_step_impl;
}

// Smallest batch the auto choice sends down the TMA pipeline (DEXSIM_TMA_MIN_ENVS overrides it for experiments).
// Measured on B200 (tools/time_small.py, us per step, register-resident kernel vs pipeline, hard curriculum, 400 steps):
//   without programmatic dependent launch the register-resident kernel won below ~80k envs (65,536 envs, counts:
//   10.2 vs 11.4) -- with it (the default, see pdl_choice) the pipeline's prologue overlaps the previous step's tail:
//   counts:  4,096 envs 7.6 vs 6.3;  16,384 8.4 vs 7.0;  65,536 10.2 vs 9.3;  131,072 15.1 vs 12.0;  196,608 20.2 vs 14.4
//   tracked: 4,096 8.7 vs 7.1;  65,536 11.1 vs 10.7;  131,072 16.8 vs 14.2;  196,608 22.5 vs 17.2
//   plain:   16,384 6.2 vs 4.9;  65,536 6.2 vs 7.0 (both at the ~5 us host issue rate);  131,072 10.3 vs 9.0
// so every batch of at least one tile takes the pipeline.
static int64_t tma_min_envs(int track, bool extra) {
    (void)track; (void)extra;
    static int64_t forced = -2;
    if (forced == -2) {
        const char* e = getenv("DEXSIM_TMA_MIN_ENVS");
        forced = e ? atoll(e) : -1;
    }
    const int64_t v = forced >= 0 ? forced : TILE;
    return v < TILE ? TILE : v;
}

// Tile width of the pipelined kernel: 0 = auto, 1 = narrow (128 envs, three CTAs of four compute warps per SM) only,
// 2 = wide (224 envs, two CTAs of seven compute warps per SM) wherever it exists.  Initialised from DEXSIM_STEP_TILE
// (narrow | wide), changeable at run time with dexsim_set_step_tile().  Identical results either way.
static int g_step_tile = -1;
static int step_tile_choice() {
    if (g_step_tile < 0) {
        const char* e = getenv("DEXSIM_STEP_TILE");
        g_step_tile = (e && !strcmp(e, "narrow")) ? 1 : (e && !strcmp(e, "wide")) ? 2 : 0;
    }
    return g_step_tile;
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
    const int choice = step_tile_choice();
    if (choice) return choice == 2;
    if (n >= (int64_t)1 << 18) return false;
    // tiles per resident CTA, rounded up -- a handful of CTAs with one tile more (5 % of a round) do not count as a round:
    // the dynamic hand-out spreads them over the SMs
    auto depth = [](int64_t tiles, int64_t ctas) { return (int64_t)ceil((double)tiles / (double)ctas - 0.05); };
    const int64_t depth_narrow = depth((n + TILE - 1) / TILE, 3 * (int64_t)sm_count);
    const int64_t depth_wide = depth((n + TILE_WIDE - 1) / TILE_WIDE, 2 * (int64_t)sm_count);
    return depth_wide < depth_narrow;
}

// track: 0 = plain step, 1 = full episode tracking (returns + history summaries -> labels), 2 = counts only
static int launch_step_tma(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups, const uint16_t* goe,
                           const DexsimStepIO* io, cudaStream_t s, int track, bool extra, int sm_count) {
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
    const bool dense = p->reward_type == 1;
#define DEXSIM_TMA_CASE(D, A, T, X)                                                                                 \
    if (dense == D && aos == A && track == T && extra == X)                                                         \
        return launch_tma_variant<D, A, T, X, DEXSIM_TMA_STAGES, TILE>(sm_count, s, *st, *p, groups, goe, *io, maps, num_tiles);
#define DEXSIM_TMA_WIDE_CASE(D, A, T, X)                                                                            \
    if (wide && dense == D && aos == A && track == T && extra == X)                                                 \
        return launch_tma_variant<D, A, T, X, 2, TILE_WIDE>(sm_count, s, *st, *p, groups, goe, *io, maps, num_tiles);
    // wide tile: plain and counts-only steps
    DEXSIM_TMA_WIDE_CASE(true, true, 0, false) DEXSIM_TMA_WIDE_CASE(true, true, 2, false)
    DEXSIM_TMA_WIDE_CASE(true, false, 0, false) DEXSIM_TMA_WIDE_CASE(true, false, 2, false)
    DEXSIM_TMA_WIDE_CASE(false, true, 0, false) DEXSIM_TMA_WIDE_CASE(false, true, 2, false)
    DEXSIM_TMA_WIDE_CASE(false, false, 0, false) DEXSIM_TMA_WIDE_CASE(false, false, 2, false)
    DEXSIM_TMA_WIDE_CASE(true, true, 0, true) DEXSIM_TMA_WIDE_CASE(true, true, 2, true)
    DEXSIM_TMA_WIDE_CASE(false, true, 0, true) DEXSIM_TMA_WIDE_CASE(false, true, 2, true)
    DEXSIM_TMA_CASE(true, true, 0, false) DEXSIM_TMA_CASE(true, true, 1, false) DEXSIM_TMA_CASE(true, true, 2, false)
    DEXSIM_TMA_CASE(true, false, 0, false) DEXSIM_TMA_CASE(true, false, 1, false) DEXSIM_TMA_CASE(true, false, 2, false)
    DEXSIM_TMA_CASE(false, true, 0, false) DEXSIM_TMA_CASE(false, true, 1, false) DEXSIM_TMA_CASE(false, true, 2, false)
    DEXSIM_TMA_CASE(false, false, 0, false) DEXSIM_TMA_CASE(false, false, 1, false) DEXSIM_TMA_CASE(false, false, 2, false)
    // noise / reward components: the reference's [n,15] action layout only (SoA callers take the register kernel)
    DEXSIM_TMA_CASE(true, true, 0, true) DEXSIM_TMA_CASE(true, true, 1, true) DEXSIM_TMA_CASE(true, true, 2, true)
    DEXSIM_TMA_CASE(false, true, 0, true) DEXSIM_TMA_CASE(false, true, 1, true) DEXSIM_TMA_CASE(false, true, 2, true)
#undef DEXSIM_TMA_WIDE_CASE
#undef DEXSIM_TMA_CASE
    return 1;
}

static int launch_step(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                       const uint16_t* goe, const DexsimStepIO* io, cudaStream_t s,
                       double* pack_out = nullptr, double pack_tag = 0.0) {
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
    // TMA pipeline: needs 16-byte aligned bases for everything its bulk copies touch; noise / reward-component /
    // float64-reward calls ride it too (their rows are accessed directly) when the actions are [n,15]
    const int impl = step_impl_choice();
    const bool extra_io = io->dyn_noise || io->obs_noise || io->reward_comps || io->reward64 || fused_dyn || fused_obs;
    const bool tracked = (p && p->auto_reset) || st->ep_return != nullptr || io->finished != nullptr;
    const int track = !tracked ? 0 : (st->ep_return != nullptr ? 1 : 2);
    const bool tma_ok = (!extra_io || io->action_layout == 1) && pack_out == nullptr &&
                        st->n >= TILE && st->n < (int64_t)0x7FFFFF00 &&
                        !(reinterpret_cast<uintptr_t>(io->action) & 15u) && !(reinterpret_cast<uintptr_t>(io->reward) & 15u) &&
                        !(reinterpret_cast<uintptr_t>(st->thr) & 15u) && !(reinterpret_cast<uintptr_t>(st->damp) & 15u) &&
                        !(reinterpret_cast<uintptr_t>(st->step_count) & 15u) && !(reinterpret_cast<uintptr_t>(st->cmask) & 15u) &&
                        !(reinterpret_cast<uintptr_t>(io->terminated) & 15u) && !(reinterpret_cast<uintptr_t>(io->truncated) & 15u) &&
                        !(reinterpret_cast<uintptr_t>(io->num_contacts) & 15u) && !(reinterpret_cast<uintptr_t>(st->episode) & 15u) &&
                        (track != 1 || (!(reinterpret_cast<uintptr_t>(st->ep_return) & 15u) && !(reinterpret_cast<uintptr_t>(st->ep_stats) & 15u))) &&
                        !(reinterpret_cast<uintptr_t>(io->finished) & 15u);
    if (impl != 1 && tma_ok && (impl == 2 || st->n >= tma_min_envs(track, extra_io))) {
        rc = launch_step_tma(st, p, groups, goe, io, s, track, extra_io, di.sm_count);
        if (rc <= 0) return rc;                      // launched (0) or CUDA error (< 0); 1 = not available
    }
    if (impl == 2) return DEXSIM_E_PARAM;            // TMA pipeline was demanded but is not eligible
    if (io->flags & DEXSIM_STEP_HOST_ALL_ROWS) return DEXSIM_E_PARAM;   // only the pipelined kernel mirrors every row
    const int grid = grid_for(st->n, STEP_THREADS, di.step_ctas, di.sm_count);
    const bool dense = p->reward_type == 1, aos = io->action_layout == 1;
    if (dense) { if (aos) launch_step_variant<true, true>(extras, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag);
                 else     launch_step_variant<true, false>(extras, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag); }
    else       { if (aos) launch_step_variant<false, true>(extras, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag);
                 else     launch_step_variant<false, false>(extras, grid, s, *st, *p, groups, goe, *io, pack_out, pack_tag); }
    return cuda_rc(cudaGetLastError());
}

}  // namespace dexsim

namespace dexsim {
// csrc/dexsim_host_expand.cpp: observation rows 40-44 of envs [lo, hi) from their 1-byte contact masks (host code)
void expand_contact_rows_range(float* h_obs, const uint8_t* mask, int64_t lo, int64_t hi, int64_t ld);
}  // namespace dexsim

using namespace dexsim;

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

int dexsim_rollout(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                   const uint16_t* group_of_env, int32_t k_steps, int32_t policy_kind, const DexsimRolloutIO* rio,
                   void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    rc = check_params(p, true, groups, st->ep_return != nullptr);
    if (rc) return rc;
    if (!rio) return DEXSIM_E_NULL;
    if (k_steps < 1) return DEXSIM_E_SIZE;
    if (policy_kind < DEXSIM_POLICY_EXTERNAL || policy_kind > DEXSIM_POLICY_LEARNER) return DEXSIM_E_PARAM;
    if (policy_kind == DEXSIM_POLICY_EXTERNAL && !rio->actions) return DEXSIM_E_NULL;
    if (policy_kind == DEXSIM_POLICY_LEARNER && (!rio->learner_mean || !rio->learner_best)) return DEXSIM_E_NULL;
    if (rio->ret_sums && !rio->counters) return DEXSIM_E_NULL;
    if ((rio->counters || rio->ep_log) && !st->ep_return) return DEXSIM_E_NULL;   // labels need the per-env history summary
    if (rio->ep_log && (!rio->ep_log_count || rio->ep_log_capacity < 0)) return DEXSIM_E_NULL;
    if (rio->hist && rio->hist_steps < 0) return DEXSIM_E_SIZE;
    if (st->n == 0) return 0;
    DeviceInfo di;
    rc = device_info_cached(di);
    if (rc) return rc;
    // Small batches are latency-bound: spread warps over as many SM sub-partitions as possible
    // (4 per SM) by shrinking the CTA; large batches use full 256-thread CTAs.
    const int64_t warps = (st->n + 31) / 32;
    int threads = DEXSIM_ROLLOUT_THREADS;
    while (threads > 32 && warps * 32 / threads < (int64_t)di.sm_count * 4) threads = (threads / 2 + 31) / 32 * 32;
    const int64_t blocks = (st->n + threads - 1) / threads;
    if (blocks > 0x7FFFFFFFll) return DEXSIM_E_SIZE;
    const int G = p->num_groups;
    const size_t smem = G <= SMEM_GROUPS_MAX
        ? (size_t)G * (sizeof(DexsimGroup) + DEXSIM_NCOUNTERS * sizeof(unsigned long long) + 2 * sizeof(double)) : 0;
    cudaStream_t s = (cudaStream_t)stream;
    const bool dense = p->reward_type == 1, learner = policy_kind == DEXSIM_POLICY_LEARNER;
    // small batches with an in-kernel policy: 5 lanes per env (dexsim_rollout_split.cuh); the crossover with the
    // one-thread-per-env kernel was measured between 4k and 16k envs on B200 (DESIGN.md 5.2)
    const bool split_ok = (rio->flags & DEXSIM_ROLLOUT_NO_DYN_NOISE) && !rio->dyn_noise && st->ep_return != nullptr &&
                          (policy_kind == DEXSIM_POLICY_RANDOM || policy_kind == DEXSIM_POLICY_HEURISTIC);
    if (split_ok && g_rollout_impl != 1 && (g_rollout_impl == 2 || st->n <= 8192)) {
        const int64_t warps_needed = (st->n + SPLIT_ENVS_PER_WARP - 1) / SPLIT_ENVS_PER_WARP;
        const int64_t sblocks = (warps_needed * 32 + SPLIT_THREADS - 1) / SPLIT_THREADS;
        if (sblocks > 0x7FFFFFFFll) return DEXSIM_E_SIZE;
        if (dense) rollout_split_kernel<true><<<(int)sblocks, SPLIT_THREADS, 0, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
        else rollout_split_kernel<false><<<(int)sblocks, SPLIT_THREADS, 0, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
    } else if (dense && learner) rollout_kernel<true, true><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
    else if (dense) rollout_kernel<true, false><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
    else if (learner) rollout_kernel<false, true><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
    else rollout_kernel<false, false><<<(int)blocks, threads, smem, s>>>(*st, *p, groups, group_of_env, k_steps, policy_kind, *rio);
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

int dexsim_pack_env(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset, double* out64,
                    void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!io || !out64 || !io->reward || !io->terminated || !io->truncated) return DEXSIM_E_NULL;
    if (index < 0 || index >= st->n) return DEXSIM_E_SIZE;
    pack_env_kernel<false><<<1, 64, 0, (cudaStream_t)stream>>>(*st, *io, index, after_reset ? 1 : 0, out64, 0.0);
    return cuda_rc(cudaGetLastError());
}

int dexsim_pack_env_tagged(const DexsimState* st, const DexsimStepIO* io, int64_t index, int32_t after_reset, double* out64,
                           double tag, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!io || !out64 || !io->reward || !io->terminated || !io->truncated) return DEXSIM_E_NULL;
    if (index < 0 || index >= st->n) return DEXSIM_E_SIZE;
    pack_env_kernel<true><<<1, 64, 0, (cudaStream_t)stream>>>(*st, *io, index, after_reset ? 1 : 0, out64, tag);
    return cuda_rc(cudaGetLastError());
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
    cudaStream_t upload;               // every chunk's action upload, back to back: the uploads run ahead of the downloads
                                       // instead of queueing behind an earlier chunk's download in the same stream
    cudaEvent_t fork_ev;
    cudaEvent_t join_ev[HOST_STREAMS + 2];
    cudaEvent_t kdone[HOST_MAX_CHUNKS];
    cudaEvent_t up_ev[HOST_MAX_CHUNKS];
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
        err = cudaStreamCreateWithFlags(&hp.upload, cudaStreamNonBlocking);
        if (err != cudaSuccess) return -(int)err;
        for (int k = 0; k < HOST_STREAMS + 2; ++k) {
            err = cudaEventCreateWithFlags(&hp.join_ev[k], cudaEventDisableTiming);
            if (err != cudaSuccess) return -(int)err;
        }
        for (int k = 0; k < HOST_MAX_CHUNKS; ++k) {
            err = cudaEventCreateWithFlags(&hp.kdone[k], cudaEventDisableTiming);
            if (err != cudaSuccess) return -(int)err;
            err = cudaEventCreateWithFlags(&hp.up_ev[k], cudaEventDisableTiming);
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

// DEXSIM_HOST_UPLOAD_STREAM=1: all action uploads of a host step on one dedicated stream, running ahead of the downloads
// (experiment; default 0 = each chunk uploads on its own stream, behind the previous download of that stream).
static bool upload_stream_choice() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DEXSIM_HOST_UPLOAD_STREAM");
        v = (e && atoi(e)) ? 1 : 0;
    }
    return v == 1;
}

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

// zero-copy transport: 1 = the step kernel reads the actions from mapped host memory itself (no copy at all),
// 0 = the copy engine uploads them chunk by chunk
static bool zc_kernel_upload() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("DEXSIM_ZC_KERNEL_UPLOAD");
        v = (e && atoi(e)) ? 1 : 0;
    }
    return v == 1;
}

int dexsim_expand_contact_rows(float* h_obs, const uint8_t* h_contact_mask, int64_t n, int64_t ld) {
    if (!h_obs || !h_contact_mask) return DEXSIM_E_NULL;
    if (n < 0 || ld < n) return DEXSIM_E_SIZE;
    expand_contact_rows_range(h_obs, h_contact_mask, 0, n, ld);
    return 0;
}

int64_t dexsim_host_zero_copy_steps(void) { return g_zero_copy_steps.load(std::memory_order_relaxed); }

int dexsim_step_host(const DexsimState* st, const DexsimParams* p, const DexsimGroup* groups,
                     const uint16_t* group_of_env, const DexsimStepIO* io, const float* h_action, float* h_obs,
                     float* h_reward, uint8_t* h_terminated, uint8_t* h_truncated, uint8_t* h_num_contacts,
                     uint8_t* h_contact_mask, int32_t chunks, int32_t flags, void* stream) {
    int rc = check_state(st);
    if (rc) return rc;
    if (!p || !io || !io->action || !h_action || !h_reward || !h_terminated || !h_truncated) return DEXSIM_E_NULL;
    if ((flags & DEXSIM_HOST_PACKED_CONTACTS) && !h_contact_mask) return DEXSIM_E_NULL;
    if (io->dyn_noise || io->obs_noise || io->noisy_obs || io->sigma_dyn != 0.0f || io->sigma_obs != 0.0f)
        return DEXSIM_E_PARAM;   // noise: use dexsim_step
    cudaStream_t user = (cudaStream_t)stream;
    const int64_t n = st->n, ld = st->ld;
    if (n == 0) return 0;
    const bool aos = io->action_layout == 1;
    // Zero-copy transport (DEXSIM_HOST_ZERO_COPY): the pipelined kernel itself writes every result into the caller's mapped
    // page-locked buffers -- the joint rows as a second bulk tensor store per tile, object z, its velocity and the contact
    // mask as three more bulk rows, x / y and their velocities when a reset changes them (h_obs must be current, as for
    // DEXSIM_HOST_STATIC_ROWS) -- so nothing is downloaded by the copy engine: no per-copy hand-over times, no pipeline
    // fill, and the download of a tile starts the moment it is computed.  The contact rows follow from the mask
    // (PACKED_CONTACTS semantics; EXPAND_CONTACTS as below).  The actions either come up chunk by chunk on the copy engine (default:
    // uploads of chunk k+1 overlap the PCIe writes of chunk k's kernel) or are read from host memory by the kernel's own
    // bulk loads (DEXSIM_ZC_KERNEL_UPLOAD=1: no copies at all).  Not eligible (a buffer that is not mapped, fewer envs
    // than a tile, DEXSIM_STEP_IMPL=register): the copy transport below runs instead.
    DexsimStepIO zio = *io;
    bool zc = false;
    if ((flags & DEXSIM_HOST_ZERO_COPY) && (flags & DEXSIM_HOST_PACKED_CONTACTS) && h_obs && n >= TILE) {
        auto alias = [](const void* h) -> void* {
            if (!h) return nullptr;
            cudaPointerAttributes attr;
            if (cudaPointerGetAttributes(&attr, h) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
                return attr.devicePointer;
            (void)cudaGetLastError();
            return nullptr;
        };
        zio.host_static_rows = static_cast<float*>(alias(h_obs));
        zio.reward = static_cast<float*>(alias(h_reward));
        zio.terminated = static_cast<uint8_t*>(alias(h_terminated));
        zio.truncated = static_cast<uint8_t*>(alias(h_truncated));
        if (h_num_contacts) zio.num_contacts = static_cast<uint8_t*>(alias(h_num_contacts));
        zio.host_cmask = static_cast<uint8_t*>(alias(h_contact_mask));
        zio.flags |= DEXSIM_STEP_HOST_ALL_ROWS;
        zc = zio.host_static_rows && zio.reward && zio.terminated && zio.truncated && zio.num_contacts && zio.host_cmask;
        if (zc && zc_kernel_upload()) {
            const float* a = static_cast<const float*>(alias(h_action));
            if (a) { zio.action = a; chunks = 1; }
            else zc = false;
        }
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
        err = cudaStreamWaitEvent(hp->upload, hp->fork_ev, 0);
        if (err != cudaSuccess) return -(int)err;
    }
    // observation rows that travel: all 45, or without the constant quaternion rows 33-36 (SKIP_QUAT), and without the
    // five 0/1 contact rows 40-44 when the 1-byte contact mask is sent instead (PACKED_CONTACTS)
    const int rows_hi = (flags & DEXSIM_HOST_PACKED_CONTACTS) ? DEXSIM_ROW_CONTACT : DEXSIM_OBS;
    bool expand_on_host = (flags & DEXSIM_HOST_EXPAND_CONTACTS) && (flags & DEXSIM_HOST_PACKED_CONTACTS) &&
                          !(flags & DEXSIM_HOST_ASYNC) && h_obs != nullptr;
    // Rows 30, 31, 37, 38 (object x, y and their velocities) only change when an episode is reset.  When h_obs is mapped
    // page-locked memory the step kernel mirrors every such change straight into it (DexsimStepIO.host_static_rows), and a
    // caller whose buffer is already current (DEXSIM_HOST_STATIC_ROWS) does not download those rows at all.
    float* mirror = nullptr;
    if (h_obs && !io->host_static_rows) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, h_obs) == cudaSuccess && attr.type == cudaMemoryTypeHost && attr.devicePointer)
            mirror = static_cast<float*>(attr.devicePointer);
        else
            (void)cudaGetLastError();                 // pageable memory: not an error, just no mirror
    }
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
        return 0;
    };
    auto enqueue_chunks = [&]() -> int {
    for (int c = 0; c < nchunks; ++c) {
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
        const bool kernel_upload = zc && zio.action != io->action;       // the kernel reads the actions from host memory
        float* d_action = const_cast<float*>(io->action) + (aos ? lo * NJ : lo);
        sio.action = kernel_upload ? zio.action + (aos ? lo * NJ : lo) : d_action;
        sio.reward += lo; sio.terminated += lo; sio.truncated += lo; sio.num_contacts += lo;
        if (sio.reward_comps) sio.reward_comps += lo;
        if (sio.reward64) sio.reward64 += lo;
        if (sio.finished) sio.finished += lo;
        if (sio.sched) sio.sched = (2 * (c + 1) + 1 < DEXSIM_SCHED_WORDS) ? io->sched + 2 * (c + 1) : nullptr;   // chunks run concurrently
        if (zc) { sio.host_static_rows = zio.host_static_rows + lo; if (sio.host_cmask) sio.host_cmask += lo; }
        else if (mirror) sio.host_static_rows = mirror + lo;
        cudaError_t err = cudaSuccess;
        cudaStream_t up = (nchunks > 1 && upload_stream_choice()) ? hp->upload : s;
        if (kernel_upload) up = s;
        else if (aos) err = cudaMemcpyAsync(d_action, h_action + lo * NJ, (size_t)m * NJ * sizeof(float), cudaMemcpyHostToDevice, up);
        else err = cudaMemcpy2DAsync(d_action, (size_t)ld * 4, h_action + lo, (size_t)ld * 4, (size_t)m * 4, NJ, cudaMemcpyHostToDevice, up);
        if (err != cudaSuccess) return -(int)err;
        if (up != s) {                                   // the chunk's stream picks up where the upload stream got to
            err = cudaEventRecord(hp->up_ev[c], up);
            if (err == cudaSuccess) err = cudaStreamWaitEvent(s, hp->up_ev[c], 0);
            if (err != cudaSuccess) return -(int)err;
        }
        if (tracing) cudaEventRecord(g_trace.up[c], s);
        rc = launch_step(&sub, &sp, groups, group_of_env ? group_of_env + lo : nullptr, &sio, s);
        if (rc) return rc;
        if (tracing) cudaEventRecord(g_trace.k[c], s);
        if (zc) {                                        // every result is already on its way to the host buffers
            if (nchunks > 1) {
                err = cudaEventRecord(hp->kdone[c], s);
                if (err != cudaSuccess) return -(int)err;
            }
            continue;
        }
        if (nchunks > 1) {
            if (expand_on_host) {                        // the chunk's contact masks first: the host expands them while its rows travel
                err = cudaMemcpyAsync(h_contact_mask + lo, st->cmask + lo, (size_t)m, cudaMemcpyDeviceToHost, s);
                if (err != cudaSuccess) return -(int)err;
            }
            err = cudaEventRecord(hp->kdone[c], s);      // this chunk's kernel has run: its per-env vectors are final
            if (err != cudaSuccess) return -(int)err;
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
            if (err != cudaSuccess) return -(int)err;
            if (tracing) cudaEventRecord(g_trace.down[c], s);
        }
        if (nchunks == 1) {
            rc = copy_vectors(s, 0, n);
            if (rc) return rc;
        }
    }
    if (nchunks > 1 && !zc) {
        // reward / flags of the whole batch in one copy per vector (5 copies instead of 5 per chunk: every copy costs
        // the DMA engine a few microseconds whatever its size), on their own stream once every chunk's kernel has run --
        // the kernels finish long before the observation downloads do, so these ride along with them
        for (int c = 0; c < nchunks; ++c) {
            cudaError_t err = cudaStreamWaitEvent(hp->small, hp->kdone[c], 0);
            if (err != cudaSuccess) return -(int)err;
        }
        rc = copy_vectors(hp->small, 0, n);
        if (rc) return rc;
        if (tracing) cudaEventRecord(g_trace.small, hp->small);
    }
    return 0;
    };
    rc = enqueue_chunks();
    if (zc && rc == DEXSIM_E_PARAM) {
        // the pipelined kernel is not available for this call (nothing has been launched): copy transport
        zc = false;
        rc = enqueue_chunks();
    }
    if (zc && rc == 0) g_zero_copy_steps.fetch_add(1, std::memory_order_relaxed);
    if (nchunks > 1) {
        for (int k = 0; k < HOST_STREAMS && k < nchunks; ++k) {
            cudaError_t err = cudaEventRecord(hp->join_ev[k], hp->streams[k]);
            if (err == cudaSuccess) err = cudaStreamWaitEvent(user, hp->join_ev[k], 0);
            if (err != cudaSuccess && rc == 0) rc = -(int)err;
        }
        {
            cudaError_t err = cudaEventRecord(hp->join_ev[HOST_STREAMS], hp->small);
            if (err == cudaSuccess) err = cudaStreamWaitEvent(user, hp->join_ev[HOST_STREAMS], 0);
            if (err == cudaSuccess) err = cudaEventRecord(hp->join_ev[HOST_STREAMS + 1], hp->upload);
            if (err == cudaSuccess) err = cudaStreamWaitEvent(user, hp->join_ev[HOST_STREAMS + 1], 0);
            if (err != cudaSuccess && rc == 0) rc = -(int)err;
        }
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

}  // extern "C"
