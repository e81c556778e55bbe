// dexsim_rollout_split.cuh -- fused rollout for SMALL batches: one env = 5 lanes (one finger each).
//
// With a few thousand envs the one-thread-per-env rollout kernel is latency-bound: ~830 dependent-ish
// instructions per env-step on a single warp per SM sub-partition (2 us per step at 4,096 envs).  Here
// every env is spread over 5 lanes (6 envs per warp, lanes 30/31 idle): each lane integrates its finger's
// 3 joints, draws their actions, evaluates its fingertip's contact test and closure term; the per-env
// aggregates come from warp primitives -- contact mask and count from one __ballot_sync, the minimum
// fingertip distance and the ordered float32 closure sum from 5-lane shuffles.  Object dynamics, reward and
// episode bookkeeping are replicated in the 5 lanes (cheaper than broadcasting).  Same arithmetic, same
// Philox streams, same results bit for bit as rollout_kernel / the oracle; ~3x shorter dependency chain per
// step, 5x more warps to fill the machine.  More total work, so the host uses it only for small batches.
#pragma once

#include "dexsim_core.cuh"

// included by dexsim_kernels.cu after finish_episode() is defined
namespace dexsim {

constexpr int SPLIT_LANES = 5;            // lanes per env == fingers
constexpr int SPLIT_ENVS_PER_WARP = 6;
constexpr int SPLIT_THREADS = 128;

struct SplitRegs {
    float    jp[3], jv[3];                // this lane's finger
    double   op[3];                       // env-level, replicated
    float    ov[3];
    double   thr;
    float    damp;
    int      sc;
    unsigned cmask;
};

// Philox word k (0..14) of a 4-block sequence, for the words 3f..3f+2 this lane needs: they live in at
// most two consecutive blocks, which the lane evaluates itself (no cross-lane traffic).
DEXSIM_D void split_words3(uint64_t seed, uint32_t gid, uint32_t episode, uint32_t step, uint32_t stream, int f,
                           uint32_t* w3) {
    const uint32_t b0 = (uint32_t)(3 * f) >> 2, b1 = (uint32_t)(3 * f + 2) >> 2;
    const U4 A = rng_block(seed, gid, episode, step, stream, b0);
    const U4 B = (b1 != b0) ? rng_block(seed, gid, episode, step, stream, b1) : A;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        const int k = 3 * f + j;
        const U4& src = ((uint32_t)k >> 2) == b0 ? A : B;
        const int c = k & 3;
        w3[j] = c == 0 ? src.x : c == 1 ? src.y : c == 2 ? src.z : src.w;
    }
}

// contact bit + squared distance of this lane's fingertip (same tests as update_contacts)
DEXSIM_D bool split_contact(const SplitRegs& e, double& sq) {
    const double thr2 = __dmul_rn(e.thr, e.thr);
    const double lo2 = __dmul_rn(thr2, 1.0 - 0x1p-50), hi2 = __dmul_rn(thr2, 1.0 + 0x1p-50);
    const float s = __fadd_rn(__fadd_rn(e.jp[0], e.jp[1]), e.jp[2]);
    const double tip = (double)__fmul_rn(s, 0.1f);
    const double dx = __dsub_rn(tip, e.op[0]), dy = __dsub_rn(tip, e.op[1]), dz = __dsub_rn(tip, e.op[2]);
    sq = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    const bool below = sq < lo2, above = sq > hi2;     // branch only for the tie band (see update_contacts)
    bool c = below;
    if (!(below || above)) c = __dsqrt_rn(sq) < e.thr;
    return c && (e.thr > 0.0);
}

template <bool DENSE>
__global__ void __launch_bounds__(SPLIT_THREADS)
rollout_split_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
                     const uint16_t* __restrict__ group_of_env, const int k_steps, const int policy_kind,
                     const DexsimRolloutIO rio) {
    constexpr unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int f = lane % SPLIT_LANES;
    const int el = lane / SPLIT_LANES;                       // 0..5 real groups, 6 = idle lanes 30, 31
    const int base = el * SPLIT_LANES;
    const int64_t n = st.n, ld = st.ld;
    int64_t i = warp * SPLIT_ENVS_PER_WARP + el;
    const bool active = el < SPLIT_ENVS_PER_WARP && i < n;   // idle lanes shadow a valid env and never write
    if (i >= n) i = n - 1;
    const bool leader = active && f == 0;

    const int64_t gid64 = p.env_gid0 + i;
    const uint32_t gid = (uint32_t)gid64;
    const int g = group_index(group_of_env, i, gid64, p.num_groups);
    const DexsimGroup& grp = groups[g];                      // read only at resets
    unsigned long long* cnt = rio.counters ? reinterpret_cast<unsigned long long*>(rio.counters) + (int64_t)g * DEXSIM_NCOUNTERS : nullptr;
    double* rs = (rio.ret_sums && rio.counters) ? rio.ret_sums + 2 * g : nullptr;

    SplitRegs e;
    const float* __restrict__ obs = st.obs;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        e.jp[j] = obs[(DEXSIM_ROW_JP + 3 * f + j) * ld + i];
        e.jv[j] = obs[(DEXSIM_ROW_JV + 3 * f + j) * ld + i];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { e.op[k] = st.op64[k * ld + i]; e.ov[k] = obs[(DEXSIM_ROW_OV + k) * ld + i]; }
    e.thr = st.thr[i]; e.damp = st.damp[i]; e.sc = st.step_count[i]; e.cmask = st.cmask[i];
    uint32_t episode = st.episode[i];
    double ep_return = st.ep_return[i];
    EpStats es{st.ep_stats[i], st.ep_stats[ld + i]};
    double size = st.size[i], mass = st.mass[i], friction = st.friction[i];
    bool params_dirty = false;
    bool stopped = false;                                    // one-episode mode: this env is done for the launch

    for (int t = 0; t < k_steps; ++t) {
        // ---- policy (policies/random_policy.py:40, policies/heuristic_policy.py:55-62), this finger's 3 joints
        uint32_t w3[3];
        split_words3(p.seed, gid, episode, (uint32_t)e.sc, STREAM_POLICY, f, w3);
        float a[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) a[j] = __fmaf_rn((float)(w3[j] >> 8), 0x1p-23f, -1.0f);
        if (policy_kind == DEXSIM_POLICY_HEURISTIC) {
#pragma unroll
            for (int j = 0; j < 3; ++j) a[j] = clip_f32(__fadd_rn(-0.5f, __fmul_rn(a[j], 0.1f)), -1.0f, 1.0f);
        }
        const int sc_before = e.sc;
        SplitRegs prev_state = e;                            // restored for envs that already stopped
        // ---- joints, envs/manipulation_env.py:199-207
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            e.jv[j] = __fadd_rn(__fmul_rn(0.9f, e.jv[j]), __fmul_rn(0.1f, a[j]));
            e.jp[j] = clip_f32(__fadd_rn(e.jp[j], __fmul_rn(e.jv[j], 0.01f)), -1.0f, 1.0f);
        }
        // ---- object, :211-235 (replicated in the 5 lanes of the env)
        constexpr double kGravZ = -9.81 * 0.01;
        e.ov[0] = (float)__dadd_rn((double)__fmul_rn(e.ov[0], e.damp), 0.0);
        e.ov[1] = (float)__dadd_rn((double)__fmul_rn(e.ov[1], e.damp), 0.0);
        e.ov[2] = (float)__dadd_rn((double)__fmul_rn(e.ov[2], e.damp), kGravZ);
        const bool first = (e.sc == 0);
        const double lo[3] = {-0.2, -0.2, 0.0};
        const double hi[3] = {0.2, 0.2, 0.3};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float dq = __fmul_rn(e.ov[k], 0.01f);
            const double p32 = (double)__fadd_rn((float)e.op[k], dq);
            const double p64 = __dadd_rn(e.op[k], (double)dq);
            e.op[k] = clip_f64(first ? p32 : p64, lo[k], hi[k]);
            if ((e.op[k] <= lo[k] && e.ov[k] < 0.0f) || (e.op[k] >= hi[k] && e.ov[k] > 0.0f)) e.ov[k] = 0.0f;
        }
        // ---- contacts, :285-310: one fingertip per lane, aggregates by warp primitives
        double sq;
        const bool c = split_contact(e, sq);
        const unsigned ballot = __ballot_sync(FULL, c);
        const unsigned prev_mask = e.cmask;
        e.cmask = (ballot >> base) & 31u;
        const int n_c = __popc(e.cmask);
        double total = 0.0;
        if (DENSE) {
            double sqmin = 0.0;
            float msum = -0.0f;
            float cs = -0.0f;
#pragma unroll
            for (int j = 0; j < 3; ++j) cs = __fadd_rn(cs, fminf(e.jp[j], 0.0f));
            cs = -cs;
#pragma unroll
            for (int k = 0; k < SPLIT_LANES; ++k) {          // finger order, like the reference's Python loops
                const double v = __shfl_sync(FULL, sq, base + k);
                sqmin = (k == 0) ? v : ((v < sqmin || v != v) ? v : sqmin);
                msum = __fadd_rn(msum, __shfl_sync(FULL, cs, base + k));
            }
            const double distance = exp(__dmul_rn(-5.0, __dsqrt_rn(sqmin)));
            const double contact = kContactReward[n_c];
            const double closure = (double)clip_f32(__fdiv_rn(__fdiv_rn(msum, 5.0f), 5.0f), 0.0f, 1.0f);
            const double stability = first ? 0.0 : (double)kStabilityReward[__popc((prev_mask ^ e.cmask) & 31u)];
            total = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(p.w_distance, distance), __dmul_rn(p.w_contact, contact)),
                                        __dmul_rn(p.w_closure, closure)), __dmul_rn(p.w_stability, stability));
        } else {
            total = (n_c >= 3) ? 1.0 : -0.01;
        }
        const bool terminated = n_c >= p.success_threshold;
        const bool truncated = sc_before >= p.max_episode_steps;
        e.sc = sc_before + 1;
        if (stopped) {                                       // shuffles above still ran warp-wide; discard the step
            e = prev_state;
        } else {
            ep_return = __dadd_rn(ep_return, total);
            epstats_push(es, e.sc - 1, n_c);
            if (leader && rio.hist && rio.step_base + t < rio.hist_steps) rio.hist[(rio.step_base + t) * ld + i] = (uint8_t)n_c;
        }
        const bool done = !stopped && (terminated || truncated || (p.loop_max_steps > 0 && e.sc >= p.loop_max_steps));
        if (done) {
            if (leader) {
                EnvRegs tmp;                                 // finish_episode only reads the step count
                tmp.sc = e.sc;
                EpisodeLog log;
                log.rec = rio.ep_log; log.count = reinterpret_cast<unsigned long long*>(rio.ep_log_count);
                log.capacity = rio.ep_log_capacity; log.t_end = (uint32_t)(rio.step_base + t);
                finish_episode(tmp, p, gid, episode, ep_return, es, terminated, n_c, cnt, rs, &log);
            }
            if (rio.one_episode) {
                stopped = true;
            } else {
                // envs/manipulation_env.py:124-182 with the Philox draws of reset_draws(); this lane takes its joints
                episode += 1u;
                uint32_t jw[3];
                split_words3(p.seed, gid, episode, 0u, STREAM_RESET, f, jw);
#pragma unroll
                for (int j = 0; j < 3; ++j) {
                    e.jp[j] = (float)__dadd_rn(-0.1, __dmul_rn(0.2, (double)u24(jw[j])));
                    e.jv[j] = 0.0f;
                }
                const U4 o = rng_block(p.seed, gid, episode, 0u, STREAM_RESET, 4u);
                const uint32_t pw[3] = {o.x, o.y, o.z};
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const float pos = (float)lerp_rn(grp.spawn_lo[k], grp.spawn_hi[k], __dmul_rn((double)pw[k], 0x1p-32));
                    e.op[k] = p.respawn ? (double)pos : (double)(float)e.op[k];
                    e.ov[k] = 0.0f;
                }
                size = grp.size; mass = grp.mass; friction = grp.friction;
                if (grp.size_ranged | grp.mass_ranged | grp.fric_ranged) {
                    const U4 ra = rng_block(p.seed, gid, episode, 0u, STREAM_RESET, 5u);
                    const U4 rb = rng_block(p.seed, gid, episode, 0u, STREAM_RESET, 6u);
                    if (grp.size_ranged) size = lerp_rn(grp.size_lo, grp.size_hi, u53(ra.x, ra.y));
                    if (grp.mass_ranged) mass = lerp_rn(grp.mass_lo, grp.mass_hi, u53(ra.z, ra.w));
                    if (grp.fric_ranged) friction = lerp_rn(grp.fric_lo, grp.fric_hi, u53(rb.x, rb.y));
                }
                e.thr = __dmul_rn(size, 1.5);
                e.damp = (float)__dsub_rn(1.0, __dmul_rn(__dmul_rn(friction, 0.1), 0.01));
                e.sc = 0;
                ep_return = 0.0;
                es.w0 = 0u; es.w1 = 0u;
                params_dirty = true;
            }
        }
        // contact flags of freshly reset envs (:176) need the ballot again: warp-uniform branch
        const bool was_reset = done && !rio.one_episode;
        if (__any_sync(FULL, was_reset)) {
            double sq2;
            const bool c2 = split_contact(e, sq2);
            const unsigned b2 = __ballot_sync(FULL, c2);
            if (was_reset) e.cmask = (b2 >> base) & 31u;
        }
        if (rio.one_episode && __all_sync(FULL, stopped || !active)) break;
    }

    if (active) {
        float* __restrict__ wobs = st.obs;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            wobs[(DEXSIM_ROW_JP + 3 * f + j) * ld + i] = e.jp[j];
            wobs[(DEXSIM_ROW_JV + 3 * f + j) * ld + i] = e.jv[j];
        }
        wobs[(DEXSIM_ROW_CONTACT + f) * ld + i] = ((e.cmask >> f) & 1u) ? 1.0f : 0.0f;
        if (f < 3) {                                         // three lanes write the three axes
            wobs[(DEXSIM_ROW_OP + f) * ld + i] = (float)e.op[f];
            wobs[(DEXSIM_ROW_OV + f) * ld + i] = e.ov[f];
            st.op64[f * ld + i] = e.op[f];
        }
        if (leader) {
            wobs[(DEXSIM_ROW_QUAT + 0) * ld + i] = 1.0f; wobs[(DEXSIM_ROW_QUAT + 1) * ld + i] = 0.0f;
            wobs[(DEXSIM_ROW_QUAT + 2) * ld + i] = 0.0f; wobs[(DEXSIM_ROW_QUAT + 3) * ld + i] = 0.0f;
            st.thr[i] = e.thr; st.damp[i] = e.damp; st.step_count[i] = e.sc; st.cmask[i] = (uint8_t)e.cmask;
            st.episode[i] = episode;
            st.ep_return[i] = ep_return;
            st.ep_stats[i] = es.w0; st.ep_stats[ld + i] = es.w1;
            if (params_dirty) { st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction; }
        }
    }
}

}  // namespace dexsim
