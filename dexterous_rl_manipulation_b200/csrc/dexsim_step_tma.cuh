// dexsim_step_tma.cuh -- the step kernel as a TMA / mbarrier pipeline (sm_100a).
//
// Same arithmetic as step_kernel (dexsim_core.cuh: env_step), different data movement.
// The register-resident version is latency-bound: ~100 scalar LDG/STG per thread, 128 registers,
// 16 warps per SM, DRAM at ~50 % (profiles/r01_step_api.md).  Here a persistent CTA owns a ring of
// shared-memory stages; one producer lane moves whole 128-env tiles with bulk-async copies
//   loads : 2-D tensor-map boxes for the obs rows (jp+jv: 30 x 128 floats, ov: 3 x 128), the float64
//           object position (3 x 128) and SoA actions; 1-D bulk copies for the per-env vectors and
//           for AoS actions (one contiguous 7,680-byte run per tile)
//   stores: the in-place updated jp+jv box, step_count, reward and the three flag vectors
// while four compute warps work out of shared memory (conflict-free: lane == column, and the
// AoS action stride of 15 words is odd).  Latency is hidden by the stage ring, not by occupancy.
// Rows that rarely change (object position, velocity, contact flags) are still written straight
// from registers, and only when they changed.
#pragma once

#include <cuda.h>

#include "dexsim_core.cuh"

// included by dexsim_kernels.cu after finish_and_reset() is defined
namespace dexsim {

#ifndef DEXSIM_TMA_TILE
#define DEXSIM_TMA_TILE 128
#endif
#ifndef DEXSIM_TMA_STAGES
#define DEXSIM_TMA_STAGES 2                        // stages per CTA: 2 (three CTAs per SM) or 3 (two CTAs per SM)
#endif
// Envs per tile.  The narrow tile (128 envs: four compute warps + the producer warp, three CTAs per SM; -DDEXSIM_TMA_TILE=96
// builds 24.7 KB stages, four CTAs per SM) serves every instantiation.  The wide tile (224 envs: seven compute warps +
// the producer warp, two CTAs per SM) puts 14 instead of 12 compute warps on an SM -- the register file (16 warps x 128
// registers) and shared memory (2 CTAs x 2 stages x 54.9 KB) are both full then -- and is used for batches whose step is
// bound by the compute warps' latency, not by HBM (launch_step_tma picks it; measured in profiles/r02_time_tile.txt).
// Its stages only fit without the full-tracking arrays, so TRACK == 1 always takes the narrow tile.
constexpr int TILE = DEXSIM_TMA_TILE;              // narrow tile; also the smallest batch the pipeline takes
constexpr int TILE_WIDE = 224;
static_assert(TILE % 32 == 0 && TILE <= 256, "a tile is a whole number of warps and one TMA box wide");
constexpr int TMA_GROUPS_MAX = 16;     // per-CTA counter staging (keeps 3 CTAs per SM with 2 stages)

// byte offsets inside one stage (all multiples of 128: TMA box destinations need 128-byte alignment)
template <int T>
struct StageLayout {
    static_assert(T % 32 == 0 && T <= 256, "a tile is a whole number of warps and one TMA box wide");
    static constexpr int OFF_JPJV = 0;                         // [30][T] f32, in/out
    static constexpr int OFF_OV = OFF_JPJV + 30 * T * 4;       // [3][T] f32, in
    static constexpr int OFF_OP64 = OFF_OV + 3 * T * 4;        // [3][T] f64, in
    static constexpr int OFF_THR = OFF_OP64 + 3 * T * 8;       // [T] f64, in
    static constexpr int OFF_ACT = OFF_THR + T * 8;            // [T][15] (AoS) or [15][T] (SoA) f32, in
    static constexpr int OFF_DAMP = OFF_ACT + NJ * T * 4;      // [T] f32, in
    static constexpr int OFF_SC = OFF_DAMP + T * 4;            // [T] i32, in/out
    static constexpr int OFF_REWARD = OFF_SC + T * 4;          // [T] f32, out
    static constexpr int OFF_CMASK = OFF_REWARD + T * 4;       // [T] u8, in
    static constexpr int OFF_TERM = OFF_CMASK + T;             // [T] u8, out
    static constexpr int OFF_TRUNC = OFF_TERM + T;             // [T] u8, out
    static constexpr int OFF_NC = OFF_TRUNC + T;               // [T] u8, out
    static constexpr int OFF_FIN = OFF_NC + T;                 // [T] u8, out (auto-reset)
    static constexpr int OFF_EPISODE = OFF_FIN + T;            // [T] u32, in (in-kernel noise / auto-reset: Philox counter word)
    static constexpr int OFF_EPRET = OFF_EPISODE + T * 4;      // [T] f64, in/out  (full tracking only: the last three arrays
    static constexpr int OFF_EPST0 = OFF_EPRET + T * 8;        // [T] u32, in/out   exist in the stages of the TRACK == 1
    static constexpr int OFF_EPST1 = OFF_EPST0 + T * 4;        // [T] u32, in/out   instantiations only)
    // every stage starts 128-byte aligned; without full tracking a stage ends after the episode words
    __host__ __device__ static constexpr int stage_bytes(int track) {
        return ((track == 1 ? OFF_EPST1 + T * 4 : OFF_EPRET) + 127) / 128 * 128;
    }
    static_assert(OFF_OV % 128 == 0 && OFF_OP64 % 128 == 0 && OFF_ACT % 128 == 0, "tensor-map box destinations");
    static_assert(OFF_THR % 16 == 0 && OFF_DAMP % 16 == 0 && OFF_SC % 16 == 0 && OFF_REWARD % 16 == 0 && OFF_CMASK % 16 == 0 &&
                  OFF_TERM % 16 == 0 && OFF_TRUNC % 16 == 0 && OFF_NC % 16 == 0 && OFF_EPRET % 16 == 0 && OFF_EPST0 % 16 == 0 &&
                  OFF_EPST1 % 16 == 0 && OFF_FIN % 16 == 0 && OFF_EPISODE % 16 == 0, "1-D bulk copy destinations");
};

struct StepMaps {             // tensor maps live in kernel parameter space (__grid_constant__)
    CUtensorMap obs_jpjv;     // obs [45, ld] f32, box {128, 30}
    CUtensorMap obs_ov;       // obs [45, ld] f32, box {128, 3}
    CUtensorMap op64;         // op64 [3, ld] f64, box {128, 3}
    CUtensorMap act_soa;      // action [15, ld] f32, box {128, 15} (only valid for layout 0)
    CUtensorMap host_jpjv;    // the caller's mapped host observation [45, ld] f32, box {128, 30} (DEXSIM_STEP_HOST_ALL_ROWS)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int c0, int c1, uint32_t src) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];"
                 ::"l"(map), "r"(c0), "r"(c1), "r"(src) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Columns a 1-D bulk copy of a tile may touch: the tile's envs rounded up to 32 (copy sizes must be multiples
// of 16 bytes, also for the 1-byte arrays).  This never leaves the allocation: every array has ld = round_up(n, 32)
// columns, and sub-states made by dexsim_step_host start at multiples of 1,024 envs of the parent, so
// round_up(offset + n, 32) <= parent ld.  (Bounding by `ld - base` instead is wrong for sub-states, whose `ld`
// is the PARENT's row pitch.)
template <int T>
__device__ __forceinline__ uint32_t tile_cols(int64_t n, int64_t base) {
    const int64_t left = n - base;
    return left >= T ? (uint32_t)T : (uint32_t)((left + 31) & ~(int64_t)31);
}

// (A warp-cooperative episode reset -- the (resetting env, Philox block) pairs of a warp flattened into work items over its
// 32 lanes -- was built and measured in round 2: bit-identical, but slower than the owner-lane reset at every reset rate
// (profiles/r02_reset_coop_vs_owner.txt: 69.4 vs 70.6 us at 0.45 % resets per env-step, 99.2 vs 104.1 us at 6.8 %), so
// the experiment build was dropped; the product resets on the owning lane.)

// DENSE: reward type.  AOS: action layout [n,15].  TRACK: 0 = plain step; 1 = episode tracking (return + history
// summary per env -> failure labels), auto-reset, counters; 2 = auto-reset and counters only (what a curriculum
// needs: episodes, successes, lengths) without the per-env return / history arrays.
// EXTRA: observation / dynamics noise (pre-drawn tensors or Philox normals drawn here), reward components and the
// float64 reward -- CombinedNoiseWrapper.step (evaluation/robustness_tests.py:177-207) on the same pipeline; their
// rows go straight from registers to HBM (coalesced 128-byte row segments per warp), the stage ring is unchanged.
// Tiles are handed out dynamically when the caller supplies DexsimStepIO.sched (two zeroed device words): a CTA's first
// tile is its block index, every further one comes from a global counter.  SMs do not progress at the same rate (ncu,
// round 2: 125k .. 152k active cycles per SM under the static round-robin, the launch lasting as long as the slowest),
// and tiles with episode resets take longer than others; with the counter every SM works until the batch is done.
// NEXT: next-step auto-reset (dexsim_step_next_reset).  An env whose stored state is what a step that ended its episode
// left behind (pending_reset) is reset on its owning lane instead of stepped, and shares the tail below with a stepped
// env; an episode that ends is counted and flagged `finished` but not reset.
template <bool DENSE, bool AOS, int TRACK, bool EXTRA, int STAGES, int TILE_, bool NEXT>
__global__ void __launch_bounds__(TILE_ + 32, (STAGES == 2) ? (TILE_ <= 96 ? 4 : (TILE_ >= 192 ? 2 : 3)) : (STAGES == 1 ? 4 : 2))
step_tma_kernel(const DexsimState st, const DexsimParams p, const DexsimGroup* __restrict__ groups,
                const uint16_t* __restrict__ group_of_env, const DexsimStepIO io,
                const __grid_constant__ StepMaps maps, const int num_tiles, const int pdl) {
    // this instantiation's tile width (shadows the namespace-level narrow width) and stage layout
    constexpr int TILE = TILE_;
    static_assert(TRACK != 1 || TILE_ <= 128, "the full-tracking arrays only fit the narrow tile's stages");
    static_assert(!NEXT || TRACK != 0, "next-step auto-reset needs the episode bookkeeping of TRACK 1 or 2");
    using SL = StageLayout<TILE_>;
    constexpr int OFF_JPJV = SL::OFF_JPJV, OFF_OV = SL::OFF_OV, OFF_OP64 = SL::OFF_OP64, OFF_THR = SL::OFF_THR, OFF_ACT = SL::OFF_ACT,
                  OFF_DAMP = SL::OFF_DAMP, OFF_SC = SL::OFF_SC, OFF_REWARD = SL::OFF_REWARD, OFF_CMASK = SL::OFF_CMASK,
                  OFF_TERM = SL::OFF_TERM, OFF_TRUNC = SL::OFF_TRUNC, OFF_NC = SL::OFF_NC, OFF_FIN = SL::OFF_FIN,
                  OFF_EPISODE = SL::OFF_EPISODE, OFF_EPRET = SL::OFF_EPRET, OFF_EPST0 = SL::OFF_EPST0, OFF_EPST1 = SL::OFF_EPST1;
    (void)OFF_EPRET; (void)OFF_EPST0; (void)OFF_EPST1; (void)OFF_ACT;
    constexpr int STAGE_BYTES = SL::stage_bytes(TRACK);
    constexpr int TMA_COMPUTE_THREADS = TILE;          // one thread per env of a tile
    constexpr int TMA_THREADS = TMA_COMPUTE_THREADS + 32;   // + the producer warp
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* stage_base = smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);      // full[S], out_ready[S]
    int* s_tile = reinterpret_cast<int*>(bars + 2 * STAGES);                         // tile held by each stage, -1 = no more
    unsigned long long* sh_cnt = reinterpret_cast<unsigned long long*>(s_tile + 2 * STAGES);
    double* sh_rs = reinterpret_cast<double*>(sh_cnt + (TRACK ? TMA_GROUPS_MAX * DEXSIM_NCOUNTERS : 0));

    constexpr int PRODUCER_TID = TMA_COMPUTE_THREADS;
    const int tid = threadIdx.x;
    const int64_t n = st.n, ld = st.ld;
    const bool count_episodes = TRACK && p.auto_reset && io.counters != nullptr;
    const bool staged_cnt = count_episodes && p.num_groups <= TMA_GROUPS_MAX;
    // The episode counter (Philox counter word) rides the stage ring whenever the kernel may need it: in-kernel noise reads
    // it every step, and an auto-reset needs it before it can draw anything -- as a dependent load from HBM inside the
    // compute phase it cost every warp with a finishing lane about a microsecond (ncu, 6.7 % resets per env-step:
    // long_scoreboard the top stall of the reset path); 4 B/env-step of extra traffic buy that latency back.
    // zero-copy host step (dexsim_step_host, DEXSIM_HOST_ZERO_COPY): EVERY observation entry that changes is also written
    // into the caller's mapped host observation -- the joint rows by a second bulk tensor store per tile, the rest from
    // registers when they change
    const bool host_all = (io.flags & DEXSIM_STEP_HOST_ALL_ROWS) != 0 && io.host_static_rows != nullptr;
    const bool load_episode = (EXTRA && ((!io.dyn_noise && io.sigma_dyn != 0.0f) || (!io.obs_noise && io.noisy_obs && io.sigma_obs != 0.0f))) ||
                              (TRACK && p.auto_reset);

    if (tid == 0) {
        for (int b = 0; b < STAGES; ++b) mbar_init(smem_u32(&bars[b]), 1);
        for (int b = 0; b < STAGES; ++b) mbar_init(smem_u32(&bars[STAGES + b]), TMA_COMPUTE_THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (TRACK && staged_cnt) {
        for (int w = tid; w < p.num_groups * DEXSIM_NCOUNTERS; w += TMA_THREADS) sh_cnt[w] = 0ull;
        for (int w = tid; w < p.num_groups * 2; w += TMA_THREADS) sh_rs[w] = 0.0;
    }
    __syncthreads();

    // Programmatic dependent launch (only when the host launched this grid with the attribute, see launch_tma_variant):
    // the next step's grid may begin its prologue while this one drains ...
    if (pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tid >= PRODUCER_TID) {
        // ===== producer warp: one lane issues every bulk copy of this CTA =====
        if (tid == PRODUCER_TID) {
            // ... and this grid touches global memory only after the previous grid has completed and flushed
            // (every access of the compute warps is ordered behind the producer's first loads by the stage barriers)
            if (pdl) asm volatile("griddepcontrol.wait;" ::: "memory");
            unsigned int* sched = io.sched;
            auto issue_stores = [&](int s, int tile) {
                const int64_t base = (int64_t)tile * TILE;
                const uint32_t sb = smem_u32(stage_base + (size_t)s * STAGE_BYTES);
                const uint32_t cols = tile_cols<TILE>(n, base);
                tma_store_2d(&maps.obs_jpjv, (int)base, DEXSIM_ROW_JP, sb + OFF_JPJV);
                // zero-copy host step: the same 30 joint rows go straight into the caller's mapped host observation
                // (object z, its velocity and the contact masks follow as three small rows: the compute warps left them in
                // the stage slots of the velocity rows / the mask; x, y and their velocities only change at a reset and are
                // written from registers then)
                if (host_all) {
                    tma_store_2d(&maps.host_jpjv, (int)base, DEXSIM_ROW_JP, sb + OFF_JPJV);
                    bulk_store(io.host_static_rows + (int64_t)(DEXSIM_ROW_OP + 2) * ld + base, sb + OFF_OV, cols * 4);
                    bulk_store(io.host_static_rows + (int64_t)(DEXSIM_ROW_OV + 2) * ld + base, sb + OFF_OV + 2 * TILE * 4, cols * 4);
                    if (io.host_cmask) bulk_store(io.host_cmask + base, sb + OFF_CMASK, cols);
                }
                bulk_store(st.step_count + base, sb + OFF_SC, cols * 4);
                bulk_store(io.reward + base, sb + OFF_REWARD, cols * 4);
                bulk_store(io.terminated + base, sb + OFF_TERM, cols);
                bulk_store(io.truncated + base, sb + OFF_TRUNC, cols);
                bulk_store(io.num_contacts + base, sb + OFF_NC, cols);
                if (TRACK == 1) {
                    bulk_store(st.ep_return + base, sb + OFF_EPRET, cols * 8);
                    bulk_store(st.ep_stats + base, sb + OFF_EPST0, cols * 4);
                    bulk_store(st.ep_stats + ld + base, sb + OFF_EPST1, cols * 4);
                }
                if (TRACK && io.finished) bulk_store(io.finished + base, sb + OFF_FIN, cols);
                bulk_commit();
            };
            unsigned held = 0u;                        // bit s: stage s still holds the outputs of tile s_tile[s]
            // `tile` counts work items 0 .. num_tiles-1 in hand-out order; with DEXSIM_STEP_REVERSE_TILES item t is tile
            // num_tiles-1-t, so that a step starts where the previous one ended (what is still in L2)
            const bool reverse = (io.flags & DEXSIM_STEP_REVERSE_TILES) != 0;
            int tile = (int)blockIdx.x;                // first tile: static
            int k = 0;
            for (;; ++k) {
                const int s = k % STAGES, use = k / STAGES;
                const uint32_t sb = smem_u32(stage_base + (size_t)s * STAGE_BYTES);
                const uint32_t full = smem_u32(&bars[s]);
                if ((held >> s) & 1u) {
                    // the tile that used this stage last: wait for its outputs, send them, and let
                    // the copy engine finish READING the stage before new data lands in it
                    mbar_wait(smem_u32(&bars[STAGES + s]), (uint32_t)((use - 1) & 1));
                    issue_stores(s, s_tile[s]);
                    held &= ~(1u << s);
                    bulk_wait_read0();
                }
                if (tile >= num_tiles) {               // no more work: tell the compute warps and leave
                    s_tile[s] = -1;
                    mbar_arrive(full);
                    break;
                }
                const int tile_id = reverse ? num_tiles - 1 - tile : tile;
                s_tile[s] = tile_id;
                held |= 1u << s;
                const int64_t base = (int64_t)tile_id * TILE;
                const uint32_t cols = tile_cols<TILE>(n, base);
                const bool full_tile = (n - base) >= TILE;
                uint32_t tx = (30 + 3) * TILE * 4 + 3 * TILE * 8 + cols * (8 + 4 + 4 + 1);
                if (AOS) tx += full_tile ? NJ * TILE * 4 : 0;
                else tx += NJ * TILE * 4;
                if (TRACK == 1) tx += cols * (8 + 4 + 4);
                if (load_episode) tx += cols * 4;
                mbar_expect_tx(full, tx);              // release: s_tile[s] is visible to whoever sees this phase complete
                tma_load_2d(sb + OFF_JPJV, &maps.obs_jpjv, (int)base, DEXSIM_ROW_JP, full);
                tma_load_2d(sb + OFF_OV, &maps.obs_ov, (int)base, DEXSIM_ROW_OV, full);
                tma_load_2d(sb + OFF_OP64, &maps.op64, (int)base, 0, full);
                // (an L2 evict-first hint on these streaming loads and on the per-env output stores was measured: no effect)
                if (AOS) { if (full_tile) bulk_load(sb + OFF_ACT, io.action + base * NJ, NJ * TILE * 4, full); }
                else tma_load_2d(sb + OFF_ACT, &maps.act_soa, (int)base, 0, full);
                bulk_load(sb + OFF_THR, st.thr + base, cols * 8, full);
                bulk_load(sb + OFF_DAMP, st.damp + base, cols * 4, full);
                bulk_load(sb + OFF_SC, st.step_count + base, cols * 4, full);
                bulk_load(sb + OFF_CMASK, st.cmask + base, cols, full);
                if (TRACK == 1) {
                    bulk_load(sb + OFF_EPRET, st.ep_return + base, cols * 8, full);
                    bulk_load(sb + OFF_EPST0, st.ep_stats + base, cols * 4, full);
                    bulk_load(sb + OFF_EPST1, st.ep_stats + ld + base, cols * 4, full);
                }
                if (load_episode) bulk_load(sb + OFF_EPISODE, st.episode + base, cols * 4, full);
                // next tile: from the global counter (its round trip overlaps this tile's transfer), else round-robin
                tile = sched ? (int)(atomicAdd(&sched[0], 1u) + gridDim.x) : tile + (int)gridDim.x;
            }
            // drain: outputs of the tiles still held by the other stages, oldest first
            for (int d = 1; d < STAGES; ++d) {
                const int kk = k - STAGES + d;
                if (kk < 0) continue;
                const int s = kk % STAGES;
                if (!((held >> s) & 1u)) continue;
                mbar_wait(smem_u32(&bars[STAGES + s]), (uint32_t)((kk / STAGES) & 1));
                issue_stores(s, s_tile[s]);
            }
            bulk_wait0();       // shared memory must outlive every outstanding bulk store
            if (sched) {        // the last CTA to finish re-arms the scheduler words for the next launch
                __threadfence();
                if (atomicAdd(&sched[1], 1u) == gridDim.x - 1) { sched[0] = 0u; sched[1] = 0u; }
            }
        }
    } else {
        // ===== compute warps: lane == column of the tile =====
        const int col = tid;
        for (int k = 0;; ++k) {
            const int s = k % STAGES;
            unsigned char* sp = stage_base + (size_t)s * STAGE_BYTES;
            mbar_wait(smem_u32(&bars[s]), (uint32_t)((k / STAGES) & 1));
            const int tile = s_tile[s];
            if (tile < 0) break;
            const int64_t base = (int64_t)tile * TILE;
            const int64_t i = base + col;
            float* s_jpjv = reinterpret_cast<float*>(sp + OFF_JPJV);
            double* s_op = reinterpret_cast<double*>(sp + OFF_OP64);
            float* __restrict__ obs = st.obs;
            const bool valid = i < n;
            bool lane_reset = false;
            bool fused_dyn = false, fused_obs = false;
            uint32_t episode = 0u;
            int g = 0;
            EnvRegs e;
            if (valid) {
                const float* s_ov = reinterpret_cast<const float*>(sp + OFF_OV);
#pragma unroll
                for (int j = 0; j < NJ; ++j) { e.jp[j] = s_jpjv[j * TILE + col]; e.jv[j] = s_jpjv[(NJ + j) * TILE + col]; }
#pragma unroll
                for (int c = 0; c < 3; ++c) { e.ov[c] = s_ov[c * TILE + col]; e.op[c] = s_op[c * TILE + col]; }
                e.thr = reinterpret_cast<const double*>(sp + OFF_THR)[col];
                e.damp = reinterpret_cast<const float*>(sp + OFF_DAMP)[col];
                e.sc = reinterpret_cast<const int*>(sp + OFF_SC)[col];
                e.cmask = reinterpret_cast<const uint8_t*>(sp + OFF_CMASK)[col];
                bool pending = false;
                if constexpr (NEXT) pending = pending_reset(e, p);
                float a[NJ];
                const float* s_act = reinterpret_cast<const float*>(sp + OFF_ACT);
                if (AOS) {
                    if ((n - base) >= TILE) {
#pragma unroll
                        for (int j = 0; j < NJ; ++j) a[j] = s_act[col * NJ + j];
                    } else {        // ragged last tile: its byte count need not be a multiple of 16
#pragma unroll
                        for (int j = 0; j < NJ; ++j) a[j] = __ldg(io.action + i * NJ + j);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < NJ; ++j) a[j] = s_act[j * TILE + col];
                }
                const int64_t gid = p.env_gid0 + i;
                if (EXTRA) {
                    // evaluation/robustness_tests.py:180-187: a <- clip(a + N(0, sigma_dyn), -1, 1)
                    fused_dyn = !io.dyn_noise && io.sigma_dyn != 0.0f;
                    fused_obs = !io.obs_noise && io.noisy_obs && io.sigma_obs != 0.0f;
                    if (fused_dyn || fused_obs) {
                        episode = reinterpret_cast<const uint32_t*>(sp + OFF_EPISODE)[col];
                        if (io.sigma_dyn < 0.0f || io.sigma_obs < 0.0f)
                            g = group_index(group_of_env, i, gid, p.num_groups);
                    }
                    if (io.dyn_noise) {
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
                }
                double op_old[3]; float ov_old[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) { op_old[c] = e.op[c]; ov_old[c] = e.ov[c]; }
                const unsigned cmask_old = e.cmask;

                StepResult r;
                if constexpr (NEXT) {
                    if (pending) {
                        // the reset the previous step left for this env, instead of a step: the action is ignored
                        g = group_index(group_of_env, i, gid, p.num_groups);
                        episode = reinterpret_cast<const uint32_t*>(sp + OFF_EPISODE)[col];     // load_episode is on with auto-reset
                        next_step_reset(e, p, groups[g], (uint32_t)gid, episode, st, i, r);
                        st.thr[i] = e.thr; st.damp[i] = e.damp;
                    } else {
                        env_step<DENSE>(e, a, p, r);
                    }
                } else {
                    env_step<DENSE>(e, a, p, r);
                }

                reinterpret_cast<float*>(sp + OFF_REWARD)[col] = (float)r.total;
                (sp + OFF_TERM)[col] = r.terminated ? 1 : 0;
                (sp + OFF_TRUNC)[col] = r.truncated ? 1 : 0;
                (sp + OFF_NC)[col] = (unsigned char)r.n_c;
                if (EXTRA) {
                    if (io.reward64) io.reward64[i] = r.total;
                    if (io.reward_comps) {
                        io.reward_comps[0 * ld + i] = (float)r.distance;
                        io.reward_comps[1 * ld + i] = (float)r.contact;
                        io.reward_comps[2 * ld + i] = (float)r.closure;
                        io.reward_comps[3 * ld + i] = (float)r.stability;
                    }
                }

                if (TRACK) {
                    double ep_return = 0.0;
                    EpStats es{0u, 0u};
                    if (TRACK == 1 && !pending) {       // a pending env's episode starts now: return and summary stay 0
                        ep_return = __dadd_rn(reinterpret_cast<double*>(sp + OFF_EPRET)[col], r.total);
                        es.w0 = reinterpret_cast<uint32_t*>(sp + OFF_EPST0)[col];
                        es.w1 = reinterpret_cast<uint32_t*>(sp + OFF_EPST1)[col];
                        epstats_push(es, e.sc - 1, r.n_c);
                    }
                    // (never true for a pending env: its reset left step count 0 and both flags 0)
                    const bool done = r.terminated || r.truncated || (p.loop_max_steps > 0 && e.sc >= p.loop_max_steps);
                    if (p.auto_reset && done) {
                        // episode end on the owning lane (counters, labels)
                        g = group_index(group_of_env, i, gid, p.num_groups);
                        episode = reinterpret_cast<const uint32_t*>(sp + OFF_EPISODE)[col];     // load_episode is on with auto-reset
                        unsigned long long* cnt = nullptr;
                        double* rs = nullptr;
                        if (count_episodes) {
                            cnt = (staged_cnt ? sh_cnt : reinterpret_cast<unsigned long long*>(io.counters)) + (int64_t)g * DEXSIM_NCOUNTERS;
                            if (io.ret_sums) rs = (staged_cnt ? sh_rs : io.ret_sums) + 2 * g;
                        }
                        if constexpr (NEXT) {
                            // counted and flagged now, reset by the env's next step
                            finish_episode(e, p, (uint32_t)gid, episode, ep_return, es, r.terminated, r.n_c, cnt, rs, nullptr,
                                           /*classify=*/TRACK == 1);
                            lane_reset = true;
                        } else
                        // the owning lane draws all of its env's Philox blocks (reset_draws + env_reset, dexsim_core.cuh)
                        {
                            double size, mass, friction;
                            finish_and_reset(e, p, groups[g], (uint32_t)gid, episode, ep_return, es, r.terminated, r.n_c,
                                             cnt, rs, size, mass, friction, nullptr, /*classify=*/TRACK == 1);
                            st.episode[i] = episode;
                            st.size[i] = size; st.mass[i] = mass; st.friction[i] = friction;
                            st.thr[i] = e.thr; st.damp[i] = e.damp;
                            lane_reset = true;
                        }
                    }
                    if (TRACK == 1) {
                        reinterpret_cast<double*>(sp + OFF_EPRET)[col] = ep_return;
                        reinterpret_cast<uint32_t*>(sp + OFF_EPST0)[col] = es.w0;
                        reinterpret_cast<uint32_t*>(sp + OFF_EPST1)[col] = es.w1;
                    }
                    (sp + OFF_FIN)[col] = lane_reset ? 1 : 0;
                }
                {
                    // always-changing state goes back through the stage (one bulk store per tile)
#pragma unroll
                    for (int j = 0; j < NJ; ++j) { s_jpjv[j * TILE + col] = e.jp[j]; s_jpjv[(NJ + j) * TILE + col] = e.jv[j]; }
                    reinterpret_cast<int*>(sp + OFF_SC)[col] = e.sc;
                    // rarely-changing rows: straight from registers, only when they changed
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        if (__double_as_longlong(e.op[c]) != __double_as_longlong(op_old[c])) {
                            st.op64[c * ld + i] = e.op[c];
                            obs[(DEXSIM_ROW_OP + c) * ld + i] = (float)e.op[c];
                            // x, y only move when an episode is reset: mirrored into the caller's host observation so that
                            // the end-to-end path need not download those rows every step (DexsimStepIO.host_static_rows)
                            if (c < 2 && io.host_static_rows) io.host_static_rows[(DEXSIM_ROW_OP + c) * ld + i] = (float)e.op[c];
                        }
                        if (__float_as_uint(e.ov[c]) != __float_as_uint(ov_old[c])) {
                            obs[(DEXSIM_ROW_OV + c) * ld + i] = e.ov[c];
                            if (c < 2 && io.host_static_rows) io.host_static_rows[(DEXSIM_ROW_OV + c) * ld + i] = e.ov[c];
                        }
                    }
                    if (host_all) {
                        // zero-copy host step: z, its velocity and the contact mask leave with the tile's bulk stores
                        // (they change too often for 4-byte writes across PCIe); the velocity slots are free by now
                        float* s_out = reinterpret_cast<float*>(sp + OFF_OV);
                        s_out[col] = (float)e.op[2];
                        s_out[2 * TILE + col] = e.ov[2];
                        (sp + OFF_CMASK)[col] = (uint8_t)e.cmask;
                    }
                    const unsigned flip = e.cmask ^ cmask_old;
                    if (flip) {
#pragma unroll
                        for (int f = 0; f < NF; ++f)
                            if ((flip >> f) & 1u) obs[(DEXSIM_ROW_CONTACT + f) * ld + i] = ((e.cmask >> f) & 1u) ? 1.0f : 0.0f;
                        st.cmask[i] = (uint8_t)e.cmask;
                    }
                }
            }
            if (EXTRA && valid && io.noisy_obs) {
                // evaluation/robustness_tests.py:204-205: all 45 entries of the observation AFTER the step (and after a
                // possible auto-reset), rows written straight from registers
                float* __restrict__ out = io.noisy_obs;
                if (io.obs_noise) {
                    const float* __restrict__ nz = io.obs_noise;
#pragma unroll
                    for (int row = 0; row < NOBS; ++row)
                        out[row * ld + i] = __fadd_rn(obs_entry(e, row), __ldg(nz + row * ld + i));
                } else if (fused_obs) {
                    // the same 45 normals dexsim_fill_normal(STREAM_OBS) would produce: one Philox block = four rows
                    const float sigma = io.sigma_obs > 0.0f ? io.sigma_obs : groups[g].sigma_obs;
                    const int64_t gid = p.env_gid0 + i;
#pragma unroll
                    for (int b = 0; b < (NOBS + 3) / 4; ++b) {
                        float z[4];
                        obs_noise_block(p.seed, (uint32_t)gid, episode, (uint32_t)e.sc, b, z);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int row = 4 * b + q;
                            if (row < NOBS) out[row * ld + i] = __fadd_rn(obs_entry(e, row), __fmul_rn(sigma, z[q]));
                        }
                    }
                }
            }
            fence_async_smem();                       // generic-proxy writes -> visible to the copy engine
            mbar_arrive(smem_u32(&bars[STAGES + s]));
        }
    }
    if (TRACK && staged_cnt) {
        __syncthreads();
        unsigned long long* gc = reinterpret_cast<unsigned long long*>(io.counters);
        for (int w = tid; w < p.num_groups * DEXSIM_NCOUNTERS; w += TMA_THREADS)
            if (sh_cnt[w]) atomicAdd(&gc[w], sh_cnt[w]);
        if (io.ret_sums)
            for (int w = tid; w < p.num_groups * 2; w += TMA_THREADS)
                if (sh_rs[w] != 0.0) atomicAdd(&io.ret_sums[w], sh_rs[w]);
    }
}

// ---- host: tensor maps ------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// 2-D row-major [rows, n] view with row pitch ld elements; box = {tile columns, box_rows rows}.
static bool make_map_2d(CUtensorMap* m, CUtensorMapDataType dt, size_t elem, void* base, int64_t n, int64_t ld,
                        int rows, int box_rows, int tile) {
    EncodeTiledFn enc = get_encode_fn();
    if (!enc) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)ld * elem};
    const cuuint32_t box[2] = {(cuuint32_t)tile, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(m, dt, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace dexsim
