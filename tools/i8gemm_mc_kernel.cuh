// EXPERIMENT (developer tool, not part of the library): cluster variant of the int8-sliced tcgen05 GEMM
// (i8gemm_kernel.cuh) in which the A chunk is TMA-multicast.  Correct (tools/i8gemm_test.cu, stages 72 / 74), but 4 %
// SLOWER than the single-CTA kernel at 2 CTAs and 40 % slower at 4 (only 33 clusters of 4 fit the 148 SMs): halving the
// L2 -> SM operand traffic buys nothing, so that traffic is not what bounds the kernel (DESIGN.md section 4.1).
//
// Hypothesis it tested: the single-CTA kernel is bound by the bytes every SM pulls from L2 into shared memory (DESIGN.md section 4.1:
// 72 KB per K-chunk -- 48 KB of A, 24 KB of B -- for 8 wide MMAs; ncu: L2 -> SM at 8.4 TB/s with the tensor pipe 60 %
// busy).  Column tiles of the same row tile read the SAME A chunk.  Here the CS CTAs of a cluster work on CS
// neighbouring column tiles of one row tile: each CTA fetches 1/CS of the A chunk's rows and multicasts it into the
// shared memory of all CS CTAs (`cp.async.bulk.tensor ... .multicast::cluster`), and fetches its own B chunk.  Per CTA
// and K-chunk L2 delivers 48/CS + 24 KB: 48 KB (CS = 2) or 36 KB (CS = 4) instead of 72 KB, for the same MMAs.
//
// Synchronisation: every CTA keeps its own stage ring and barriers.  A stage of a CTA is written by all CS producers,
// so a producer may refill stage s only when ALL CTAs have consumed it: every MMA warp multicasts its
// `tcgen05.commit` to the empty barrier of stage s in all CTAs (arrival count CS).  The full barrier of a stage
// expects the whole stage (its own B + the CS parts of A); bytes that arrive from a peer before the local producer has
// armed the barrier just drive the transaction count negative until it does.  TMEM, the MMA schedule and the
// epilogue are those of the single-CTA kernel (cta_group::1).
#pragma once
#include "i8gemm_kernel.cuh"

namespace sgpr {
namespace i8g {

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

struct ProblemMC {
    CUtensorMap mapAs;    // A operand (as Problem::mapA) with a box of {64 B, BM / CS rows, 1 chunk, 1 slice}
    CUtensorMap mapB;     // as Problem::mapB
    int N, Kpad;
    const double* aux;    // as Problem::aux
};

__device__ __forceinline__ void tma_load_4d_mc(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                               int c3, uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "h"(cta_mask)
        : "memory");
}
// arrive on the barrier at the same offset in every CTA of the mask once all MMAs issued so far have retired
__device__ __forceinline__ void tc_commit_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}

template <int NS, int TR, int STAGES, class Epi, int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(NTHREADS, 1)
    i8gemm_mc_kernel(const Common* __restrict__ cmp, const ProblemMC* __restrict__ probs, Epi epi) {
    static_assert(CS == 2 || CS == 4, "cluster of 2 or 4 CTAs");
    using SC = Scheme<NS, TR>;
    constexpr int AROWS = BM / CS;                  // A rows fetched (and multicast) by one CTA
    constexpr uint16_t kMask = (uint16_t)((1u << CS) - 1u);
    __shared__ Common cm;
    __shared__ int gstart[9];                       // first tile GROUP (CS column tiles of one row tile) of each problem
    if (threadIdx.x < sizeof(Common) / 4) reinterpret_cast<int*>(&cm)[threadIdx.x] = reinterpret_cast<const int*>(cmp)[threadIdx.x];
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = (uint64_t*)(smem + (size_t)STAGES * SC::STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint64_t* tmem_empty = tmem_full + 1;
    uint32_t* tmem_slot = (uint32_t*)(tmem_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int cluster_id = blockIdx.x / CS, n_clusters = gridDim.x / CS;
    constexpr uint32_t tmem_cols = 512;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);        // the local producer (expecting the bytes of the whole stage)
            mbar_init(&empty_bar[s], CS);      // multicast commits of all CS MMA warps
        }
        mbar_init(tmem_full, 1);
        mbar_init(tmem_empty, 8);              // one arrive per epilogue warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, tmem_cols);
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int p = 0; p < 8; ++p) {
            gstart[p] = t;
            if (p < cm.n_prob) {
                const int tiles_n = (probs[p].N + BN - 1) / BN;
                t += ((cm.M[p] + BM - 1) / BM) * ((tiles_n + CS - 1) / CS);
            }
        }
        gstart[8] = t;
    }
    __syncthreads();
    cluster_sync_all();                        // every CTA's barriers are initialised before a peer signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int n_groups = gstart[8];

    auto locate = [&](int gg, int& pi, int& tm, int& tn) {
        pi = 0;
        for (int q = 1; q < cm.n_prob; ++q)
            if (gg >= gstart[q]) pi = q;
        const int g = gg - gstart[pi];
        const int groups_n = ((probs[pi].N + BN - 1) / BN + CS - 1) / CS;
        tm = g / groups_n;
        tn = (g - tm * groups_n) * CS + rank;  // may lie beyond the last column tile: that CTA computes on zeros
    };

    if (warp == 0) {
        // ===================== TMA producer =====================
        int stage = 0;
        uint32_t phase = 0;
        for (int gg = cluster_id; gg < n_groups; gg += n_clusters) {
            int pi, tm, tn;
            locate(gg, pi, tm, tn);
            const ProblemMC& P = probs[pi];
            const int nk = P.Kpad / BKB;
            for (int kt = 0; kt < nk; ++kt) {
                mbar_wait(&empty_bar[stage], phase ^ 1);     // all CTAs of the cluster have consumed this stage
                if (elect_one()) {
                    uint8_t* sa = smem + (size_t)stage * SC::STAGE_BYTES;
                    mbar_expect_tx(&full_bar[stage], SC::STAGE_BYTES);
                    // this CTA's rows of the A chunk, slice by slice ([slice][128 rows][64 B] in every CTA)
#pragma unroll
                    for (int t = 0; t < NS; ++t)
                        tma_load_4d_mc(sa + t * (BM * BKB) + rank * (AROWS * BKB), &P.mapAs, &full_bar[stage], 0,
                                       cm.row0[pi] + tm * BM + rank * AROWS, kt, t, kMask);
                    tma_load_4d(sa + SC::A_BYTES, &P.mapB, &full_bar[stage], 0, tn * BN, kt, 0);
                }
                __syncwarp();
                if (++stage == STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        constexpr MmaPlan<NS, TR> plan{};
        const uint32_t idesc_n[4] = {make_idesc_i8(BM, BN), make_idesc_i8(BM, 2 * BN), make_idesc_i8(BM, 3 * BN),
                                     make_idesc_i8(BM, 4 * BN)};
        const uint64_t desc_hi = make_desc_sw64(0);
        int stage = 0;
        uint32_t phase = 0, tphase = 0;
        for (int gg = cluster_id; gg < n_groups; gg += n_clusters) {
            int pi, tm, tn;
            locate(gg, pi, tm, tn);
            const int nk = probs[pi].Kpad / BKB;
            if (nk == 0) continue;
            mbar_wait(tmem_empty, tphase ^ 1);
            tc_fence_after();
            for (int kt = 0; kt < nk; ++kt) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)stage * SC::STAGE_BYTES);
                const uint64_t adesc = desc_hi | (uint64_t)((sa >> 4) & 0x3FFF);
                const uint64_t bdesc = desc_hi | (uint64_t)(((sa + SC::A_BYTES) >> 4) & 0x3FFF);
                const uint32_t later = kt > 0 ? 1u : 0u;
                if (elect_one()) {
#pragma unroll
                    for (int ks = 0; ks < BKB / 32; ++ks) {
#pragma unroll
                        for (int i = 0; i < plan.n; ++i) {
                            const int t = plan.seg[i].t, u0 = plan.seg[i].u0, nu = plan.seg[i].nu;
                            const uint32_t accum = (ks == 0 && plan.seg[i].fresh) ? later : 1u;
                            mma_i8(tmem_base + (t + u0 - 2) * BN, adesc + (((t - 1) * (BM * BKB) + ks * 32) >> 4),
                                   bdesc + (((u0 - 1) * (BN * BKB) + ks * 32) >> 4), idesc_n[nu - 1], accum);
                        }
                    }
                    tc_commit_mc(&empty_bar[stage], kMask);   // this CTA is done with the stage: tell every producer
                    if (kt == nk - 1) tc_commit(tmem_full);
                }
                __syncwarp();
                if (++stage == STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
            tphase ^= 1;
        }
    } else {
        // ===================== epilogue: warps 2..9 =====================
        const int q = warp & 3, half = (warp - 2) >> 2;
        const int row_in_tile = q * 32 + lane;
        constexpr int HC = BN / 2;
        uint32_t tphase = 0;
        for (int gg = cluster_id; gg < n_groups; gg += n_clusters) {
            int pi, tm, tn;
            locate(gg, pi, tm, tn);
            const ProblemMC& P = probs[pi];
            if (P.Kpad / BKB == 0) continue;
            double v[HC];
            mbar_wait(tmem_full, tphase);
            tc_fence_after();
            const bool live = tn * BN < P.N;           // a CTA past the last column tile has nothing to write
            const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + half * HC;
            if (live) {
#pragma unroll
                for (int cc = 0; cc < HC; cc += 8) combine8<SC::NG>(lane_addr + cc, v + cc);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tmem_empty);
            tphase ^= 1;
            if (live) {
#pragma unroll
                for (int cc = 0; cc < HC; cc += 16)
                    epi(pi, cm.row0[pi], tm * BM + row_in_tile, tn * BN + half * HC + cc, v + cc, cm.M[pi], P.N, P.aux);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                // no CTA leaves while a peer may still signal its barriers
    if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

}  // namespace i8g
}  // namespace sgpr
