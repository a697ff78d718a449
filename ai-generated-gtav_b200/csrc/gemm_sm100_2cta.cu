// bf16 GEMM for sm_100a on CTA PAIRS: out[M,N] = epilogue(A[M,K] @ W[N,K]^T) with tcgen05.mma.cta_group::2.
//
// Same contract, epilogues and rounding points as gemm_sm100.cu (every nn.Linear of the reference at large row
// counts: B >= 8 rollouts, the VAE at N >= 4 frames).  Why a second kernel: a 128 x 256 tile on ONE SM needs
// ~175 GB/s of operand ingest at full tensor rate and a CTA gets ~160 GB/s out of its TMA unit (DESIGN.md 5b), so
// the single-CTA kernel tops out at ~73 % of the MMA rate.  Here two CTAs of a cluster (two SMs of a TPC) share one
// 256 x 256 tile: each loads its own 128 rows of A and only HALF of the W rows (128 of 256), the leader CTA's single
// thread issues UMMA 256 x 256 x 16 that reads both CTAs' shared memory, and each CTA ends up with its own 128 x 256
// accumulator half in its own TMEM - one third less ingest per SM for the same MMA work.
//
// Structure per CTA (416 threads, persistent over tile pairs, double-buffered TMEM accumulator = all 512 columns):
//   warps 0,7: TMA producers of A (this CTA's 128 rows), one 64-wide K chunk each per stage
//   warps 6,8: TMA producers of W (this CTA's half of the 256 weight rows); not gated by the previous kernel (PDL)
//   warp 1   : TMEM allocator (cta_group::2, both CTAs) + in the LEADER the single-thread MMA issuer
//   warps 2-5, 9-12: epilogue of this CTA's 128 rows (tcgen05.ld from its own TMEM, two warps per lane quadrant, half of
//              the 256 columns each), the fused math of epilogue.cuh.  Eight warps because with four a K = 1024 tile's
//              GELU epilogue (~10k issue cycles) outlasts its mainloop (8k cycles): measured 668 TFLOP/s on fc1 whatever
//              the MMA path, against 1089 on the same shape with a plain store.
// Barriers: every TMA load of both CTAs completes its bytes on the LEADER's full barrier (the leader's producers
// post the expected byte count of both CTAs); tcgen05.commit multicasts "slot free" and "accumulator complete" to
// the same barrier in both CTAs; the epilogue warps of both CTAs arrive on the leader's "accumulator drained".
#include "common.cuh"
#include "kernels.h"
#include "epilogue.cuh"

namespace gtav {

static constexpr int G2_BM = 128;              // rows per CTA (256 per pair)
static constexpr int G2_BN = 256;
static constexpr int G2_BK = 64;
static constexpr int G2_KC = 2;                // 64-wide K chunks per stage
static constexpr int G2_STAGES = 3;
static constexpr int G2_THREADS = 416;             // 13 warps: 5 producer / MMA + 8 epilogue
static constexpr int G2_A_CHUNK = G2_BM * G2_BK * 2;           // 16 KB
static constexpr int G2_B_CHUNK = (G2_BN / 2) * G2_BK * 2;     // 16 KB: this CTA's half of the weight rows
static constexpr int G2_STAGE = G2_KC * (G2_A_CHUNK + G2_B_CHUNK);
static constexpr int G2_BAR_OFF = G2_STAGES * G2_STAGE;
static constexpr int G2_SMEM = G2_BAR_OFF + (2 * G2_STAGES + 4) * 8 + 16 + 1024;

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory object in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load issued by either CTA of the pair; the bytes complete on the LEADER's barrier (peer bit of the barrier
// address cleared, as CUTLASS' SM100_TMA_2SM_LOAD does)
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {     // one whole warp in EACH CTA
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                  uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive on the barrier at this shared-memory offset in BOTH CTAs once the MMAs issued so far are complete
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
                 : "memory");
}

template <int EPI>
__global__ void __launch_bounds__(G2_THREADS, 1)
gemm2_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;                                           // [stage][chunk][128 rows][128 B]
    uint8_t* sB = smem + G2_STAGES * G2_KC * G2_A_CHUNK;          // [stage][chunk][128 weight rows][128 B]
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + G2_BAR_OFF);
    uint64_t* empty_bar = full_bar + G2_STAGES;
    uint64_t* tfull_bar = empty_bar + G2_STAGES;       // [2] accumulator complete (multicast to both CTAs)
    uint64_t* tempty_bar = tfull_bar + 2;              // [2] accumulator drained (leader's copy counts both CTAs)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int n_tiles_n = p.N / G2_BN;
    const int n_tiles = n_tiles_n * ((p.M + 2 * G2_BM - 1) / (2 * G2_BM));     // tile pairs of 256 x 256
    const int num_ks = p.K / (G2_KC * G2_BK);
    const int cluster_id = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;

    if (warp == 0 && lane == 0) tma_prefetch_desc(&tmA);
    if (warp == 6 && lane == 0) tma_prefetch_desc(&tmB);
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < G2_STAGES; ++s) {
                mbar_init(&full_bar[s], 2 * G2_KC);   // the leader's four producer threads (they post both CTAs' bytes)
                mbar_init(&empty_bar[s], 1);
            }
            for (int a = 0; a < 2; ++a) {
                mbar_init(&tfull_bar[a], 1);
                mbar_init(&tempty_bar[a], 16);        // one arrival per epilogue warp (8) of both CTAs
            }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc_pair(tmem_slot, 2 * G2_BN);
        tmem_relinquish_pair();
    }
    tcgen05_fence_before();
    cluster_sync_all();                               // barriers and TMEM of BOTH CTAs exist before anyone touches them
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_trigger();

    if (warp == 0 || warp == 7) {
        // producers: warp-uniform loops, one elected lane issues; ring position kept as a counter
        const int j = warp == 0 ? 0 : 1;
        pdl_wait();                                   // A is the previous kernel's output
        int s = 0;
        uint32_t ph = 1;
        for (int tile = cluster_id; tile < n_tiles && j < G2_KC; tile += n_clusters) {
            const int m_row = ((tile / n_tiles_n) * 2 + static_cast<int>(rank)) * G2_BM;
            for (int ks = 0; ks < num_ks; ++ks) {
                mbar_wait(&empty_bar[s], ph);
                if (elect_one()) {
                    if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * G2_A_CHUNK);
                    tma_load_2d_pair(sA + (s * G2_KC + j) * G2_A_CHUNK, &tmA, &full_bar[s], (ks * G2_KC + j) * G2_BK, m_row);
                }
                __syncwarp();
                if (++s == G2_STAGES) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 6 || warp == 8) {
        const int j = warp == 6 ? 0 : 1;
        int s = 0;
        uint32_t ph = 1;
        for (int tile = cluster_id; tile < n_tiles && j < G2_KC; tile += n_clusters) {
            const int n_row = (tile % n_tiles_n) * G2_BN + static_cast<int>(rank) * (G2_BN / 2);
            for (int ks = 0; ks < num_ks; ++ks) {
                mbar_wait(&empty_bar[s], ph);
                if (elect_one()) {
                    if (leader) mbar_arrive_expect_tx(&full_bar[s], 2 * G2_B_CHUNK);
                    tma_load_2d_pair(sB + (s * G2_KC + j) * G2_B_CHUNK, &tmB, &full_bar[s], (ks * G2_KC + j) * G2_BK, n_row);
                }
                __syncwarp();
                if (++s == G2_STAGES) { s = 0; ph ^= 1u; }
            }
        }
        pdl_wait();
    } else if (warp == 1) {
        if (leader) {
            // warp-uniform control flow, elect.sync picks the issuing lane (see gemm_sm100.cu: the lone-thread form of this
            // loop paid ~100 cycles of its own per MMA and ~170 per barrier probe)
            constexpr uint32_t idesc = umma_idesc_bf16(2 * G2_BM, G2_BN);
            const uint64_t da0 = umma_desc_sw128(smem_u32(sA));
            const uint64_t db0 = umma_desc_sw128(smem_u32(sB));
            int s = 0, local = 0;
            uint32_t ph = 0;
            for (int tile = cluster_id; tile < n_tiles; tile += n_clusters, ++local) {
                const int acc = local & 1;
                mbar_wait(&tempty_bar[acc], ((local >> 1) & 1) ^ 1);      // both CTAs have drained this accumulator
                tcgen05_fence_after();
                const uint32_t tmem_acc = tmem_base + acc * G2_BN;
                for (int ks = 0; ks < num_ks; ++ks) {
                    mbar_wait(&full_bar[s], ph);
                    tcgen05_fence_after();
                    if (elect_one()) {
                        const uint64_t da = da0 + static_cast<uint64_t>(s * ((G2_KC * G2_A_CHUNK) >> 4));
                        const uint64_t db = db0 + static_cast<uint64_t>(s * ((G2_KC * G2_B_CHUNK) >> 4));
#pragma unroll
                        for (int c = 0; c < G2_KC; ++c) {
#pragma unroll
                            for (int k = 0; k < G2_BK / 16; ++k)
                                umma_bf16_ss_pair(tmem_acc, da + (c * (G2_A_CHUNK >> 4) + 2 * k), db + (c * (G2_B_CHUNK >> 4) + 2 * k), idesc,
                                                  (ks | c | k) != 0 ? 1u : 0u);
                        }
                        umma_commit_pair(&empty_bar[s]);  // slot reusable in both CTAs once these MMAs have read it
                    }
                    __syncwarp();
                    if (++s == G2_STAGES) { s = 0; ph ^= 1u; }
                }
                if (elect_one()) umma_commit_pair(&tfull_bar[acc]);    // accumulator halves complete in both CTAs
                __syncwarp();
            }
        }
        pdl_wait();
    } else {
        if (warp < 9) l2_prefetch_share(p.prefetch, p.prefetch_bytes, (blockIdx.x * 4 + (warp - 2)) * 32 + lane, gridDim.x * 128);
        pdl_wait();                                   // bias / gate / residual may come from the previous kernel
        const int q = warp & 3;                       // TMEM lane quadrant this warp may read
        const int chalf = warp >= 9 ? 1 : 0;          // which 128 of the tile's 256 columns
        int local = 0;
        for (int tile = cluster_id; tile < n_tiles; tile += n_clusters, ++local) {
            const int m_row = ((tile / n_tiles_n) * 2 + static_cast<int>(rank)) * G2_BM;
            const int n_blk = tile % n_tiles_n;
            const int acc = local & 1;
            const int row = m_row + q * 32 + lane;
            const bf16* gate_row = nullptr;
            if (EPI == EPI_BIAS_GATE_RES && row < p.M) {
                int f = row / p.rows_per_frame;
                if (p.frame_row != nullptr) f = p.frame_row[f];
                gate_row = p.gate + static_cast<size_t>(f) * p.gate_ld;
            }
            mbar_wait(&tfull_bar[acc], (local >> 1) & 1);
            tcgen05_fence_after();
            // Two register buffers: the tcgen05.ld of the next 32 columns is in flight while the current ones go through the
            // epilogue math and their stores.  Not for the erf GELU: two inlined copies of that epilogue cost more than
            // the overlap gains (VAE fc1 at M = 18432: 961 -> 858 TFLOP/s), so it keeps the serial load -> wait -> math loop.
            {
                constexpr int C0 = G2_BN / 64;                                   // chunks of 32 columns per warp
                const uint32_t tbase = tmem_base + acc * G2_BN + (static_cast<uint32_t>(q * 32) << 16) + chalf * C0 * 32;
                const int colb = n_blk * G2_BN + chalf * C0 * 32;
                if (EPI == EPI_BIAS_GELU_ERF) {
#pragma unroll 1
                    for (int c = 0; c < C0; ++c) {
                        uint32_t v[32];
                        tmem_ld_32x32(tbase + c * 32, v);
                        tmem_ld_wait();
                        if (row < p.M) epilogue_chunk<EPI>(p, row, colb + c * 32, v, gate_row);
                    }
                } else {
                    uint32_t va[32], vb[32];
                    tmem_ld_32x32(tbase, va);
#pragma unroll
                    for (int c = 0; c < C0; ++c) {
                        tmem_ld_wait();
                        if (c + 1 < C0) {
                            if (c & 1) tmem_ld_32x32(tbase + (c + 1) * 32, va);
                            else tmem_ld_32x32(tbase + (c + 1) * 32, vb);
                        }
                        if (row < p.M) {
                            if (c & 1) epilogue_chunk<EPI>(p, row, colb + c * 32, vb, gate_row);
                            else epilogue_chunk<EPI>(p, row, colb + c * 32, va, gate_row);
                        }
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty_bar[acc]), 0));   // on the leader's barrier
        }
    }
    tcgen05_fence_before();
    cluster_sync_all();                               // no CTA leaves while its peer may still read its smem / signal it
    if (warp == 1) tmem_dealloc_pair(tmem_base, 2 * G2_BN);
}

// ------------------------------------------------------------------------------------------ host
bool gemm2_eligible(int M, int N, int K) {
    return M >= 2 * G2_BM && N % G2_BN == 0 && K % (G2_KC * G2_BK) == 0;
}

template <int EPI>
static int launch2(const GemmOp* op, cudaStream_t stream) {
    static bool configured = false;
    auto kern = gemm2_bf16_kernel<EPI>;
    if (!configured) {
        GTAV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM));
        configured = true;
    }
    int sms = 148, dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) sms = n;
    const int pairs = (op->p.N / G2_BN) * ((op->p.M + 2 * G2_BM - 1) / (2 * G2_BM));
    const int clusters = pairs < sms / 2 ? pairs : sms / 2;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * clusters);
    cfg.blockDim = dim3(G2_THREADS);
    cfg.dynamicSmemBytes = G2_SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    GTAV_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, op->tmA, op->tmB2, op->p));
    return 0;
}

int gemm2_run(const GemmOp* op, cudaStream_t stream) {
    switch (op->epi) {
        case EPI_STORE: return launch2<EPI_STORE>(op, stream);
        case EPI_BIAS: return launch2<EPI_BIAS>(op, stream);
        case EPI_BIAS_GELU_TANH: return launch2<EPI_BIAS_GELU_TANH>(op, stream);
        case EPI_BIAS_GELU_ERF: return launch2<EPI_BIAS_GELU_ERF>(op, stream);
        case EPI_BIAS_SILU: return launch2<EPI_BIAS_SILU>(op, stream);
        case EPI_BIAS_GATE_RES: return launch2<EPI_BIAS_GATE_RES>(op, stream);
        case EPI_BIAS_RES: return launch2<EPI_BIAS_RES>(op, stream);
        case EPI_BIAS_RES_SILU: return launch2<EPI_BIAS_RES_SILU>(op, stream);
    }
    set_error("gemm (2-CTA): unknown epilogue %d", op->epi);
    return -1;
}

}  // namespace gtav
