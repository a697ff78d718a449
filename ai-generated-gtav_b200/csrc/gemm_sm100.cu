// bf16 GEMM for sm_100a: out[M,N] = epilogue(A[M,K] @ W[N,K]^T), fp32 accumulation in TMEM.
//
// Replaces every nn.Linear / patchify-conv on the hot path (reference model/attention.py:27-28,86-87;
// model/dit.py:60-62,87-91,134,138,171-198; model/vae.py:65-67,147-152,192,214-215,233 and timm Mlp),
// with the surrounding elementwise ops (bias, GELU/SiLU, adaLN gate, residual) fused as epilogues that
// round to bf16 exactly where the reference's autocast graph does.
//
// Structure (persistent CTAs over 128 x BN output tiles, double-buffered TMEM accumulator, 416 threads):
//   warps 0,7: TMA producers of A - a stage is KC = 2 consecutive 64-wide K chunks of 128 rows, one box per warp
//   warps 6,8: TMA producers of W - the same for BN weight rows; they run ahead of the previous kernel (PDL): weights
//              do not depend on it
//   warp 1   : TMEM allocator + tcgen05.mma issue (UMMA 128 x BN x 16, cta_group::1): warp-uniform loops, elect.sync
//              picks the issuing lane
//   warps 2-5, 9-12: epilogue - tcgen05.ld 32x32b from their TMEM lane quadrant (two warps per quadrant, half of the
//              tile's columns each), fused math, 16-byte stores.  Eight warps: with four, a K = 1024 tile's GELU
//              epilogue outlasts its mainloop (measured on the CTA-pair kernel: 668 -> 968 TFLOP/s on fc1)
// smem full/empty mbarrier ring between the producers and the issuer; tcgen05.commit frees slots and signals
// the epilogue.  Out-of-range rows / columns / K are zero-filled by TMA and masked in the epilogue.
// Why four producer warps: measured on B200 (scripts/probe_tma*.cu, scripts/probe_mcast.cu, profiles/r01), one
// thread gets a bulk copy accepted only every ~0.4 us whatever its size, so a stage issued by one thread caps a CTA
// at ~45 GB/s (5x short of what a 128x128 tile needs) and two threads with 32 KB boxes at ~160 GB/s; copies from
// different threads proceed in parallel, and a 128 x 256 tile at full tensor rate needs ~175 GB/s.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.h"
#include "epilogue.cuh"

namespace gtav {

static constexpr int BM = 128;
static constexpr int BK = 64;                 // one 128-byte-swizzled chunk
static constexpr int GEMM_THREADS = 416;      // 13 warps: 5 producer / MMA + 8 epilogue

template <int BN, int STAGES, int KC>
struct GemmSmem {
    static constexpr int A_CHUNK = BM * BK * 2;
    static constexpr int B_CHUNK = BN * BK * 2;
    static constexpr int A_BYTES = KC * A_CHUNK;           // per stage
    static constexpr int B_BYTES = KC * B_CHUNK;
    static constexpr int BAR_OFF = STAGES * (A_BYTES + B_BYTES);
    static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 4) * 8 + 16 + 1024;   // +1024: manual alignment slack
};

// Persistent: CTA b works on output tiles b, b + gridDim.x, ... (n fastest, so neighbouring CTAs share the A rows in
// L2).  The accumulator is double-buffered in TMEM (2 x BN columns): while the epilogue warps drain tile i, the MMA
// issuer already accumulates tile i + 1, and the two TMA producers run ahead across tile boundaries - the per-tile
// prologue / epilogue (as long as a K = 1024 mainloop) leaves the critical path.
template <int BN, int STAGES, int KC, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
    using L = GemmSmem<BN, STAGES, KC>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + STAGES * L::A_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tfull_bar = empty_bar + STAGES;      // [2] accumulator complete
    uint64_t* tempty_bar = tfull_bar + 2;          // [2] accumulator drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n_tiles_n = (p.N + BN - 1) / BN;
    const int n_tiles = n_tiles_n * ((p.M + BM - 1) / BM);
    const int num_ks = (p.K + KC * BK - 1) / (KC * BK);      // pipeline stages along K (KC chunks each)

    if (warp == 0 && lane == 0) tma_prefetch_desc(&tmA);
    if (warp == 6 && lane == 0) tma_prefetch_desc(&tmB);
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < STAGES; ++s) {
                mbar_init(&full_bar[s], 2 * KC);      // one arrive.expect_tx per producer thread
                mbar_init(&empty_bar[s], 1);
            }
            for (int a = 0; a < 2; ++a) {
                mbar_init(&tfull_bar[a], 1);
                mbar_init(&tempty_bar[a], blockDim.x > 288 ? 8 : 4);   // one arrival per epilogue warp
            }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(tmem_slot, 2 * BN);
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_trigger();                                // the next kernel may start its own set-up now

    if (warp == 0 || warp == 7) {
        // A producers: warp j (warp 0 -> j = 0, warp 7 -> j = 1) loads K chunk j of every stage.  Warp-uniform loops, one
        // elected lane issues (same reason as the MMA warp below); ring position kept as a counter.
        const int j = warp == 0 ? 0 : 1;
        pdl_wait();                               // A is the previous kernel's output
        if (j < KC) {
            int s = 0;
            uint32_t ph = 1;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int m_blk = tile / n_tiles_n;
                for (int ks = 0; ks < num_ks; ++ks) {
                    mbar_wait(&empty_bar[s], ph);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&full_bar[s], L::A_CHUNK);
                        tma_load_2d(sA + s * L::A_BYTES + j * L::A_CHUNK, &tmA, &full_bar[s], (ks * KC + j) * BK, m_blk * BM);
                    }
                    __syncwarp();
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 6 || warp == 8) {
        // W producers, the same split; weights are never written by the kernel before us: stream them without waiting
        const int j = warp == 6 ? 0 : 1;
        if (j < KC) {
            int s = 0;
            uint32_t ph = 1;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int n_blk = tile % n_tiles_n;
                for (int ks = 0; ks < num_ks; ++ks) {
                    mbar_wait(&empty_bar[s], ph);
                    if (elect_one()) {
                        mbar_arrive_expect_tx(&full_bar[s], L::B_CHUNK);
                        tma_load_2d(sB + s * L::B_BYTES + j * L::B_CHUNK, &tmB, &full_bar[s], (ks * KC + j) * BK, n_blk * BN);
                    }
                    __syncwarp();
                    if (++s == STAGES) { s = 0; ph ^= 1u; }
                }
            }
        }
        pdl_wait();
    } else if (warp == 1) {
        // MMA issue with WARP-UNIFORM control flow: all 32 lanes run the loops and wait on the barriers, elect.sync picks the
        // issuing lane.  Inside `if (lane == 0)` the compiler keeps descriptors in vector registers and moves them to
        // uniform registers per tcgen05.mma, and every barrier probe of the lone thread costs ~170 cycles: measured
        // 106 -> 76 cycles per small MMA and 43 -> 7 cycles per MMA for one wait per four (scripts/probe_umma_chunks.cu) -
        // with 8 MMAs of 130 cycles per stage the lone thread was as slow as the tensor pipe.  Descriptors are a base
        // plus compile-time offsets; the ring position is a counter, not it % STAGES.
        constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
        const uint64_t da0 = umma_desc_sw128(smem_u32(sA));
        const uint64_t db0 = umma_desc_sw128(smem_u32(sB));
        int s = 0, local = 0;
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++local) {
            const int acc = local & 1;
            mbar_wait(&tempty_bar[acc], ((local >> 1) & 1) ^ 1);          // epilogue has drained this accumulator
            tcgen05_fence_after();
            const uint32_t tmem_acc = tmem_base + acc * BN;
            for (int ks = 0; ks < num_ks; ++ks) {
                mbar_wait(&full_bar[s], ph);
                tcgen05_fence_after();
                if (elect_one()) {
                    const uint64_t da = da0 + static_cast<uint64_t>(s * (L::A_BYTES >> 4));
                    const uint64_t db = db0 + static_cast<uint64_t>(s * (L::B_BYTES >> 4));
#pragma unroll
                    for (int c = 0; c < KC; ++c) {
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            // +32 bytes (16 bf16) along K inside the 128-byte swizzle row: +2 in 16-byte units
                            umma_bf16_ss(tmem_acc, da + (c * (L::A_CHUNK >> 4) + 2 * k), db + (c * (L::B_CHUNK >> 4) + 2 * k), idesc,
                                         (ks | c | k) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(&empty_bar[s]);       // slot reusable once these MMAs have read it
                }
                __syncwarp();
                if (++s == STAGES) { s = 0; ph ^= 1u; }
            }
            if (elect_one()) umma_commit(&tfull_bar[acc]);     // accumulator complete
            __syncwarp();
        }
        pdl_wait();
    } else {
        // idle until the first accumulator is ready: pull the NEXT GEMM's weights into L2 meanwhile
        if (warp < 9) l2_prefetch_share(p.prefetch, p.prefetch_bytes, (blockIdx.x * 4 + (warp - 2)) * 32 + lane, gridDim.x * 128);
        pdl_wait();                               // bias / gate / residual may come from the previous kernel
        const int q = warp & 3;                   // TMEM lane quadrant this warp may read
        const bool wide = blockDim.x > 288;       // 8 epilogue warps: two per quadrant, half of the columns each
        const int c_lo = wide ? (warp >= 9 ? BN / 64 : 0) : 0, c_hi = wide ? (warp >= 9 ? BN / 32 : BN / 64) : BN / 32;
        int local = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++local) {
            const int m_blk = tile / n_tiles_n, n_blk = tile % n_tiles_n;
            const int acc = local & 1;
            const int row = m_blk * BM + q * 32 + lane;
            const bf16* gate_row = nullptr;
            if (EPI == EPI_BIAS_GATE_RES && row < p.M) {
                int f = row / p.rows_per_frame;
                if (p.frame_row != nullptr) f = p.frame_row[f];
                gate_row = p.gate + static_cast<size_t>(f) * p.gate_ld;
            }
            mbar_wait(&tfull_bar[acc], (local >> 1) & 1);
            tcgen05_fence_after();
            // Two register buffers: the tcgen05.ld of the next 32 columns is in flight while the current ones go through the
            // epilogue math and their stores (context pass 1.88 -> 1.83 ms, dense B = 1 step 1.89 -> 1.87 ms).  Not for the
            // erf GELU, whose two inlined epilogue copies cost more than the overlap gains (see gemm_sm100_2cta.cu).
            {
                const uint32_t tbase = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);
                if (EPI == EPI_BIAS_GELU_ERF) {
#pragma unroll 1
                    for (int c = c_lo; c < c_hi; ++c) {
                        uint32_t v[32];
                        tmem_ld_32x32(tbase + c * 32, v);
                        tmem_ld_wait();
                        const int col0 = n_blk * BN + c * 32;
                        if (row < p.M && col0 < p.N) epilogue_chunk<EPI>(p, row, col0, v, gate_row);
                    }
                } else {
                    uint32_t va[32], vb[32];
                    tmem_ld_32x32(tbase + c_lo * 32, va);
#pragma unroll 1
                    for (int c = c_lo; c < c_hi; c += 2) {
                        tmem_ld_wait();
                        if (c + 1 < c_hi) tmem_ld_32x32(tbase + (c + 1) * 32, vb);
                        int col0 = n_blk * BN + c * 32;
                        if (row < p.M && col0 < p.N) epilogue_chunk<EPI>(p, row, col0, va, gate_row);
                        if (c + 1 < c_hi) {
                            tmem_ld_wait();
                            if (c + 2 < c_hi) tmem_ld_32x32(tbase + (c + 2) * 32, va);
                            col0 += 32;
                            if (row < p.M && col0 < p.N) epilogue_chunk<EPI>(p, row, col0, vb, gate_row);
                        }
                    }
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty_bar[acc]);     // this warp's quadrant of the accumulator is free
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 2 * BN);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn == nullptr) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// [rows, cols] bf16 row-major with leading dimension ld -> tiles of box_rows x 64, 128-byte swizzle.
static int make_tmap(CUtensorMap* out, const bf16* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    EncodeTiledFn enc = encode_fn();
    if (enc == nullptr) {
        set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
        return -3;
    }
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld % 8) != 0) {
        set_error("GEMM operand must be 16-byte aligned with a leading dimension multiple of 8 (ptr=%p ld=%llu)", ptr,
                  (unsigned long long)ld);
        return -1;
    }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstride[1] = {ld * sizeof(bf16)};
    cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<bf16*>(ptr), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%llu cols=%llu ld=%llu box_rows=%u)", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows);
        return -3;
    }
    return 0;
}

int make_tmap_3d(CUtensorMap* out, const bf16* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                 uint32_t box_chunks) {
    EncodeTiledFn enc = encode_fn();
    if (enc == nullptr) {
        set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
        return -3;
    }
    if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0 || (ld % 8) != 0 || (cols % BK) != 0 || box_rows > 256 || box_chunks > 256) {
        set_error("GEMM operand (3-D view) must be 16-byte aligned, ld %% 8 == 0, K %% 64 == 0 (ptr=%p ld=%llu K=%llu)", ptr,
                  (unsigned long long)ld, (unsigned long long)cols);
        return -1;
    }
    cuuint64_t gdim[3] = {static_cast<cuuint64_t>(BK), rows, cols / BK};
    cuuint64_t gstride[2] = {ld * sizeof(bf16), BK * sizeof(bf16)};
    cuuint32_t box[3] = {static_cast<cuuint32_t>(BK), box_rows, box_chunks};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<bf16*>(ptr), gdim, gstride, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (3-D) failed with CUresult %d (rows=%llu cols=%llu ld=%llu box=%ux%u)", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_chunks);
        return -3;
    }
    return 0;
}

static int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

int gemm_prepare(GemmOp* op, const bf16* A, int lda, const bf16* W, int ldw, const GemmParams& p, int epi,
                 int bn_override) {
    if (p.M <= 0 || p.N <= 0 || p.K <= 0 || (p.N % 8) != 0 || (p.K % 8) != 0) {
        set_error("gemm: unsupported shape M=%d N=%d K=%d (N and K must be positive multiples of 8)", p.M, p.N, p.K);
        return -1;
    }
    if (epi < 0 || epi >= EPI_COUNT) {
        set_error("gemm: unknown epilogue %d", epi);
        return -1;
    }
    if (epi != EPI_STORE && p.bias == nullptr) {
        set_error("gemm: epilogue %d needs a bias vector", epi);
        return -1;
    }
    if (epi == EPI_BIAS_GATE_RES && (p.gate == nullptr || p.res == nullptr || p.rows_per_frame <= 0)) {
        set_error("gemm: gated-residual epilogue needs gate, residual and rows_per_frame");
        return -1;
    }
    if ((p.ldo % 8) != 0 || (p.res != nullptr && (p.ldr % 8) != 0) || (p.gate != nullptr && (p.gate_ld % 8) != 0)) {
        set_error("gemm: output / residual / gate leading dimensions must be multiples of 8");
        return -1;
    }
    const int m_tiles = (p.M + BM - 1) / BM;
    int bn = bn_override;
    double best = 1e30;                     // cost of the best single-CTA tiling (cycles per K = 16 step x rounds)
    if (bn == 0) {
        // cost of one tile per K = 16 step, in cycles: the larger of the MMA (61 / 68 / 130 cycles at BN = 64 / 128 / 256,
        // scripts/probe_umma_rate.cu) and the operand ingest at the ~160 GB/s per SM two TMA producer warps reach
        // (71 / 95 / 142); times the number of rounds the persistent CTAs need.  Ties go to the wider tile.
        const int cand[3] = {256, 128, 64};
        const double cost[3] = {142.0, 95.0, 71.0};
        for (int i = 0; i < 3; ++i) {
            if (cand[i] > 64 && p.N <= cand[i] / 2) continue;               // mostly padding
            const int tiles = m_tiles * ((p.N + cand[i] - 1) / cand[i]);
            const double c = static_cast<double>((tiles + num_sms() - 1) / num_sms()) * cost[i];
            if (c < best - 1e-9) { best = c; bn = cand[i]; }
        }
        // One round of 256-wide tiles (M <= 1152 at N = 3072 / 4096): two rounds of 128-wide tiles are faster - the first
        // round's epilogue runs under the second round's mainloop and each tile's prologue / epilogue is half as long.
        // In-graph, scripts/sweep_gemm_tiles.py --graph: fc1 at M = 1152 / 720 / 576 14.45 / 13.96 / 14.19 -> 13.37 / 12.78 /
        // 12.53 us, to_qkv at M = 1152 12.73 -> 12.04 us.
        if (bn == 256 && m_tiles * ((p.N + 255) / 256) <= num_sms()) bn = 128;
    }
    // Few tiles and a long K (fc2 at M <= 1152): the K-serial mainloop dominates - two CTAs per 128 x 128 tile, half of K
    // each (gemm_sm100_splitk.cu).  GTAV_GEMM_SPLITK=0 / 1 forces the choice (1: whenever eligible).
    op->split_k = 0;
    if (bn_override == 0 && gemm_splitk_eligible(p.M, p.N, p.K, num_sms())) {
        const char* e = getenv("GTAV_GEMM_SPLITK");
        op->split_k = e != nullptr ? (e[0] == '1') : 1;
        if (op->split_k) bn = 128;
    }
    if (bn != 64 && bn != 128 && bn != 256) {
        set_error("gemm: tile width %d not in {64,128,256}", bn);
        return -1;
    }
    op->p = p;
    op->bn = bn;
    op->epi = epi;
    // two 64-wide K chunks per pipeline stage (one per producer thread) unless K is a single chunk
    op->kc = p.K > BK ? 2 : 1;
    // one 2-D box (rows x 64) per K chunk and producer thread, whatever the stage depth
    int rc = make_tmap(&op->tmA, A, p.M, p.K, lda, BM);
    if (rc) return rc;
    // CTA pairs (gemm_sm100_2cta.cu) where the shape allows and the GEMM is large enough to be ingest-bound on one
    // SM.  GTAV_GEMM_2CTA=0 / 1 forces the choice (1: whenever eligible).
    op->two_cta = 0;
    if (bn_override == 0 && !op->split_k && gemm2_eligible(p.M, p.N, p.K)) {
        const char* e = getenv("GTAV_GEMM_2CTA");
        // same cost model for the CTA pair: a 256 x 256 tile pair on two SMs is MMA-bound (130 cycles per K = 16 step:
        // each SM ingests a third less), rounds over the num_sms / 2 clusters.  E.g. (scripts/bench_2cta.py) M = 1152
        // fc1: 80 pairs = 2 rounds x 130 vs 144 single tiles = 1 round x 142 -> single (22.5 vs 28.7 us measured);
        // M = 5760 fc2: 92 pairs = 260 vs 184 tiles = 284 -> pair (57.3 vs 69.7 us measured).
        const int pairs = ((p.M + 255) / 256) * (p.N / 256), clusters = num_sms() / 2;
        // (several rounds only: its eight epilogue warps cost a single-round GEMM more than they save, see launch_one)
        const bool big = pairs > clusters && static_cast<double>((pairs + clusters - 1) / clusters) * 130.0 < best;
        op->two_cta = e != nullptr ? (e[0] == '1') : big;
    }
    if (op->two_cta && (rc = make_tmap(&op->tmB2, W, p.N, p.K, ldw, 128))) return rc;
    return make_tmap(&op->tmB, W, p.N, p.K, ldw, bn);
}

template <int BN, int STAGES, int KC, int EPI>
static int launch_one(const GemmOp* op, cudaStream_t stream) {
    using L = GemmSmem<BN, STAGES, KC>;
    static bool configured = false;
    auto kern = gemm_bf16_kernel<BN, STAGES, KC, EPI>;
    if (!configured) {
        GTAV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
        configured = true;
    }
    const int tiles = ((op->p.N + BN - 1) / BN) * ((op->p.M + BM - 1) / BM);
    dim3 grid(tiles < num_sms() ? tiles : num_sms(), 1, 1);
    // 8 epilogue warps (416 threads) when the CTAs run several tiles each (the epilogue of tile i must not outlast the
    // mainloop of tile i + 1: fc1 at M = 9216 674 -> 993 TFLOP/s) and, whatever the number of rounds, for the GELU epilogues:
    // a single-round GEMM's epilogue is fully exposed, and the GELU one is the longest (measured in the real steps,
    // scripts/bench_step_b8.py: B = 8 last-frame step 2.645 -> 2.505 ms, dense B = 1 step 2.275 -> 2.119 ms).  4 warps (288
    // threads) for the other single-round GEMMs, where the extra warps only cost (gated-residual epilogue with 8: 2.84 ms;
    // plain store: no change).
    const bool gelu = EPI == EPI_BIAS_GELU_TANH || EPI == EPI_BIAS_GELU_ERF;
    const int epi_warps = (tiles > num_sms() || gelu) ? 8 : 4;
    GTAV_CUDA_OK(launch_k(kern, grid, dim3(epi_warps == 8 ? GEMM_THREADS : 288), L::TOTAL, stream, op->tmA, op->tmB, op->p));
    return 0;
}

template <int EPI>
static int launch_epi(const GemmOp* op, cudaStream_t stream) {
    if (op->kc == 2) {
        switch (op->bn) {
            case 64: return launch_one<64, 4, 2, EPI>(op, stream);       // 4 x 48 KB
            case 128: return launch_one<128, 3, 2, EPI>(op, stream);     // 3 x 64 KB
            default: return launch_one<256, 2, 2, EPI>(op, stream);      // 2 x 96 KB
        }
    }
    switch (op->bn) {
        case 64: return launch_one<64, 4, 1, EPI>(op, stream);
        case 128: return launch_one<128, 3, 1, EPI>(op, stream);
        default: return launch_one<256, 4, 1, EPI>(op, stream);
    }
}

int gemm_run(const GemmOp* op, cudaStream_t stream) {
    if (op->split_k) return gemm_splitk_run(op, stream);
    if (op->two_cta) return gemm2_run(op, stream);
    switch (op->epi) {
        case EPI_STORE: return launch_epi<EPI_STORE>(op, stream);
        case EPI_BIAS: return launch_epi<EPI_BIAS>(op, stream);
        case EPI_BIAS_GELU_TANH: return launch_epi<EPI_BIAS_GELU_TANH>(op, stream);
        case EPI_BIAS_GELU_ERF: return launch_epi<EPI_BIAS_GELU_ERF>(op, stream);
        case EPI_BIAS_SILU: return launch_epi<EPI_BIAS_SILU>(op, stream);
        case EPI_BIAS_GATE_RES: return launch_epi<EPI_BIAS_GATE_RES>(op, stream);
        case EPI_BIAS_RES: return launch_epi<EPI_BIAS_RES>(op, stream);
        case EPI_BIAS_RES_SILU: return launch_epi<EPI_BIAS_RES_SILU>(op, stream);
    }
    set_error("gemm: unknown epilogue %d", op->epi);
    return -1;
}

// ------------------------------------------------------------------------------------------
// error text
// ------------------------------------------------------------------------------------------
bool pdl_enabled() {
    static int on = -1;
    if (on < 0) {
        const char* e = getenv("GTAV_PDL");
        on = (e != nullptr && e[0] == '0') ? 0 : 1;
    }
    return on != 0;
}

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char* get_error() { return g_err; }

}  // namespace gtav
