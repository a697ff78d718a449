// Non-causal multi-head attention over short sequences on the 5th-generation tensor cores, rotary embedding fused
// into the operand staging.
//
// Replaces SpatialAxialAttention's rearrange + get_axial_freqs + apply_rotary_emb + SDPA (reference
// model/attention.py:99-129: S = 144 tokens per frame, rotary on all 64 head dims) and the VAE Attention
// (reference model/vae.py:78-107: S = 576, rotary on head dims 0..31 only).  Head dim 64; one CTA per (sequence, head).
//
//   * K and V of the whole head are brought ONCE into shared memory with cp.async (all copies of a thread in flight
//     together) as 128-byte-swizzled rows of 64 bf16; K is then rotated in place (rounded fp32 products and sum, then
//     bf16 - apply_rotary_emb, rotary_embedding_torch.py:46-73).  K is the K-major B operand of S = Q K^T, the same kind of
//     image of V is the MN-major B operand of O = P V (no transpose anywhere);
//   * queries are processed in tiles of 128 rows (UMMA M = 128), staged the same way by two loader warps into a
//     double-buffered slot while the previous tile is being worked on;
//   * the (query tile, key block) pairs form ONE flat sequence n = 0, 1, ...: the MMA warp issues S(n + 1), S(n + 2) = Q K^T
//     into a ring of TMEM S buffers ahead of the P V product of block n, and the softmax warpgroups take the blocks round
//     robin (group g the blocks n = g mod G; thread = query row = TMEM lane), so that one group's TMEM loads, stores and
//     barrier waits run under the other groups' exponentials.  S = 576: three buffers of 144 keys and three groups (a
//     group's next S tile is ready when it finishes the current one); S = 144: one buffer, two groups, two CTAs per SM.
//     The MUFU pipe (one ex2 per score, 16 per clock per SM) and the softmax warps' instruction issue (~8 instructions
//     per score) are the bounds of this kernel: ~0.6 us per 128 x 144 block each, against ~1.2 us measured;
//   * softmax across key blocks is the online one with LAZY rescaling: a block adopts the previous blocks' row
//     maximum unless its own exceeds it by more than 2^8 (probabilities then stay below 256, harmless in fp32 / bf16);
//     only then are the row's partial O (tcgen05.ld / st) and row sum rescaled - with bounded logits that is rare.  The
//     result is the exact softmax (every probability of a row is scaled by the same factor);
//   * probabilities are rounded to bf16 like the reference's fused SDPA backends and written straight back into TENSOR
//     MEMORY with tcgen05.st, over the S columns they were computed from (two bf16 per 32-bit column, row = lane): the
//     second product takes its A operand P from TMEM (tcgen05.mma [d], [a], b-desc), so the probabilities never touch
//     shared memory - no 48 KB staging buffer, no generic -> async proxy fence, and the softmax threads stream
//     load -> exp -> store 32 columns at a time without holding a whole row in registers;
//   * O [128 x 64] accumulates in TMEM (double-buffered across query tiles) and is normalised by the fp32 row sum in
//     the epilogue;
//   * every hand-off is an mbarrier (tcgen05.commit on the tensor side); no CTA-wide barrier inside the loop.
#include <stdlib.h>

#include "common.cuh"
#include "kernels.h"

namespace gtav {

namespace {

constexpr int AT_GROUP_WARPS = 4;                     // one softmax warpgroup = 128 query rows (one warp per TMEM lane quadrant)
constexpr int AT_LOADER_WARPS = 2;
constexpr int AT_MMA_WARPS = 1;                       // one warp (one elected lane) issues every MMA.  Measured alternatives (32 VAE frames, this
                                                      // kernel 127 us): one issuing thread per product with blocking waits 134 us
                                                      // (and, with 96-key blocks in four buffers, a hang in later-wave CTAs that
                                                      // was not understood); 96-key blocks with a fixed issue order and blocking
                                                      // waits 162 us, with the polling scheduler 146 us; four softmax groups 146 us
__host__ __device__ constexpr int at_threads(int groups) { return (groups * AT_GROUP_WARPS + AT_MMA_WARPS + AT_LOADER_WARPS) * 32; }   // 352 (2 groups), 480 (3 groups)
constexpr int AT_QTILE = 128;
constexpr int AT_ROWB = 128;                          // bytes per staged row (64 bf16)
constexpr float AT_LAZY = 8.0f;                       // rescale only when the maximum grows by more than 2^8

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
          "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
          "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]: A = 128 lanes (rows) x 16 bf16 (8 columns of 32 bits) starting at tmem_a
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(src_bytes) : "memory");
}

// rotate the adjacent pair packed in `u` by (cos, sin) and re-round to bf16: two rounded fp32 products, a rounded fp32
// sum, then the bf16 rounding, as the reference's t * cos + rotate_half(t) * sin (no FMA contraction)
__device__ __forceinline__ uint32_t rot_pair(uint32_t u, float2 cs) {
    const float2 x = unpack_bf16x2(u);
    return pack_bf16x2(__fsub_rn(__fmul_rn(x.x, cs.x), __fmul_rn(x.y, cs.y)),
                       __fadd_rn(__fmul_rn(x.y, cs.x), __fmul_rn(x.x, cs.y)));
}
// byte offset of chunk c of row r inside a [rows][128 B] image with the 128-byte swizzle (chunk index ^ row % 8)
__device__ __forceinline__ uint32_t sw128(int r, int c) { return static_cast<uint32_t>(r) * AT_ROWB + ((c ^ (r & 7)) << 4); }
// Copy chunk c (16 bytes = 8 features) of rows r0, r0 + RSTRIDE, ... (< n_rows of the image; sequence position pos0 + row,
// rows at positions >= seq are zero-filled) from global memory into the swizzled image with cp.async - every copy of
// the thread in flight at once - and rotate the chunks that carry rotary pairs in place.  The rotary angles of a batch
// of rows are fetched into registers while the copies are in flight (fetched row by row after the wait, each was an
// exposed L2 round trip: 4 us per 128-row tile).  A thread only ever touches chunks it copied itself, so no barrier is
// needed between the copy and the rotation.  src2 / img2: optional second matrix copied alongside without rotation (V).
template <int ROT_PAIRS, int RSTRIDE, int MAXROWS, int RB>
__device__ __forceinline__ void stage_rows(uint8_t* img, const bf16* src, uint8_t* img2, const bf16* src2, int ld, int r0, int c,
                                           int n_rows, int pos0, int seq, const float2* __restrict__ rot) {
    for (int r = r0; r < n_rows; r += RSTRIDE) {
        const bool ok = pos0 + r < seq;
        const size_t goff = ok ? static_cast<size_t>(pos0 + r) * ld + c * 8 : 0;
        cp_async16(img + sw128(r, c), src + goff, ok ? 16 : 0);
        if (img2 != nullptr) cp_async16(img2 + sw128(r, c), src2 + goff, ok ? 16 : 0);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (c * 4 < ROT_PAIRS) {
#pragma unroll 1
        for (int k0 = 0; k0 < MAXROWS; k0 += RB) {
            float4 tb[RB][2];
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const int r = r0 + (k0 + i) * RSTRIDE;
                if (r < n_rows && pos0 + r < seq) {
                    const float4* tp = reinterpret_cast<const float4*>(rot + (pos0 + r) * ROT_PAIRS + c * 4);
                    tb[i][0] = tp[0];
                    tb[i][1] = tp[1];
                }
            }
            if (k0 == 0) asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
            for (int i = 0; i < RB; ++i) {
                const int r = r0 + (k0 + i) * RSTRIDE;
                if (r < n_rows && pos0 + r < seq) {
                    uint4* p = reinterpret_cast<uint4*>(img + sw128(r, c));
                    uint4 w = *p;
                    w.x = rot_pair(w.x, make_float2(tb[i][0].x, tb[i][0].y));
                    w.y = rot_pair(w.y, make_float2(tb[i][0].z, tb[i][0].w));
                    w.z = rot_pair(w.z, make_float2(tb[i][1].x, tb[i][1].y));
                    w.w = rot_pair(w.w, make_float2(tb[i][1].z, tb[i][1].w));
                    *p = w;
                }
            }
        }
    } else {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
}

// kind::f16 instruction descriptor with an MN-major B operand (bit 16): V staged as [key][64 dims]
__host__ __device__ constexpr uint32_t idesc_bf16_bmn(int m, int n) { return umma_idesc_bf16(m, n) | (1u << 16); }

template <int SEQ, int KB, int NBUF, int TMC, int G>
struct AttnCfg {
    static constexpr int NKB = SEQ / KB;                               // key blocks per query tile
    static constexpr int QTILES = (SEQ + AT_QTILE - 1) / AT_QTILE;
    static constexpr int NBLK = QTILES * NKB;                          // length of the flat (tile, block) sequence
    static constexpr int KV_BYTES = SEQ * AT_ROWB;
    static constexpr int Q_BYTES = AT_QTILE * AT_ROWB;                 // 16 KB
    static constexpr int OFF_V = KV_BYTES;
    static constexpr int OFF_Q = 2 * KV_BYTES;
    static constexpr int OFF_M = OFF_Q + 2 * Q_BYTES;                  // running row maximum handed from block to block
    static constexpr int OFF_L = OFF_M + AT_QTILE * 4;                 // (row sum, its reference maximum) of each group, per tile parity
    static constexpr int OFF_BAR = OFF_L + 2 * G * AT_QTILE * 8;
    static constexpr int L_PUBLISHERS = (NKB < G ? NKB : G) - 1;       // groups other than the one that finishes a tile
    static constexpr int SMEM = OFF_BAR + 256 + 1024;                  // + alignment slack
    // TMEM columns: S_0 | ... | S_{NBUF-1} | O_0 (| O_1); P(n) overwrites S(n)[0, KB/2)
    static constexpr int S_COLS = KB;
    static constexpr int TM_O = NBUF * S_COLS;
    static constexpr int OBUF = (TMC - TM_O) >= 128 ? 2 : 1;
    static constexpr int TM_COLS = TMC;                                // 256: two CTAs of the S = 144 variant share an SM
    static_assert(SEQ % KB == 0 && KB % 16 == 0 && KB <= 256 && (KB % 32 == 0 || KB % 32 == 16), "key blocking");
    static_assert((KB * AT_ROWB) % 1024 == 0, "key blocks must start on a swizzle-atom boundary");
    static_assert(NBUF >= 1 && NBUF <= 4 && TM_O + 64 * OBUF <= TMC && (TMC == 256 || TMC == 512), "TMEM budget");
    static_assert(G >= NBUF, "the S_FULL wait of the softmax groups assumes no more S buffers than groups");
    static_assert(SMEM <= 232448, "shared memory budget");
};

// Barrier slots.  S_FREE[k] is committed by the tensor core after the P V product that read P out of S buffer k.  Every
// barrier that a producer could otherwise complete twice before its consumer has looked (a parity wait cannot tell phase
// i from phase i + 2) exists once per S buffer / O buffer / query slot, so that the producer's next arrival depends on
// the consumer having gone through.
enum { B_QFULL = 0, B_QFREE = 2, B_SFULL = 4, B_SFREE = 8, B_PREADY = 12, B_OFULL = 16, B_OFREE = 18, B_MREADY = 20,
       B_LREADY = 24, B_DBG = 25, B_COUNT = 26 };   // M_READY: one barrier per softmax group (up to 4)

__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {       // non-blocking probe (try_wait may suspend)
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}

template <int SEQ, int KB, int NBUF, int TMC, int G, int ROT_PAIRS>
__global__ void __launch_bounds__(at_threads(G), (TMC == 256 ? 2 : 1))
attn_tc_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int heads, const float2* __restrict__ rot, long long* trace) {
    using C = AttnCfg<SEQ, KB, NBUF, TMC, G>;
    constexpr int AT_SOFTMAX_WARPS = G * AT_GROUP_WARPS;
    constexpr int AT_THREADS = at_threads(G);
    // optional phase trace (profiling aid, null in production): [cta][role 0 softmax A / 1 mma / 2 loader / 3 softmax B][64] ns
    int n_stamp = 0;
#define AT_STAMP(role)                                                                                          \
    do {                                                                                                        \
        if (trace != nullptr && n_stamp < 64) {                                                                 \
            long long t__;                                                                                      \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t__));                                            \
            reinterpret_cast<long long*>(reinterpret_cast<uintptr_t>(trace) & ~uintptr_t(15))[(static_cast<size_t>(blockIdx.x) * 4 + (role)) * 64 + n_stamp++] = t__; \
        }                                                                                                       \
    } while (0)
    extern __shared__ uint8_t smem_raw[];
    // (offset arithmetic on the __shared__ array itself: the compiler keeps the address space and emits LDS / STS - a
    // pointer rebuilt from an integer made every shared access a generic LD / ST with long-scoreboard stalls)
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t* sK = smem;
    uint8_t* sV = smem + C::OFF_V;
    uint8_t* sQ = smem + C::OFF_Q;
    float* sM = reinterpret_cast<float*>(smem + C::OFF_M);
    float2* sL = reinterpret_cast<float2*>(smem + C::OFF_L);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::OFF_BAR);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + B_COUNT);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int head = blockIdx.x % heads, group = blockIdx.x / heads;
    const int ld = 3 * heads * 64;
    const size_t row_base = static_cast<size_t>(group) * SEQ;
    const bf16* qbase = qkv + row_base * ld + head * 64;
    const bf16* kbase = qbase + heads * 64;
    const bf16* vbase = kbase + heads * 64;

    if (threadIdx.x == 0) {
        for (int i = 0; i < 2; ++i) {
            mbar_init(&bars[B_QFULL + i], AT_LOADER_WARPS * 32);
            mbar_init(&bars[B_QFREE + i], 1);
            mbar_init(&bars[B_OFULL + i], 1);
            mbar_init(&bars[B_OFREE + i], AT_GROUP_WARPS * 32);
        }
        for (int i = 0; i < 4; ++i) {
            mbar_init(&bars[B_SFULL + i], 1);
            mbar_init(&bars[B_SFREE + i], 1);
            mbar_init(&bars[B_PREADY + i], AT_GROUP_WARPS * 32);
        }
        for (int i = 0; i < 4; ++i) mbar_init(&bars[B_MREADY + i], AT_GROUP_WARPS * 32);
        mbar_init(&bars[B_LREADY], (C::L_PUBLISHERS > 0 ? C::L_PUBLISHERS : 1) * AT_GROUP_WARPS * 32);
        mbar_init(&bars[B_DBG], 1);
        fence_barrier_init();
    }
    if (warp == AT_SOFTMAX_WARPS) {
        tmem_alloc(tmem_slot, C::TM_COLS);
        tmem_relinquish();
    }
    pdl_trigger();
    if (threadIdx.x == 0) AT_STAMP(0);             // entry
    pdl_wait();                                    // qkv is the previous kernel's output

    // ---- K and V of the whole head -> shared memory (see stage_rows), by the softmax and MMA warps; the loader warps
    // stage the first query tile meanwhile
    constexpr int KV_THREADS = (AT_SOFTMAX_WARPS + AT_MMA_WARPS) * 32;
    if (warp < AT_SOFTMAX_WARPS + AT_MMA_WARPS) {
        constexpr int RS = KV_THREADS / 8, MAXR = (SEQ + RS - 1) / RS;
        stage_rows<ROT_PAIRS, RS, MAXR, (MAXR + 1) / 2>(sK, kbase, sV, vbase, ld, threadIdx.x >> 3, threadIdx.x & 7, SEQ, 0, SEQ, rot);
        fence_proxy_async_smem();                  // generic-proxy stores -> visible to the tensor core's async proxy
    } else {
        const int lt = threadIdx.x - KV_THREADS;
        constexpr int RS = AT_LOADER_WARPS * 4, MAXR = AT_QTILE / RS;
        stage_rows<ROT_PAIRS, RS, MAXR, MAXR / 2>(sQ, qbase, nullptr, nullptr, ld, lt >> 3, lt & 7, AT_QTILE, 0, SEQ, rot);
        fence_proxy_async_smem();                  // (q_full[0] is arrived on after the barrier below has published the mbarriers)
    }
    tcgen05_fence_before();
    __syncthreads();                               // (the loaders arrive at once; mbarriers / TMEM address are published here)
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) AT_STAMP(0);             // K / V staged

    if (warp < AT_SOFTMAX_WARPS) {
        // =========================================================================== softmax + epilogue warpgroups
        const int grp = warp >> 2, q = warp & 3;                         // group g takes the blocks n = g, g + G, g + 2G, ...
        const int row = q * 32 + lane;                                   // row of the query tile = TMEM lane
        const int tr_role = grp == 0 ? 0 : 3;
        const bool tr = trace != nullptr && lane == 0 && q == 0 && grp < 2;
        const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
        const float sl2 = 0.125f * 1.4426950408889634f;                  // 1/sqrt(64) * log2(e)
        const int ldo = heads * 64;
        float l = 0.f, m_mine = -INFINITY;                               // this thread's share of the row sum, relative to m_mine
        // epilogue of tile t: O / (row sum) -> bf16 -> out[row][head*64 ..]; l_fin / m_fin: this thread's share of the row sum
        auto epilogue = [&](int t, float l_fin, float m_fin) {
            float lt = l_fin;
            if (C::L_PUBLISHERS > 0) {
                mbar_wait(&bars[B_LREADY], t & 1);
                const int g_fin = (t * C::NKB + C::NKB - 1) % G;         // the group running this epilogue
#pragma unroll
                for (int i = 1; i <= C::L_PUBLISHERS; ++i) {             // the groups of the tile's last blocks before the final one
                    const float2 o = sL[((t & 1) * G + (g_fin + G - i) % G) * AT_QTILE + row];
                    lt += o.x * ex2_approx((o.y - m_fin) * sl2);
                }
            }
            const float inv = 1.0f / lt;
            const uint32_t ob = t % C::OBUF;
            mbar_wait(&bars[B_OFULL + ob], (t / C::OBUF) & 1);
            tcgen05_fence_after();
            if (tr) AT_STAMP(tr_role);                                   // O full
            const int grow = t * AT_QTILE + row;
            bf16* dst = out + (row_base + grow) * ldo + head * 64;
            uint32_t o0[32], o1[32];
            tmem_ld_32x32(tlane + C::TM_O + ob * 64, o0);
            tmem_ld_32x32(tlane + C::TM_O + ob * 64 + 32, o1);
            tmem_ld_wait();
            tcgen05_fence_before();
            mbar_arrive(&bars[B_OFREE + ob]);                            // O is in registers: a later tile may overwrite it
            if (grow < SEQ) {
#pragma unroll
                for (int c = 0; c < 32; c += 8) {
                    uint4 w;
                    w.x = pack_bf16x2(__uint_as_float(o0[c]) * inv, __uint_as_float(o0[c + 1]) * inv);
                    w.y = pack_bf16x2(__uint_as_float(o0[c + 2]) * inv, __uint_as_float(o0[c + 3]) * inv);
                    w.z = pack_bf16x2(__uint_as_float(o0[c + 4]) * inv, __uint_as_float(o0[c + 5]) * inv);
                    w.w = pack_bf16x2(__uint_as_float(o0[c + 6]) * inv, __uint_as_float(o0[c + 7]) * inv);
                    *reinterpret_cast<uint4*>(dst + c) = w;
                }
#pragma unroll
                for (int c = 0; c < 32; c += 8) {
                    uint4 w;
                    w.x = pack_bf16x2(__uint_as_float(o1[c]) * inv, __uint_as_float(o1[c + 1]) * inv);
                    w.y = pack_bf16x2(__uint_as_float(o1[c + 2]) * inv, __uint_as_float(o1[c + 3]) * inv);
                    w.z = pack_bf16x2(__uint_as_float(o1[c + 4]) * inv, __uint_as_float(o1[c + 5]) * inv);
                    w.w = pack_bf16x2(__uint_as_float(o1[c + 6]) * inv, __uint_as_float(o1[c + 7]) * inv);
                    *reinterpret_cast<uint4*>(dst + 32 + c) = w;
                }
            }
            if (tr) AT_STAMP(tr_role);                                   // tile stored
        };
        int pend_t = -1;
        float pend_l = 0.f, pend_m = 0.f;
#pragma unroll 1
        for (int n = grp; n < C::NBLK; n += G) {
            const int t = n / C::NKB, j = n - t * C::NKB;
            const uint32_t k = n % NBUF, u = n / NBUF;                   // S buffer and how often it has been used before
            // A parity wait only tells the current phase from the previous one, so before waiting for phase u of S_FULL[k] the
            // group must know that phase u - 1 (the buffer's previous use, block n - NBUF) has completed.
            //  * NBUF a multiple of G: the previous use was this group's own block.
            //  * otherwise (NBUF = 1, G = 2: two blocks in all): go through phase u - 1 first; S(n) cannot be complete yet,
            //    it needs the P V product of block n - NBUF >= n - G + 1, i.e. of a block not older than this group's last.
            if ((NBUF % G) != 0 && u > 0) mbar_wait(&bars[B_SFULL + k], (u - 1) & 1);
            mbar_wait(&bars[B_SFULL + k], u & 1);
            tcgen05_fence_after();
            if (tr) AT_STAMP(tr_role);                                   // S full
            const uint32_t ta = tlane + k * C::S_COLS;
            constexpr int FULL = KB / 32 * 32;                           // columns swept 32 at a time; 16-column tail (KB = 144)
            constexpr int NCH = FULL / 32;
            // ---- row maximum of this block (first sweep over the S tile; the next chunk's load is in flight while one is reduced)
            float bm0 = -INFINITY, bm1 = -INFINITY;
            {
                uint32_t va[32], vb[32];
                tmem_ld_32x32(ta, va);
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    tmem_ld_wait();
                    if (ch + 1 < NCH) {
                        if (ch & 1) tmem_ld_32x32(ta + (ch + 1) * 32, va);
                        else tmem_ld_32x32(ta + (ch + 1) * 32, vb);
                    }
                    const uint32_t(&v)[32] = (ch & 1) ? vb : va;
#pragma unroll
                    for (int i = 0; i < 32; i += 2) {
                        bm0 = fmaxf(bm0, __uint_as_float(v[i]));
                        bm1 = fmaxf(bm1, __uint_as_float(v[i + 1]));
                    }
                }
                if (FULL < KB) {
                    uint32_t v[16];
                    tmem_ld_32x16(ta + FULL, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; i += 2) {
                        bm0 = fmaxf(bm0, __uint_as_float(v[i]));
                        bm1 = fmaxf(bm1, __uint_as_float(v[i + 1]));
                    }
                }
            }
            const float bm = fmaxf(bm0, bm1);
            if (tr) AT_STAMP(tr_role);                                   // block maximum known
            // ---- the maximum this row is expressed in: the previous block's, unless this block's exceeds it by > 2^8
            float m_use = bm, o_scale = 1.0f;
            // The row maximum travels from block n - 1 to block n through M_READY[(n - 1) % G]: one barrier per PRODUCING
            // group, so that its only waiter - the next group - sees every phase of it.  With a single barrier for all blocks
            // a group of G >= 3 skipped two phases between its waits, and a parity wait posted while the barrier was still
            // two phases behind returned at once: stale maximum, arrivals in the wrong phase and, eventually, a stalled
            // scheduler (seen once in a VAE decode, never in the unit tests).
            if (n > 0) mbar_wait(&bars[B_MREADY + (n - 1) % G], ((n - 1) / G) & 1);
            if (j > 0) {
                const float m_prev = sM[row];
                if ((bm - m_prev) * sl2 > AT_LAZY) o_scale = ex2_approx((m_prev - bm) * sl2);
                else m_use = m_prev;
            }
            sM[row] = m_use;
            mbar_arrive(&bars[B_MREADY + n % G]);
            if (tr) AT_STAMP(tr_role);                                   // row maximum handed on
            if (j < G) {                                                 // this group's first block of the tile (its blocks are G apart)
                l = 0.f;
                m_mine = m_use;
            }
            if (m_use != m_mine) {                                       // the row's reference moved since this thread's last block
                l *= ex2_approx((m_mine - m_use) * sl2);
                m_mine = m_use;
            }
            if (j > 0 && __any_sync(0xffffffffu, o_scale != 1.0f)) {
                // rare: this block raised the row maximum by more than 2^8 - rescale the row's partial output once the
                // previous P V product has completed (its commit on the S_FREE of its buffer), before the next one
                // accumulates onto it
                mbar_wait(&bars[B_SFREE + (n - 1) % NBUF], ((n - 1) / NBUF) & 1);
                tcgen05_fence_after();
                const uint32_t to = tlane + C::TM_O + (t % C::OBUF) * 64;
#pragma unroll
                for (int c = 0; c < 64; c += 32) {
                    uint32_t o[32];
                    tmem_ld_32x32(to + c, o);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * o_scale);
                    tmem_st_32x32(to + c, o);
                }
            }
            // ---- exponentials (second sweep): 32 S columns in, 16 P columns (bf16 pairs) out over the columns just read; the
            // next chunk's load is issued before the current one is exponentiated
            const float mo = m_use * sl2;
            float l0 = 0.f, l1 = 0.f, l2 = 0.f, l3 = 0.f;                // independent partial sums (no serial FADD chain)
            {
                uint32_t va[32], vb[32];
                tmem_ld_32x32(ta, va);
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    tmem_ld_wait();
                    if (ch + 1 < NCH) {
                        if (ch & 1) tmem_ld_32x32(ta + (ch + 1) * 32, va);
                        else tmem_ld_32x32(ta + (ch + 1) * 32, vb);
                    } else if (FULL < KB) {
                        // (tail handled below with its own load)
                    }
                    const uint32_t(&v)[32] = (ch & 1) ? vb : va;
                    uint32_t pk[16];
#pragma unroll
                    for (int i = 0; i < 32; i += 4) {
                        const float p0 = ex2_approx(__uint_as_float(v[i]) * sl2 - mo), p1 = ex2_approx(__uint_as_float(v[i + 1]) * sl2 - mo);
                        const float p2 = ex2_approx(__uint_as_float(v[i + 2]) * sl2 - mo), p3 = ex2_approx(__uint_as_float(v[i + 3]) * sl2 - mo);
                        l0 += p0; l1 += p1; l2 += p2; l3 += p3;          // fp32 sum of the unrounded probabilities
                        pk[i / 2] = pack_bf16x2(p0, p1);
                        pk[i / 2 + 1] = pack_bf16x2(p2, p3);
                    }
                    tmem_st_32x16(ta + ch * 16, pk);
                }
                if (FULL < KB) {
                    uint32_t v[16], pk[8];
                    tmem_ld_32x16(ta + FULL, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 16; i += 4) {
                        const float p0 = ex2_approx(__uint_as_float(v[i]) * sl2 - mo), p1 = ex2_approx(__uint_as_float(v[i + 1]) * sl2 - mo);
                        const float p2 = ex2_approx(__uint_as_float(v[i + 2]) * sl2 - mo), p3 = ex2_approx(__uint_as_float(v[i + 3]) * sl2 - mo);
                        l0 += p0; l1 += p1; l2 += p2; l3 += p3;
                        pk[i / 2] = pack_bf16x2(p0, p1);
                        pk[i / 2 + 1] = pack_bf16x2(p2, p3);
                    }
                    tmem_st_32x8(ta + FULL / 2, pk);
                }
            }
            l += (l0 + l1) + (l2 + l3);
            tmem_st_wait();
            tcgen05_fence_before();
            mbar_arrive(&bars[B_PREADY + k]);                            // P(n) is in tensor memory
            if (tr) AT_STAMP(tr_role);                                   // P written
            // ---- end of this group's work on the tile
            if (pend_t >= 0) {                                           // the tile this group finished one block ago: its O is complete by now
                // (before the hand-off below: L_READY must not complete its next phase while a thread of this group still
                // waits for the previous one - a parity wait cannot tell them apart)
                epilogue(pend_t, pend_l, pend_m);
                pend_t = -1;
            }
            if (C::L_PUBLISHERS > 0 && j != C::NKB - 1 && j + G >= C::NKB) {
                // this group's last block of the tile, and another group finishes the tile: hand it our share of the row sum
                sL[((t & 1) * G + grp) * AT_QTILE + row] = make_float2(l, m_mine);
                mbar_arrive(&bars[B_LREADY]);
            }
            if (j == C::NKB - 1) {
                // This group owns the epilogue of tile t.  With two O buffers it is deferred until after the group's next
                // block: waiting here for the last P V product would hold up the other group through the row-maximum chain.
                if (C::OBUF == 2 && n + G < C::NBLK) { pend_t = t; pend_l = l; pend_m = m_mine; }
                else epilogue(t, l, m_mine);
            }
        }
        } else if (warp == AT_SOFTMAX_WARPS) {
        // =========================================================================== MMA issuer (one warp, one elected lane)
        // WARP-UNIFORM control flow: all 32 lanes run the scheduler and probe the barriers, the decisions are made uniform
        // with a vote and elect.sync picks the lane that issues.  Inside `if (lane == 0)` the compiler keeps descriptors and
        // addresses in vector registers and moves them to uniform registers per tcgen05.mma: ~106 instead of ~76 cycles per
        // small MMA, and every barrier probe of the lone thread ~170 cycles (scripts/probe_umma_chunks.cu) - the P V product
        // is 12 MMAs of 61 cycles per block, so the issuing thread was the limiter.
        {
            constexpr uint32_t idesc_s = umma_idesc_bf16(AT_QTILE, KB);              // S = Q K^T: both operands K-major
            constexpr uint32_t idesc_o = idesc_bf16_bmn(AT_QTILE, 64);               // O = P V: V MN-major
            constexpr int PV_STEPS = KB / 16;
            uint32_t n_dbg = 0;
            const bool dbg_pv = (reinterpret_cast<uintptr_t>(trace) & 8) != 0;      // GTAV_ATTN_TRACE address + 8: time every P V product
            const uint64_t desc_q0 = umma_desc_sw128(smem_u32(sQ)), desc_k0 = umma_desc_sw128(smem_u32(sK));
            const uint64_t desc_v0 = umma_desc_sw128(smem_u32(sV));
            auto ready_pv = [&](int n) -> bool {                 // O += P(n) V: needs P written (and, first block of a tile, O read out)
                const int t = n / C::NKB, j = n - t * C::NKB;
                const uint32_t k = n % NBUF, ob = t % C::OBUF;
                if (j == 0 && t >= C::OBUF && !mbar_test(&bars[B_OFREE + ob], (t / C::OBUF - 1) & 1)) return false;
                return mbar_test(&bars[B_PREADY + k], (n / NBUF) & 1);
            };
            auto issue_pv = [&](int n) {
                const int t = n / C::NKB, j = n - t * C::NKB;
                const uint32_t k = n % NBUF, ob = t % C::OBUF;
                tcgen05_fence_after();
                const uint32_t d = tmem_base + C::TM_O + ob * 64;
                const uint32_t pa = tmem_base + k * C::S_COLS;                   // P(n): 8 columns per K step of 16 keys
                // B descriptors = a base built once + compile-time offsets (16-byte units)
                const uint64_t db0 = desc_v0 + static_cast<uint64_t>(j * (KB * AT_ROWB / 16));
                if (elect_one()) {
                    AT_STAMP(1);                   // P ready
#pragma unroll
                    for (int ks = 0; ks < PV_STEPS; ++ks)
                        umma_bf16_ts(d, pa + ks * 8, db0 + ks * (16 * AT_ROWB / 16), idesc_o, (j | ks) != 0 ? 1u : 0u);
                    umma_commit(&bars[B_SFREE + k]);                             // S buffer (and the P inside it) consumed
                    if (j == C::NKB - 1) umma_commit(&bars[B_OFULL + ob]);
                    if (trace != nullptr && dbg_pv) {  // profiling only: time the product itself
                        umma_commit(&bars[B_DBG]);
                        mbar_wait(&bars[B_DBG], n_dbg++ & 1);
                        AT_STAMP(1);               // P V done
                    }
                }
                __syncwarp();
            };
            auto ready_s = [&](int n) -> bool {                  // S(n) = Q K^T: needs the query tile staged and the S buffer consumed
                const int t = n / C::NKB, j = n - t * C::NKB;
                const uint32_t k = n % NBUF;
                if (j == 0 && !mbar_test(&bars[B_QFULL + (t & 1)], (t >> 1) & 1)) return false;
                if (n >= NBUF && !mbar_test(&bars[B_SFREE + k], (n / NBUF - 1) & 1)) return false;
                return true;
            };
            auto issue_s = [&](int n) {
                const int t = n / C::NKB, j = n - t * C::NKB;
                const uint32_t k = n % NBUF;
                tcgen05_fence_after();
                const uint32_t d = tmem_base + k * C::S_COLS;
                const uint64_t da0 = desc_q0 + static_cast<uint64_t>((t & 1) * (C::Q_BYTES / 16));
                const uint64_t db0 = desc_k0 + static_cast<uint64_t>(j * (KB * AT_ROWB / 16));
                if (elect_one()) {
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) umma_bf16_ss(d, da0 + 2 * kk, db0 + 2 * kk, idesc_s, kk != 0 ? 1u : 0u);
                    umma_commit(&bars[B_SFULL + k]);
                    if (j == C::NKB - 1) umma_commit(&bars[B_QFREE + (t & 1)]);      // last read of this query tile
                    AT_STAMP(1);                   // S(n) issued
                }
                __syncwarp();
            };
            // Whichever of the two next products has its operands ready is issued, S first: an S tile must not queue behind
            // a P V product that is still waiting for its probabilities - the softmax group that owns the buffer would sit
            // idle for that long.  Non-blocking probes (mbarrier.test_wait): try_wait may suspend the thread for a
            // microsecond while the OTHER product became ready.
            int next_s = 0, next_pv = 0;
            uint32_t idle = 0;
            while (next_pv < C::NBLK) {
                bool did = false;
                if (next_s < C::NBLK && __all_sync(0xffffffffu, ready_s(next_s))) {
                    issue_s(next_s);
                    ++next_s;
                    did = true;
                } else if (next_pv < next_s && __all_sync(0xffffffffu, ready_pv(next_pv))) {
                    issue_pv(next_pv);
                    ++next_pv;
                    did = true;
                }
                if (did) idle = 0;
                else if (++idle > (1u << 26)) {
                    if (lane == 0) printf("gtav: attention MMA scheduler stalled (block %d)\n", blockIdx.x);
                    __trap();
                }
            }
        }
    } else {
        // =========================================================================== query-tile loaders
        const int lt = threadIdx.x - KV_THREADS;                         // 0 .. 63: chunk lt % 8 of rows lt / 8, lt / 8 + 8, ...
        const int c = lt & 7;
#pragma unroll 1
        for (int t = 0; t < C::QTILES; ++t) {
            if (t >= 2) mbar_wait(&bars[B_QFREE + (t & 1)], ((t >> 1) - 1) & 1);
            if (lt == 0) AT_STAMP(2);              // slot free
            if (t > 0) {                           // (tile 0 was staged next to the K / V staging, before the set-up barrier)
                uint8_t* dstq = sQ + (t & 1) * C::Q_BYTES;
                constexpr int RS = AT_LOADER_WARPS * 4, MAXR = AT_QTILE / RS;
                stage_rows<ROT_PAIRS, RS, MAXR, MAXR / 2>(dstq, qbase, nullptr, nullptr, ld, lt >> 3, c, AT_QTILE, t * AT_QTILE, SEQ, rot);
                fence_proxy_async_smem();
            }
            mbar_arrive(&bars[B_QFULL + (t & 1)]);
            if (lt == 0) AT_STAMP(2);              // staged
        }
    }
    // ---- all roles done: the last tile's epilogue has read O, every MMA has completed (o_full was waited on)
    tcgen05_fence_before();
    __syncthreads();
    if (threadIdx.x == 0) AT_STAMP(0);             // end
    if (warp == AT_SOFTMAX_WARPS) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, C::TM_COLS);
    }
#undef AT_STAMP
}

template <int SEQ, int KB, int NBUF, int TMC, int G, int ROT_PAIRS>
int launch_tc(const bf16* qkv, bf16* out, int groups, int heads, const float2* rot, cudaStream_t s) {
    using C = AttnCfg<SEQ, KB, NBUF, TMC, G>;
    static bool configured = false;
    auto kern = attn_tc_kernel<SEQ, KB, NBUF, TMC, G, ROT_PAIRS>;
    if (!configured) {
        GTAV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
        configured = true;
    }
    // GTAV_ATTN_TRACE=<device address of [CTAs][4][64] int64, + 8 to also time every P V product>: scripts/trace_attn.py
    long long* trace = nullptr;
    if (const char* e = getenv("GTAV_ATTN_TRACE")) trace = reinterpret_cast<long long*>(strtoull(e, nullptr, 0));
    GTAV_CUDA_OK(launch_k(kern, dim3(groups * heads), dim3(at_threads(G)), C::SMEM, s, qkv, out, heads, rot, trace));
    return 0;
}

}  // namespace

// seq 576 / rot_pairs 16: VAE attention; seq 144 / rot_pairs 32: DiT spatial attention.
int launch_attention_tc(const bf16* qkv, bf16* out, int groups, int seq, int heads, const float2* rot, int rot_pairs,
                        cudaStream_t s) {
    if (groups <= 0) return 0;
    if (seq == 576 && rot_pairs == 16) {
        // 4 key blocks of 144 keys per query tile in THREE S buffers, one softmax warpgroup per buffer (480 threads): a
        // group's next S tile is computed while it works on the current one, instead of waiting for its own P V product to
        // release one of two buffers.  32 frames: 122.8 us against 131.8 us for 3 blocks of 192 keys in 2 buffers with 2
        // groups; 6 blocks of 96 keys in 4 buffers: 146 us with 2 groups, 146 us with 4 - the per-block hand-offs cost more
        // than the extra buffers save.  144 keys x 3 buffers with TWO groups (a spare buffer per group, so no group ever
        // waits for its own P V product): 132 us - the third buffer alone buys nothing, the third group's instruction issue
        // does.
        return launch_tc<576, 144, 3, 512, 3, 16>(qkv, out, groups, heads, rot, s);
    }
    // S = 144: one S buffer and one O buffer in 256 TMEM columns, 72 KB of shared memory -> two CTAs per SM hide each other's
    // staging and hand-off latencies (one CTA has only two (tile, block) steps to pipeline)
    if (seq == 144 && rot_pairs == 32) return launch_tc<144, 144, 1, 256, 2, 32>(qkv, out, groups, heads, rot, s);
    set_error("attention (tcgen05): unsupported (seq=%d, rot_pairs=%d); built for (144,32) and (576,16)", seq, rot_pairs);
    return -1;
}

}  // namespace gtav
