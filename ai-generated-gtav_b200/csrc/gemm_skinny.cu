// Weight-streaming bf16 GEMM for the last-frame DiT step: out[T,N] = epilogue(A[T,K] @ W[N,K]^T) with very
// few token rows (T = 144 per rollout, at most 3 rollouts per call) and large weights.
//
// Same reference ops as gemm_sm100.cu (to_qkv / to_out / Mlp.fc1 / Mlp.fc2 of reference
// model/attention.py:27-28,86-87 and model/dit.py:171-198) - this is the shape they take once the
// context frames' K/V are cached and only the frame being denoised is recomputed (M = 144*B).
// At that size the op is bound by moving bytes (W from HBM, A and the split-K partials through L2) and by the
// latency chain of its phases, not by the tensor pipe, so the kernel is organised around getting all SMs to pull
// bytes at once and around overlapping consecutive launches:
//   * operands are swapped: the UMMA "M" side is a block of 128 weight rows, the "N" side one
//     144-token frame tile (a legal UMMA N, no padding), accumulator D[128 x 144] fp32 in TMEM;
//   * K is split over S CTAs per weight-row block so that (N/128)*S ~ the SM count; the W slab is ONE TMA box
//     (3-D box spanning all its 64-wide K chunks: several small boxes per operand measured slower, bench_graph.py);
//   * the W slab is requested before griddepcontrol.wait (weights do not depend on the previous kernel).  Measured
//     alternatives for the operand loads, all slower in the real step (profiles/r01/bench_engine_v6.log): 2 / 4 boxes
//     per operand from different warps (+1 % / +8 % step time: every extra TMA instruction costs), the token slab
//     through cp.async with a software swizzle next to the TMA-loaded weights (+6 %);
//   * partial accumulators go to an fp32 workspace (L2) and each of the S CTAs of a row block reduces + runs the fused
//     epilogue for its 1/S share of the tokens, summing the partials in split order (deterministic).  How a CTA knows
//     that the others' partial sums are there: in the engine's passes every element carries the launch's parity in its
//     last mantissa bit and is its own ready flag (SkTag below: no fence, counter, poll or CTA barrier); stand-alone
//     calls and GTAV_SK_TAG=0 release the stores with one gpu-scope fence of the arriving thread after a CTA barrier
//     and meet on a counter;
//   * optionally the reduce is done per token row by every CTA (plus reduce-only CTAs up to one per token), which lets
//     the row-wise kernel that would follow - LayerNorm + modulate, or the last-frame temporal attention - run inside
//     it; everything those need besides the partial sums is loaded BEFORE the partial sums.
// Warp roles (256 threads): 0 = W producer, 1 = A producer, 2 = TMEM allocator + MMA issue (warp-uniform loop, elect.sync); all 8 warps drain the
// accumulator (one TMEM lane quadrant each, half of the columns) and reduce.
#include "attn_temporal_core.cuh"
#include "common.cuh"
#include "kernels.h"
#include "ln_row.cuh"

namespace gtav {

static constexpr int SK_THREADS = 256;
static constexpr int SK_NT = 144;                  // tokens per tile (one frame)
static constexpr int SK_W_CHUNK = 128 * 128;       // bytes: 128 weight rows x 64 bf16
static constexpr int SK_A_CHUNK = SK_NT * 128;     // bytes: 144 tokens x 64 bf16
static constexpr int SK_SMEM_BUDGET = 200 * 1024;  // operand bytes per CTA
static constexpr int SK_TAIL_BYTES = 128 + 4096 + 2048;   // barriers | shift + scale of the fused LayerNorm | one bf16 row
static constexpr int SK_TMAX = 7;                  // cached context frames of the fused temporal attention

struct SkinnyParams {
    GemmParams g;
    SkinnyFuseParams f;    // what the reduce produces besides / instead of the Linear's output (FUSE template parameter)
    int splits, chunks, tiles;
    int gemm_ctas;         // (N/128) * splits; CTAs beyond that (fused modes) only take part in the per-token reduce
    float* ws;
    int* counters;
    int tag;               // 0: rendezvous protocol; 2 | parity: tagged partial sums (see SkTag)
    long long* trace;      // optional [gridDim.x][8] globaltimer stamps (ns) of the phase boundaries; null in production
};

// Tagged partial sums: the exchange without fence, counter and poll.  The producer clears the lowest mantissa bit of every
// fp32 partial sum and writes the launch's parity there; the consumer loads straight away and accepts an element once it
// carries that parity, re-loading the ones that do not yet - every 4-byte element is its own ready flag, so no ordering
// between elements is needed (relaxed gpu-scope stores and loads, L2 is the meeting point; ld.global.cg in the retry loop
// never sees the other CTAs' stores, DESIGN.md 5b).  Stale elements always carry the other parity because the caller
// (dit_engine.cu) gives each GEMM kind its own workspace, zeroed once, and alternates the parity along the launches that
// share it: 1, 0, 1, 0 ... with an even number per pass.  Against the rendezvous protocol this
// removes the gpu-scope fence after the stores, the atomic arrival, the polling round trip and two CTA barriers from the
// critical path of every launch.  The sums lose their last mantissa bit (2^-24 relative, far below the bf16 rounding of the
// Linear's output) and stay deterministic: summed in split order as before.  chk = 0: untagged, every element is accepted.
static constexpr int SK_TAG_DELAY = 600;           // SM clocks between a warp's last partial store and its first reduce load
struct SkTag {
    uint32_t chk, par;
};
__device__ __forceinline__ bool tag_ok(uint32_t x, SkTag t) { return ((x ^ t.par) & t.chk) == 0u; }
__device__ __forceinline__ bool tag_ok(uint2 v, SkTag t) { return (((v.x ^ t.par) | (v.y ^ t.par)) & t.chk) == 0u; }
__device__ __forceinline__ bool tag_ok(uint4 v, SkTag t) {
    return (((v.x ^ t.par) | (v.y ^ t.par) | (v.z ^ t.par) | (v.w ^ t.par)) & t.chk) == 0u;
}
__device__ __forceinline__ uint32_t ld_relaxed_u1(const float* p) {
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint2 ld_relaxed_u2(const float* p) {
    uint2 v;
    asm volatile("ld.relaxed.gpu.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint4 ld_relaxed_u4(const float* p) {
    uint4 v;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u1(float* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void tag_spin_check(uint32_t& spins) {
    if (++spins > (1u << 21)) __trap();          // a protocol bug (parity out of step) fails the launch instead of hanging
}

__device__ __forceinline__ long long globaltimer_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define SK_STAMP(slot)                                                                     \
    do {                                                                                   \
        if (p.trace != nullptr) p.trace[static_cast<size_t>(blockIdx.x) * 8 + (slot)] = globaltimer_ns(); \
    } while (0)

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// Rendezvous of the n CTAs of a group (one thread per CTA) on grp[0..3] = {count A, count B, which, -}, all zero before
// the first launch.  `which` (read by the caller BEFORE this CTA's arrival, any time after griddepcontrol.wait - the flip
// needs every CTA's arrival, so the value read cannot be the flipped one) selects the counter this launch counts on; the
// other one still holds the previous launch's total and is cleared here, and `which` is flipped for the next launch, by
// every CTA that gets through (same values from everyone: plain stores, nobody waits for them).  So an arrival is one
// fire-and-forget reduction plus polling, and the kernel's exit path carries no atomic round trip (the former
// departure counter cost ~0.7 us per launch; a returning atomicAdd on arrival costs the same: scripts/trace_step.py).
// The caller has made its partial sums visible (fence + CTA barrier) before arriving.
__device__ __forceinline__ void skinny_rendezvous(int* grp, int n, int which) {
    int* cnt = grp + (which & 1);
    asm volatile("red.relaxed.gpu.global.add.s32 [%0], 1;" ::"l"(cnt) : "memory");
    uint32_t spins = 0;
    while (ld_acquire_gpu(cnt) < n) {
        // (no back-off: one polling thread per CTA, the wake-up latency is on the critical path of every launch)
        if (++spins > (1u << 24)) __trap();    // a protocol bug fails the launch instead of hanging the GPU
    }
    *reinterpret_cast<volatile int*>(grp + ((which & 1) ^ 1)) = 0;
    *reinterpret_cast<volatile int*>(grp + 2) = (which & 1) ^ 1;
}
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}

// One output element: column n (this thread's weight row), token `tok`, fp32 pre-bias value `acc`.
template <int EPI>
__device__ __forceinline__ void skinny_store(const GemmParams& g, int tok, int n, float acc, float bias_n) {
    float y = acc;
    if (EPI != EPI_STORE) y += bias_n;
    y = bf16_round(y);                                           // the Linear's own bf16 output
    if (EPI == EPI_BIAS_GELU_TANH) {
        y = gelu_tanh_f(y);
    } else if (EPI == EPI_BIAS_GATE_RES) {
        int f = tok / g.rows_per_frame;
        if (g.frame_row != nullptr) f = g.frame_row[f];
        const float gt = __bfloat162float(g.gate[static_cast<size_t>(f) * g.gate_ld + n]);
        const float r = __bfloat162float(g.res[static_cast<size_t>(tok) * g.ldr + n]);
        y = r + bf16_round(gt * y);
    }
    g.out[static_cast<size_t>(tok) * g.ldo + n] = __float2bfloat16_rn(y);
}

// The epilogue's vector operands for four consecutive output columns n..n+3 of one token (packed bf16).
struct Epi4Ops {
    uint2 bias, gate, res;
};
template <int EPI>
__device__ __forceinline__ Epi4Ops skinny_epi4_load(const GemmParams& g, int tok, int n) {
    Epi4Ops o;
    o.bias = o.gate = o.res = make_uint2(0u, 0u);
    if (EPI != EPI_STORE) o.bias = *reinterpret_cast<const uint2*>(g.bias + n);
    if (EPI == EPI_BIAS_GATE_RES) {
        int f = tok / g.rows_per_frame;
        if (g.frame_row != nullptr) f = g.frame_row[f];
        o.gate = *reinterpret_cast<const uint2*>(g.gate + static_cast<size_t>(f) * g.gate_ld + n);
        o.res = *reinterpret_cast<const uint2*>(g.res + static_cast<size_t>(tok) * g.ldr + n);
    }
    return o;
}
// Four consecutive output columns of one token (split-K reduce path): the epilogue's bf16 results, packed.
template <int EPI>
__device__ __forceinline__ uint2 skinny_epi4(float4 acc, const Epi4Ops& e) {
    float y[4] = {acc.x, acc.y, acc.z, acc.w};
    if (EPI != EPI_STORE) {
        const float2 b0 = unpack_bf16x2(e.bias.x), b1 = unpack_bf16x2(e.bias.y);
        y[0] += b0.x; y[1] += b0.y; y[2] += b1.x; y[3] += b1.y;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) y[j] = bf16_round(y[j]);
    if (EPI == EPI_BIAS_GELU_TANH) {
#pragma unroll
        for (int j = 0; j < 4; ++j) y[j] = gelu_tanh_f(y[j]);
    } else if (EPI == EPI_BIAS_GATE_RES) {
        const float2 g0 = unpack_bf16x2(e.gate.x), g1 = unpack_bf16x2(e.gate.y), r0 = unpack_bf16x2(e.res.x), r1 = unpack_bf16x2(e.res.y);
        y[0] = r0.x + bf16_round(g0.x * y[0]);
        y[1] = r0.y + bf16_round(g0.y * y[1]);
        y[2] = r1.x + bf16_round(g1.x * y[2]);
        y[3] = r1.y + bf16_round(g1.y * y[3]);
    }
    uint2 o;
    o.x = pack_bf16x2(y[0], y[1]);
    o.y = pack_bf16x2(y[2], y[3]);
    return o;
}
// Not inlined: the reduce below calls it from up to 5 x 4 unrolled sites, and with the GELU epilogue inlined everywhere
// the kernel grew to 50 KB of SASS - instruction fetch shows up in the ncu stall reasons of these ~9 us kernels.
template <int EPI>
__device__ __noinline__ void skinny_store4(const GemmParams& g, int tok, int n, float4 acc, uint2 bias) {
    Epi4Ops e;
    if (EPI == EPI_BIAS_GATE_RES) e = skinny_epi4_load<EPI>(g, tok, n);
    e.bias = bias;
    *reinterpret_cast<uint2*>(g.out + static_cast<size_t>(tok) * g.ldo + n) = skinny_epi4<EPI>(acc, e);
}

// Sum the S partial tiles of this row block for tokens lo + wid, lo + wid + 8, ... (one warp per token, lane = 4
// consecutive weight rows) in split order and run the epilogue.  S is a template parameter so that all S loads of a
// token are in flight together: the loop is otherwise a chain of exposed L2 latencies.  bias: this lane's four
// columns, loaded by the caller before the rendezvous.
template <int EPI, int S>
__device__ __forceinline__ void skinny_reduce(const GemmParams& g, const float* part, int total, int lo, int hi, int wid, int lane,
                                              int n0, uint2 bias, SkTag tg) {
    static_assert(S <= 4, "the unrolled reduce is instantiated for S = 4 only; other split counts use skinny_reduce_any");
    const float* base = part + 4 * lane;
    const uint32_t keep = ~tg.chk;
    // few splits: a warp's tokens (at most 5 per 144-token tile share) are loaded together, so the whole reduce costs
    // one L2 round trip instead of one per token (tagged: plus one per round of elements that had not arrived yet)
    constexpr int IT = 5;
#pragma unroll 1
    for (int t0 = lo + wid; t0 < hi; t0 += 8 * IT) {
        // first attempt: every load of the warp's tokens back to back; then only what had not arrived yet is loaded again
        uint4 v[IT][S];
        uint32_t pending = 0u, spins = 0u;
#pragma unroll
        for (int it = 0; it < IT; ++it)
#pragma unroll
            for (int s2 = 0; s2 < S; ++s2)
                if (t0 + 8 * it < hi) v[it][s2] = ld_relaxed_u4(base + (static_cast<size_t>(s2) * total + t0 + 8 * it) * 128);
#pragma unroll
        for (int it = 0; it < IT; ++it)
#pragma unroll
            for (int s2 = 0; s2 < S; ++s2)
                if (t0 + 8 * it < hi && !tag_ok(v[it][s2], tg)) pending |= 1u << (S * it + s2);
        while (pending) {                          // (all missing loads in flight together, then the checks)
            tag_spin_check(spins);
#pragma unroll
            for (int it = 0; it < IT; ++it)
#pragma unroll
                for (int s2 = 0; s2 < S; ++s2)
                    if (pending >> (S * it + s2) & 1u) v[it][s2] = ld_relaxed_u4(base + (static_cast<size_t>(s2) * total + t0 + 8 * it) * 128);
#pragma unroll
            for (int it = 0; it < IT; ++it)
#pragma unroll
                for (int s2 = 0; s2 < S; ++s2)
                    if ((pending >> (S * it + s2) & 1u) && tag_ok(v[it][s2], tg)) pending &= ~(1u << (S * it + s2));
        }
#pragma unroll
        for (int it = 0; it < IT; ++it) {
            const int tok = t0 + 8 * it;
            if (tok < hi) {
                float4 acc = make_float4(__uint_as_float(v[it][0].x & keep), __uint_as_float(v[it][0].y & keep),
                                         __uint_as_float(v[it][0].z & keep), __uint_as_float(v[it][0].w & keep));
#pragma unroll
                for (int s2 = 1; s2 < S; ++s2) {
                    acc.x += __uint_as_float(v[it][s2].x & keep); acc.y += __uint_as_float(v[it][s2].y & keep);
                    acc.z += __uint_as_float(v[it][s2].z & keep); acc.w += __uint_as_float(v[it][s2].w & keep);
                }
                skinny_store4<EPI>(g, tok, n0 + 4 * lane, acc, bias);
            }
        }
    }
}

// Sum of the S partials at p0, p0 + stride, ... in split order, all loads in flight together.
template <int S>
__device__ __forceinline__ float4 skinny_sum4(const float* p0, size_t stride, SkTag tg) {
    uint4 v[S];
    const uint32_t keep = ~tg.chk;
    uint32_t pending = 0u, spins = 0u;
#pragma unroll
    for (int s2 = 0; s2 < S; ++s2) v[s2] = ld_relaxed_u4(p0 + s2 * stride);
#pragma unroll
    for (int s2 = 0; s2 < S; ++s2)
        if (!tag_ok(v[s2], tg)) pending |= 1u << s2;
    while (pending) {                              // only what had not arrived yet is loaded again
        tag_spin_check(spins);
#pragma unroll
        for (int s2 = 0; s2 < S; ++s2)
            if (pending >> s2 & 1u) v[s2] = ld_relaxed_u4(p0 + s2 * stride);
#pragma unroll
        for (int s2 = 0; s2 < S; ++s2)
            if ((pending >> s2 & 1u) && tag_ok(v[s2], tg)) pending &= ~(1u << s2);
    }
    float4 acc = make_float4(__uint_as_float(v[0].x & keep), __uint_as_float(v[0].y & keep), __uint_as_float(v[0].z & keep),
                             __uint_as_float(v[0].w & keep));
#pragma unroll
    for (int s2 = 1; s2 < S; ++s2) {
        acc.x += __uint_as_float(v[s2].x & keep); acc.y += __uint_as_float(v[s2].y & keep);
        acc.z += __uint_as_float(v[s2].z & keep); acc.w += __uint_as_float(v[s2].w & keep);
    }
    return acc;
}
// Any split count: one token per warp at a time, partials summed in split order, up to 16 loads in flight.
template <int EPI>
__device__ __forceinline__ void skinny_reduce_any(const GemmParams& g, const float* part, int S, int total, int lo, int hi, int wid,
                                                  int lane, int n0, uint2 bias, SkTag tg) {
    const float* base = part + 4 * lane;
    const size_t stride = static_cast<size_t>(total) * 128;
#pragma unroll 1
    for (int tok = lo + wid; tok < hi; tok += 8) {
        const float* p0 = base + static_cast<size_t>(tok) * 128;
        float4 acc;
        switch (S) {
            case 2: acc = skinny_sum4<2>(p0, stride, tg); break;
            case 8: acc = skinny_sum4<8>(p0, stride, tg); break;
            default: acc = skinny_sum4<16>(p0, stride, tg); break;
        }
        skinny_store4<EPI>(g, tok, n0 + 4 * lane, acc, bias);
    }
}

// ---- fused reduces: the CTAs meet on ALL row-block counters and every CTA then owns whole token rows (token
// blockIdx.x, blockIdx.x + gridDim.x, ...), so that row-wise work that follows the Linear can run right here instead
// of in another kernel of the latency-bound last-frame chain.  Their operands other than the partial sums (epilogue
// vectors, modulation vectors, K/V cache) are loaded by the *_preload functions, which the kernel calls right after
// griddepcontrol.wait: by the time the rendezvous completes they are in registers / shared memory.
//
// SK_FUSE_LN (N = 1024, gated-residual epilogue: to_out and fc2 of reference model/dit.py:205-224): warp w sums the
// partials of row block w and writes its part of the new residual-stream row to g.out; the 8 warps then run the NEXT
// LayerNorm + modulate on the row together, each on its own 128 features, exchanging only the 8 segment sums of the
// two statistics passes through shared memory (ln_row.cuh: same bits as the stand-alone one-warp-per-row kernel).
// smod: 2 KB shift | 2 KB scale of the token's frame, filled cooperatively (thread i: 16 bytes).
__device__ __forceinline__ Epi4Ops skinny_ln_preload(const SkinnyParams& p, int tok, int warp, uint8_t* smod) {
    const GemmParams& g = p.g;
    const SkinnyFuseParams& f = p.f;
    int fr = tok / g.rows_per_frame;
    if (g.frame_row != nullptr) fr = g.frame_row[fr];
    const bf16* mrow = f.ln_mod + static_cast<size_t>(fr) * f.ln_mod_ld;
    const int i = threadIdx.x & 127;
    const uint4 m = *reinterpret_cast<const uint4*>(mrow + (threadIdx.x < 128 ? f.ln_shift_off : f.ln_scale_off) + i * 8);
    Epi4Ops e;
    const int n = warp * 128 + 4 * (threadIdx.x & 31);
    e.bias = *reinterpret_cast<const uint2*>(g.bias + n);
    e.gate = *reinterpret_cast<const uint2*>(g.gate + static_cast<size_t>(fr) * g.gate_ld + n);
    e.res = *reinterpret_cast<const uint2*>(g.res + static_cast<size_t>(tok) * g.ldr + n);
    *reinterpret_cast<uint4*>(smod + threadIdx.x * 16) = m;
    return e;
}
__device__ __forceinline__ void skinny_reduce_ln(const SkinnyParams& p, int S, int total, int warp, int lane, uint8_t* smod,
                                                 uint8_t* srow, Epi4Ops e, SkTag tg) {
    const GemmParams& g = p.g;
    const SkinnyFuseParams& f = p.f;
    const int n = warp * 128 + 4 * lane;
    const float* base = p.ws + static_cast<size_t>(warp) * S * total * 128 + 4 * lane;
    const size_t stride = static_cast<size_t>(total) * 128;
    float* sred = reinterpret_cast<float*>(srow);            // [2][8] segment sums (values, then squared deviations)
#pragma unroll 1
    for (int tok = blockIdx.x; tok < total; tok += gridDim.x) {
        const float* p0 = base + static_cast<size_t>(tok) * 128;
        float4 acc;
        switch (S) {                           // only the partial-sum loads depend on S: one copy of everything else
            case 4: acc = skinny_sum4<4>(p0, stride, tg); break;
            case 8: acc = skinny_sum4<8>(p0, stride, tg); break;
            default: acc = skinny_sum4<16>(p0, stride, tg); break;
        }
        const uint2 o = skinny_epi4<EPI_BIAS_GATE_RES>(acc, e);
        *reinterpret_cast<uint2*>(g.out + static_cast<size_t>(tok) * g.ldo + n) = o;
        // LayerNorm of the row held by the 8 warps (128 features each, one quad per lane) in the summation order ln_row.cuh
        // defines on exactly this layout - the stand-alone kernel reproduces it with one warp.  Two CTA barriers for the two
        // passes of the statistics instead of a round trip of the whole row through shared memory and one warp's serial work.
        const float2 x01 = unpack_bf16x2(o.x), x23 = unpack_bf16x2(o.y);
        const float x[4] = {x01.x, x01.y, x23.x, x23.y};
        const float s1 = warp_sum(ln_quad_sum(x[0], x[1], x[2], x[3]));
        if (lane == 0) sred[warp] = s1;
        __syncthreads();                       // (first time round this also publishes the preloaded shift / scale)
        const float mean = __fmul_rn(ln_combine8(sred[0], sred[1], sred[2], sred[3], sred[4], sred[5], sred[6], sred[7]), 1.0f / 1024);
        const float s2 = warp_sum(ln_quad_sq(x[0], x[1], x[2], x[3], mean));
        if (lane == 0) sred[8 + warp] = s2;
        __syncthreads();
        const float rstd = ln_rstd(ln_combine8(sred[8], sred[9], sred[10], sred[11], sred[12], sred[13], sred[14], sred[15]), 1024);
        const uint2 sh = *reinterpret_cast<const uint2*>(smod + n * 2);
        const uint2 sc = *reinterpret_cast<const uint2*>(smod + 2048 + n * 2);
        *reinterpret_cast<uint2*>(f.ln_out + static_cast<size_t>(tok) * 1024 + n) = ln_modulate_quad(x, mean, rstd, sh, sc);
        if (tok + static_cast<int>(gridDim.x) < total) {
            __syncthreads();                   // everyone is done with sred / smod before they are rewritten
            e = skinny_ln_preload(p, tok + gridDim.x, warp, smod);
        }
    }
}

// SK_FUSE_TATTN (N = 3072 = q | k | v of 16 heads, plain-store epilogue: to_qkv of the temporal half, reference
// model/attention.py:41-66): warp w sums the partials of heads 2w and 2w + 1 (row blocks w, 8 + w, 16 + w), lane =
// one rotary pair, and runs the last-frame temporal attention against the K/V cache with attn_temporal_last_kernel's
// own code; g.out receives the ATTENTION output [tokens, 1024] (the q/k/v row itself is not needed afterwards).
struct TattnPre {
    uint32_t kc[2][SK_TMAX], vc[2][SK_TMAX];
};
__device__ __forceinline__ void skinny_tattn_preload(const SkinnyParams& p, int tok, int warp, int lane, TattnPre& pre) {
    const SkinnyFuseParams& f = p.f;
    constexpr int D = 1024;
    const int P = f.positions, tc = f.ctx_frames;
    const int b = tok / P, pos = tok - b * P;
#pragma unroll
    for (int hh = 0; hh < 2; ++hh) {
        const bf16* cache = f.kv_cache + (static_cast<size_t>(b) * tc * P + pos) * (2 * D) + (2 * warp + hh) * 64 + 2 * lane;
        temporal_cache_load(pre.kc[hh], pre.vc[hh], tc, cache, static_cast<size_t>(P) * 2 * D, D);
    }
}
template <int S>
__device__ __forceinline__ void skinny_reduce_tattn(const SkinnyParams& p, int total, int warp, int lane, TattnPre& pre, SkTag tg) {
    const GemmParams& g = p.g;
    const uint32_t keep = ~tg.chk;
    const int tc = p.f.ctx_frames;
    const float2 cs = p.f.rot[tc * 32 + lane];
#pragma unroll 1
    for (int tok = blockIdx.x; tok < total; tok += gridDim.x) {
        uint2 a[2][3][S];
        uint32_t pending = 0u, spins = 0u;                                   // 6 S <= 24 loads
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int part = 0; part < 3; ++part) {
                const float* base = p.ws + (static_cast<size_t>(part * 8 + warp) * S * total + tok) * 128 + hh * 64 + 2 * lane;
#pragma unroll
                for (int s2 = 0; s2 < S; ++s2) a[hh][part][s2] = ld_relaxed_u2(base + static_cast<size_t>(s2) * total * 128);
            }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh)
#pragma unroll
            for (int part = 0; part < 3; ++part)
#pragma unroll
                for (int s2 = 0; s2 < S; ++s2)
                    if (!tag_ok(a[hh][part][s2], tg)) pending |= 1u << ((hh * 3 + part) * S + s2);
        while (pending) {                          // only what had not arrived yet is loaded again
            tag_spin_check(spins);
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int part = 0; part < 3; ++part) {
                    const float* base = p.ws + (static_cast<size_t>(part * 8 + warp) * S * total + tok) * 128 + hh * 64 + 2 * lane;
#pragma unroll
                    for (int s2 = 0; s2 < S; ++s2)
                        if (pending >> ((hh * 3 + part) * S + s2) & 1u) a[hh][part][s2] = ld_relaxed_u2(base + static_cast<size_t>(s2) * total * 128);
                }
#pragma unroll
            for (int hh = 0; hh < 2; ++hh)
#pragma unroll
                for (int part = 0; part < 3; ++part)
#pragma unroll
                    for (int s2 = 0; s2 < S; ++s2) {
                        const int bit = (hh * 3 + part) * S + s2;
                        if ((pending >> bit & 1u) && tag_ok(a[hh][part][s2], tg)) pending &= ~(1u << bit);
                    }
        }
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            float2 qkv[3];
#pragma unroll
            for (int part = 0; part < 3; ++part) {
                float2 acc = make_float2(__uint_as_float(a[hh][part][0].x & keep), __uint_as_float(a[hh][part][0].y & keep));
#pragma unroll
                for (int s2 = 1; s2 < S; ++s2) { acc.x += __uint_as_float(a[hh][part][s2].x & keep); acc.y += __uint_as_float(a[hh][part][s2].y & keep); }
                qkv[part] = make_float2(bf16_round(acc.x), bf16_round(acc.y));       // the Linear's bf16 output
            }
            *reinterpret_cast<uint32_t*>(g.out + static_cast<size_t>(tok) * g.ldo + (2 * warp + hh) * 64 + 2 * lane) =
                temporal_last_core(tc, qkv[0], qkv[1], qkv[2], pre.kc[hh], pre.vc[hh], cs);
        }
        if (tok + static_cast<int>(gridDim.x) < total) skinny_tattn_preload(p, tok + gridDim.x, warp, lane, pre);
    }
}

template <int EPI, int FUSE>
__global__ void __launch_bounds__(SK_THREADS, 1)
gemm_skinny_kernel(const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmA, const SkinnyParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int chunks = p.chunks, tiles = p.tiles, S = p.splits;
    uint8_t* sW = smem;
    uint8_t* sA = smem + chunks * SK_W_CHUNK;
    uint8_t* tail = sA + tiles * chunks * SK_A_CHUNK;
    uint64_t* bar_w = reinterpret_cast<uint64_t*>(tail);
    uint64_t* bar_a = bar_w + 1;                   // [tiles] (<= 3)
    uint64_t* bar_acc = bar_w + 6;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_w + 7);
    uint8_t* smod = tail + 128;                    // fused LayerNorm: shift | scale (4 KB), then one bf16 row (2 KB)
    uint8_t* srow = smod + 4096;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 128) SK_STAMP(0);                                       // kernel entry
    // fused modes launch extra CTAs that own token rows in the reduce but no tile of the GEMM
    const bool gemm_cta = FUSE == SK_FUSE_NONE || static_cast<int>(blockIdx.x) < p.gemm_ctas;
    const int rb = blockIdx.x / S, split = blockIdx.x - rb * S;
    const int kc0 = split * chunks;
    const int total = tiles * SK_NT;
    const uint32_t tmem_cols = total <= 256 ? 256u : 512u;
    const bool tagged = p.tag != 0;                // tagged partial sums instead of the counter rendezvous (SkTag)
    SkTag tg;
    tg.chk = tagged ? 1u : 0u;
    tg.par = tagged ? static_cast<uint32_t>(p.tag & 1) : 0u;

    // Both operand loads go out BEFORE the CTA-wide set-up barrier: thread 0 initialises the W barrier and requests the
    // W slab at once (weights do not depend on the previous kernel), warp 1 initialises the token-slab barriers, waits for
    // the previous kernel (griddepcontrol.wait) and requests the slab - neither needs the TMEM allocation that the
    // barrier below publishes, and the MMA thread first touches these barriers after it.
    if (gemm_cta && warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmW);
        mbar_init(bar_w, 1);
        mbar_init(bar_acc, 1);
        fence_barrier_init();
        mbar_arrive_expect_tx(bar_w, chunks * SK_W_CHUNK);
        tma_load_3d(sW, &tmW, bar_w, 0, rb * 128, kc0);
        SK_STAMP(1);                                                           // W requested
    }
    if (gemm_cta && warp == 1) {
        if (lane == 0) {
            tma_prefetch_desc(&tmA);
            for (int t = 0; t < 3; ++t) mbar_init(&bar_a[t], 1);
            fence_barrier_init();
        }
        pdl_wait();
        if (lane == 0) {
            for (int t = 0; t < tiles; ++t) {
                mbar_arrive_expect_tx(&bar_a[t], chunks * SK_A_CHUNK);
                tma_load_3d(sA + t * chunks * SK_A_CHUNK, &tmA, &bar_a[t], 0, t * SK_NT, kc0);
            }
        }
    }
    if (gemm_cta && warp == 2) {
        tmem_alloc(tmem_slot, tmem_cols);
        tmem_relinquish();
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = gemm_cta ? *tmem_slot : 0u;
    pdl_trigger();
    if (!gemm_cta && threadIdx.x == 128) SK_STAMP(1);                          // set-up done
    if (gemm_cta && warp == 2) {
        // warp-uniform control flow, elect.sync picks the issuing lane: inside `if (lane == 0)` every tcgen05.mma cost the lone
        // thread ~106 cycles (descriptors moved from vector to uniform registers per instruction) against the 75 the tensor
        // pipe needs for 128 x 144 x 16 (scripts/probe_umma_chunks.cu)
        constexpr uint32_t idesc = umma_idesc_bf16(128, SK_NT);
        const uint64_t dw0 = umma_desc_sw128(smem_u32(sW));
        const uint64_t da0 = umma_desc_sw128(smem_u32(sA));
        mbar_wait(bar_w, 0);
        if (lane == 0) SK_STAMP(2);                                            // W slab landed
#pragma unroll 1
        for (int t = 0; t < tiles; ++t) {
            mbar_wait(&bar_a[t], 0);
            if (t == 0 && lane == 0) SK_STAMP(3);                              // first A tile landed
            tcgen05_fence_after();
            // (the chunk loop stays OUTSIDE the elected branch: descriptor arithmetic runs on the uniform datapath only where
            // control flow is warp-uniform)
            uint64_t dw = dw0, da = da0 + static_cast<uint64_t>(t * chunks * (SK_A_CHUNK >> 4));
#pragma unroll 1
            for (int ch = 0; ch < chunks; ++ch) {
                if (elect_one()) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_bf16_ss(tmem_base + t * SK_NT, dw + 2 * k, da + 2 * k, idesc, (ch | k) != 0 ? 1u : 0u);
                }
                __syncwarp();
                dw += SK_W_CHUNK >> 4;
                da += SK_A_CHUNK >> 4;
            }
        }
        if (elect_one()) umma_commit(bar_acc);
        __syncwarp();
        pdl_wait();
    } else {
        pdl_wait();
    }
    // ---- past griddepcontrol.wait: the previous kernels' results are visible.  Start the loads the reduce will need.
    // Rendezvous group: the S CTAs of this row block (group rb of `counters`, 4 ints each), or, in the fused modes, ALL
    // CTAs of the grid (group 64).
    int* const meet = tagged ? nullptr : p.counters + 4 * (FUSE == SK_FUSE_NONE ? rb : 64);     // (tagged: no counters at all)
    const int meet_n = FUSE == SK_FUSE_NONE ? S : static_cast<int>(gridDim.x);
    int sense0 = 0;
    if (threadIdx.x == 128 && meet_n > 1 && !tagged) sense0 = ld_acquire_gpu(meet + 2);
    Epi4Ops epre;
    epre.bias = epre.gate = epre.res = make_uint2(0u, 0u);
    TattnPre tpre;
    if (FUSE == SK_FUSE_LN) {
        if (static_cast<int>(blockIdx.x) < total) epre = skinny_ln_preload(p, blockIdx.x, warp, smod);
    } else if (FUSE == SK_FUSE_TATTN) {
        if (static_cast<int>(blockIdx.x) < total) skinny_tattn_preload(p, blockIdx.x, warp, lane, tpre);
    } else if (EPI != EPI_STORE && S > 1) {
        epre.bias = *reinterpret_cast<const uint2*>(p.g.bias + rb * 128 + 4 * lane);
    }

    if (FUSE == SK_FUSE_NONE && S == 1 && warp >= 4) {
        const GemmParams& g = p.g;
        const int q = warp & 3;
        const int n = rb * 128 + q * 32 + lane;
        float bias_n = 0.f;
        if (EPI != EPI_STORE) bias_n = __bfloat162float(g.bias[n]);
        mbar_wait(bar_acc, 0);
        tcgen05_fence_after();
        const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
        for (int c = 0; c < total; c += 16) {
            uint32_t v[16];
            tmem_ld_32x16(tlane + c, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) skinny_store<EPI>(g, c + i, n, __uint_as_float(v[i]), bias_n);
        }
    }
    if (S > 1 && gemm_cta) {
        // ---- accumulator -> fp32 partial tile ws[cta][token][128 weight rows], drained by ALL 8 warps: warp w reads the
        // TMEM lane quadrant w % 4, warps 4-7 the first half of the token columns, warps 0-3 (whose producer / MMA roles
        // are over) the second half
        const int half = total / 2;
        const int q = warp & 3, row = q * 32 + lane;
        mbar_wait(bar_acc, 0);
        tcgen05_fence_after();
        if (threadIdx.x == 128) SK_STAMP(4);                                   // accumulator complete
        const int c0 = warp < 4 ? half : 0;
        const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + c0;
        float* mine = p.ws + static_cast<size_t>(blockIdx.x) * total * 128 + static_cast<size_t>(c0) * 128 + row;
        const uint32_t keep = ~tg.chk;
#pragma unroll 1
        for (int c = 0; c < half; c += 24) {                                   // half = 72 * tiles
            uint32_t v[3][8];
#pragma unroll
            for (int j = 0; j < 3; ++j) tmem_ld_32x8(tlane + c + 8 * j, v[j]);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 3; ++j)
#pragma unroll
                for (int i = 0; i < 8; ++i) st_relaxed_u1(mine + static_cast<size_t>(c + 8 * j + i) * 128, (v[j][i] & keep) | tg.par);
        }
        if (!tagged) {
            // release: partial stores ordered before the arrival below - CTA barrier, then ONE gpu-scope fence by the arriving
            // thread (cumulative over the barrier, the grid-sync idiom), then the relaxed atomic.
            tcgen05_fence_before();
            __syncthreads();
            if (warp == 2) {                           // the accumulator has been read by everyone: give the TMEM back now,
                tcgen05_fence_after();                 // off the kernel's exit path
                tmem_dealloc(tmem_base, tmem_cols);
            }
            if (threadIdx.x == 128) {
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                SK_STAMP(5);                                                       // partials written + fenced
                skinny_rendezvous(meet, meet_n, sense0);
            }
        } else {
            if (threadIdx.x == 128) SK_STAMP(5);                                   // this warp's partials issued
            // The other CTAs' partial sums become visible ~0.5 us after they were issued; loads sent before that come back
            // without them and cost a second round trip.  Wait that long before the first attempt - and give the TMEM back
            // meanwhile, off the kernel's exit path: the other warps only signal that they have read their part of the
            // accumulator (named barrier 1, non-blocking arrive), warp 2 waits for them and deallocates.
            const long long t0 = clock64();
            tcgen05_fence_before();
            if (warp == 2) {
                asm volatile("bar.sync 1, 256;" ::: "memory");
                tcgen05_fence_after();
                tmem_dealloc(tmem_base, tmem_cols);
            } else {
                asm volatile("bar.arrive 1, 256;" ::: "memory");
            }
            while (clock64() - t0 < SK_TAG_DELAY) {}
            if (threadIdx.x == 128) SK_STAMP(6);
        }
    } else if (FUSE != SK_FUSE_NONE && !tagged && threadIdx.x == 128) {
        skinny_rendezvous(meet, meet_n, sense0);                               // reduce-only CTA: nothing to publish
    } else if (FUSE != SK_FUSE_NONE && tagged) {
        // reduce-only CTA: its partial sums will not exist for a few microseconds - one thread watches a single element of the
        // CTA's first token row (last row block, last split) instead of all 256 re-loading whole rows through L2 meanwhile
        if (threadIdx.x == 0 && static_cast<int>(blockIdx.x) < total) {
            const float* probe = p.ws + (static_cast<size_t>(p.gemm_ctas - 1) * total + blockIdx.x) * 128 + 127;
            uint32_t spins = 0u;
            while (!tag_ok(ld_relaxed_u1(probe), tg)) tag_spin_check(spins);
        }
        __syncthreads();
    }
    if (S > 1 && FUSE == SK_FUSE_NONE) {
        // all 8 warps reduce once the rendezvous of the row block has completed (tagged: each warp as soon as it has stored)
        if (!tagged) {
            __syncthreads();
            if (threadIdx.x == 128) SK_STAMP(6);                               // rendezvous passed
        }
        const GemmParams& g = p.g;
        const int lo = split * total / S, hi = (split + 1) * total / S;
        const float* part = p.ws + static_cast<size_t>(rb) * S * total * 128;
        // S = 4 (to_qkv, to_out, fc1 of one rollout: the hot launches) gets the fully unrolled reduce with every load of
        // a warp's tokens in flight at once; the other split counts share one run-time loop - four unrolled variants
        // made these latency-bound kernels ~50 % larger, and instruction fetch is a measured cost for them.
        if (S == 4) skinny_reduce<EPI, 4>(g, part, total, lo, hi, warp, lane, rb * 128, epre.bias, tg);
        else skinny_reduce_any<EPI>(g, part, S, total, lo, hi, warp, lane, rb * 128, epre.bias, tg);
        if (threadIdx.x == 128) SK_STAMP(7);                                   // reduced + stored (this warp)
    }
    if (FUSE != SK_FUSE_NONE) {
        // ---- every CTA has met every other one (thread 128 above; tagged: the loads themselves wait): it now owns whole token rows
        if (!tagged) {
            __syncthreads();
            if (threadIdx.x == 128) SK_STAMP(6);
        }
        if (FUSE == SK_FUSE_LN) {
            skinny_reduce_ln(p, S, total, warp, lane, smod, srow, epre, tg);   // S in {4, 8, 16} (checked on the host)
        } else {
            skinny_reduce_tattn<4>(p, total, warp, lane, tpre, tg);            // S == 4, <= 7 cached frames (checked on the host)
        }
        if (threadIdx.x == 128) SK_STAMP(7);
    }
    if (S == 1 && gemm_cta) {                      // no split: the epilogue warps read the accumulator until here
        tcgen05_fence_before();
        __syncthreads();
        if (warp == 2) tmem_dealloc(tmem_base, tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------ host
bool skinny_supported(int M, int N, int K, int epi) {
    if (M <= 0 || M % SK_NT != 0 || M / SK_NT > 3) return false;
    if (N % 128 != 0 || K % 64 != 0) return false;
    return epi == EPI_STORE || epi == EPI_BIAS || epi == EPI_BIAS_GELU_TANH || epi == EPI_BIAS_GATE_RES;
}

// Largest K split S (dividing the 64-wide chunk count) such that the per-CTA operand slab fits shared memory and
// all (N/128)*S CTAs are co-resident (they rendezvous on a counter).  0 = this shape does not fit the kernel.
int skinny_pick_splits(int M, int N, int K) {
    if (M <= 0 || M % SK_NT != 0 || M / SK_NT > 3 || N % 128 != 0 || K % 64 != 0 || N / 128 > 64) return 0;
    int sms = 148;
    {
        int dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
            sms = n;
    }
    if (sms > 160) sms = 160;
    const int tiles = M / SK_NT, rbs = N / 128, kchunks = K / 64;
    const int per_chunk = SK_W_CHUNK + tiles * SK_A_CHUNK;
    int best = 0;
    for (int s = 1; s <= 16; s *= 2) {                 // the reduction is instantiated for S = 1, 2, 4, 8, 16
        if (kchunks % s) continue;
        if ((kchunks / s) * per_chunk > SK_SMEM_BUDGET) continue;
        if (rbs * s > sms) break;
        best = s;
    }
    // Small weight matrices (to_out of one rollout: N = K = 1024): 4 splits instead of the 16 that would fill the SMs -
    // the split-K exchange (S x 144 x N fp32 through L2, both ways) costs more than the idle SMs save.  Measured in the
    // real step (scripts/bench_graph.py --engine): 16 splits 1.318 ms, 8 splits 1.306 ms, 4 splits 1.297 ms per step.
    if (tiles == 1 && rbs <= 8 && kchunks <= 16 && best > 4) best = 4;
    return best;
}

size_t skinny_workspace_bytes(int M) { return static_cast<size_t>(160) * M * 128 * sizeof(float); }

int skinny_prepare(SkinnyOp* op, const bf16* A, int lda, const bf16* W, int ldw, const GemmParams& p, int epi, float* ws,
                   int* counters, int splits_override, const SkinnyFuseParams* fuse) {
    if (!skinny_supported(p.M, p.N, p.K, epi)) {
        set_error("skinny gemm: unsupported shape/epilogue M=%d N=%d K=%d epi=%d", p.M, p.N, p.K, epi);
        return -1;
    }
    if (epi == EPI_BIAS_GATE_RES && (p.gate == nullptr || p.res == nullptr || p.rows_per_frame != SK_NT)) {
        set_error("skinny gemm: gated-residual epilogue needs gate, residual and rows_per_frame == %d", SK_NT);
        return -1;
    }
    const int tiles = p.M / SK_NT, rbs = p.N / 128, kchunks = p.K / 64;
    const int per_chunk = SK_W_CHUNK + tiles * SK_A_CHUNK;
    int S = splits_override > 0 ? splits_override : skinny_pick_splits(p.M, p.N, p.K);
    if (S <= 0 || S > 16 || (S & (S - 1)) || kchunks % S || (kchunks / S) * per_chunk > SK_SMEM_BUDGET || rbs * S > 160 || rbs > 64) {
        set_error("skinny gemm: no valid K split for M=%d N=%d K=%d (S=%d)", p.M, p.N, p.K, S);
        return -1;
    }
    op->p = p;
    op->epi = epi;
    op->splits = S;
    op->chunks = kchunks / S;
    op->tiles = tiles;
    op->ws = ws;
    op->counters = counters;
    op->trace = nullptr;
    op->tag = 0;
    op->f = SkinnyFuseParams{};
    op->grid = rbs * S;
    if (fuse != nullptr && fuse->mode != SK_FUSE_NONE) {
        // per-token reduce: one CTA per token row up to the SM count (all CTAs must be co-resident: they rendezvous)
        const bool ln_ok = fuse->mode == SK_FUSE_LN && epi == EPI_BIAS_GATE_RES && p.N == 1024 && (S == 4 || S == 8 || S == 16) && fuse->ln_out != nullptr &&
                           fuse->ln_mod != nullptr && fuse->ln_mod_ld % 8 == 0 && fuse->ln_shift_off % 8 == 0 && fuse->ln_scale_off % 8 == 0;
        const bool ta_ok = fuse->mode == SK_FUSE_TATTN && epi == EPI_STORE && p.N == 3072 && S == 4 && fuse->rot != nullptr &&
                           fuse->ctx_frames >= 0 && fuse->ctx_frames <= 7 && (fuse->ctx_frames == 0 || fuse->kv_cache != nullptr) &&
                           fuse->positions > 0 && p.M % fuse->positions == 0;
        if (!ln_ok && !ta_ok) {
            set_error("skinny gemm: fused reduce mode %d does not fit M=%d N=%d K=%d epi=%d splits=%d", fuse->mode, p.M, p.N, p.K, epi, S);
            return -1;
        }
        op->f = *fuse;
        int sms = 148, dev = 0, n = 0;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) sms = n;
        const int want = p.M < sms ? p.M : sms;
        if (want > op->grid) op->grid = want;
    }
    int rc = make_tmap_3d(&op->tmW, W, p.N, p.K, ldw, 128, op->chunks);
    if (rc) return rc;
    return make_tmap_3d(&op->tmA, A, p.M, p.K, lda, SK_NT, op->chunks);
}

template <int EPI, int FUSE>
static int skinny_launch(const SkinnyOp* op, cudaStream_t stream) {
    static bool configured = false;
    auto kern = gemm_skinny_kernel<EPI, FUSE>;
    if (!configured) {
        GTAV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SK_SMEM_BUDGET + SK_TAIL_BYTES + 1024));
        configured = true;
    }
    SkinnyParams sp;
    sp.g = op->p; sp.f = op->f; sp.splits = op->splits; sp.chunks = op->chunks; sp.tiles = op->tiles; sp.ws = op->ws;
    sp.counters = op->counters; sp.gemm_ctas = (op->p.N / 128) * op->splits;
    sp.trace = op->trace;
    sp.tag = op->tag;
    // At least half of the SM's shared memory, so that exactly one CTA of this kernel fits on an SM: the CTAs of a
    // row block wait for each other, and a second CTA on the same SM could block in tcgen05.alloc behind a waiting one.
    // (Two CTAs per SM - the next launch starting under the current one - was measured and dropped: TMA loads of an
    // early-launched CTA that shares its SM with a CTA of the previous kernel do not complete before that CTA exits,
    // profiles/r01/skinny_coresident_trace.txt.)
    size_t smem = static_cast<size_t>(op->chunks) * (SK_W_CHUNK + op->tiles * SK_A_CHUNK) + SK_TAIL_BYTES + 1024;
    if (smem < 120 * 1024) smem = 120 * 1024;
    GTAV_CUDA_OK(launch_k(kern, dim3(op->grid), dim3(SK_THREADS), smem, stream, op->tmW, op->tmA, sp));
    return 0;
}

int skinny_run(const SkinnyOp* op, cudaStream_t stream) {
    if (op->f.mode == SK_FUSE_LN) return skinny_launch<EPI_BIAS_GATE_RES, SK_FUSE_LN>(op, stream);
    if (op->f.mode == SK_FUSE_TATTN) return skinny_launch<EPI_STORE, SK_FUSE_TATTN>(op, stream);
    switch (op->epi) {
        case EPI_STORE: return skinny_launch<EPI_STORE, SK_FUSE_NONE>(op, stream);
        case EPI_BIAS: return skinny_launch<EPI_BIAS, SK_FUSE_NONE>(op, stream);
        case EPI_BIAS_GELU_TANH: return skinny_launch<EPI_BIAS_GELU_TANH, SK_FUSE_NONE>(op, stream);
        case EPI_BIAS_GATE_RES: return skinny_launch<EPI_BIAS_GATE_RES, SK_FUSE_NONE>(op, stream);
    }
    set_error("skinny gemm: unknown epilogue %d", op->epi);
    return -1;
}

}  // namespace gtav
