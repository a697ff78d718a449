// Temporal attention for long sliding windows: 9..32 frames (dense) and 8..31 cached frames (last frame only).
//
// The short-window kernels of attn_temporal.cu are unrolled per window length and keep q, k and v of every frame as
// float2 registers; at 32 frames those 3 T float2 would spill.  Here the window length is a run-time value bounded by a
// compile-time maximum.  The dense kernel stages the rotated K and the V of its problem in shared memory as packed bf16
// pairs (rotated K is already rounded to bf16 and V is bf16 in memory, so packing loses nothing): 8 KB per warp at 32
// frames, each lane reading back only the words it wrote, so no barrier is needed.  Kept in registers instead, they
// take 227 registers (the compiler unpacks them once, outside the query loop) and leave one block per SM.  The semantics are
// attn_temporal_kernel's: one warp per (rollout, position, head), one lane per rotary pair, rotation with
// rotary_pair_rn and one bf16 rounding, the optional K/V cache in the same [row][k | v] layout, probabilities rounded to
// bf16 before P.V.  Per query the max, exp, sum and P.V run over keys j = 0..i in the order of temporal_last_core, so
// the last-frame kernel below (which runs temporal_last_core itself) returns row T - 1 of the dense kernel bit for bit.
#include "attn_temporal_core.cuh"
#include "common.cuh"
#include "kernels.h"

namespace gtav {

static constexpr int TL_WARPS = 8;         // last-frame kernel (registers only, like attn_temporal_last_kernel)
static constexpr int TLD_WARPS = 4;        // dense kernel: 32 KB of static shared memory per block
static constexpr int TL_MAX_FRAMES = 32;   // dense window
static constexpr int TL_KEY_CHUNK = 8;     // keys whose warp reductions are issued back to back

// qkv [B*T*P, 3D] rows (b, t, pos), out [B*T*P, D], rot float2 [T][32], kv_cache (optional) [B*T*P, 2D].
// RAGGED: as attn_temporal_kernel<T, true> (attn_temporal.cu) - slots before the rollout's trailing valid frames are
// padding (output and cache rows 0), valid slot t sits at rotary position t - off and attends to valid keys only, with the
// arithmetic and order of row t - off of an (T - off)-frame window.
template <int TMAX, bool RAGGED = false>
__global__ void __launch_bounds__(TLD_WARPS * 32)
attn_temporal_long_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int B, int T, int P, int heads,
                          const float2* __restrict__ rot, bf16* __restrict__ kv_cache, TemporalLens lens) {
    __shared__ uint32_t sk[TLD_WARPS][TMAX][32], sv[TLD_WARPS][TMAX][32];
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long wg = static_cast<long>(blockIdx.x) * TLD_WARPS + warp;
    if (wg >= static_cast<long>(B) * P * heads) return;
    const int head = static_cast<int>(wg % heads);
    const int pos = static_cast<int>((wg / heads) % P);
    const int b = static_cast<int>(wg / (static_cast<long>(heads) * P));
    const int D = heads * 64;
    const int ld = 3 * D;
    const bf16* base = qkv + (static_cast<size_t>(b) * T * P + pos) * ld + head * 64 + 2 * lane;
    const size_t frame_ld = static_cast<size_t>(P) * ld;
    uint32_t (&kc)[TMAX][32] = sk[warp];
    uint32_t (&vc)[TMAX][32] = sv[warp];
    const int off = RAGGED ? T - ragged_valid(lens, b, T) : 0;      // padded slots of this rollout

    // rotated K and V of every frame, packed bf16x2; the loads of a group of frames are issued before their first use
    constexpr int G = 8;
#pragma unroll
    for (int t0 = 0; t0 < TMAX; t0 += G) {
        if (t0 < T) {
            uint32_t ku[G], vu[G];
#pragma unroll
            for (int t = t0; t < t0 + G; ++t) {
                ku[t - t0] = 0u;
                vu[t - t0] = 0u;
                if (t < T) {
                    ku[t - t0] = *reinterpret_cast<const uint32_t*>(base + t * frame_ld + D);
                    vu[t - t0] = *reinterpret_cast<const uint32_t*>(base + t * frame_ld + 2 * D);
                }
            }
#pragma unroll
            for (int t = t0; t < t0 + G; ++t) {
                const float2 k = rotary_pair_rn(unpack_bf16x2(ku[t - t0]), rot[(t < T && t >= off ? t - off : 0) * 32 + lane]);
                kc[t][lane] = pack_bf16x2(k.x, k.y);          // exact: rotary_pair_rn rounded both halves to bf16
                vc[t][lane] = vu[t - t0];
                if (kv_cache != nullptr && t < T) {
                    const size_t row = (static_cast<size_t>(b) * T + t) * P + pos;
                    bf16* c = kv_cache + row * (2 * D) + head * 64 + 2 * lane;
                    const bool pad = RAGGED && t < off;
                    *reinterpret_cast<uint32_t*>(c) = pad ? 0u : kc[t][lane];
                    *reinterpret_cast<uint32_t*>(c + D) = pad ? 0u : vu[t - t0];
                }
            }
        }
    }

    if (RAGGED) {
        for (int i = 0; i < off; ++i) {
            const size_t row = (static_cast<size_t>(b) * T + i) * P + pos;
            *reinterpret_cast<uint32_t*>(out + row * D + head * 64 + 2 * lane) = 0u;
        }
    }
#pragma unroll 1
    for (int i = off; i < T; ++i) {
        const float2 q = rotary_pair_rn(unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base + i * frame_ld)), rot[(i - off) * 32 + lane]);
        // Scores of keys 0..i.  Keys go in chunks: the five butterfly steps of a chunk's dot products are issued key after
        // key within each step (as temporal_last_core does), and chunks past the query are skipped (warp-uniform).  Per
        // key the additions are warp_sum's, in its order.  Keys i < j (and padded keys j < off) of a live chunk are computed
        // and ignored.
        float s[TMAX];
#pragma unroll
        for (int c = 0; c < TMAX; c += TL_KEY_CHUNK) {
            if (c <= i && c + TL_KEY_CHUNK > off) {
#pragma unroll
                for (int j = c; j < c + TL_KEY_CHUNK; ++j) s[j] = dot_pair_rn(q, unpack_bf16x2(kc[j][lane]));
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int j = c; j < c + TL_KEY_CHUNK; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
                }
            }
        }
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j < TMAX; ++j)
            if (j <= i && j >= off) {
                s[j] = __fmul_rn(s[j], 0.125f);
                m = fmaxf(m, s[j]);
            }
        float l = 0.f;
#pragma unroll
        for (int j = 0; j < TMAX; ++j)
            if (j <= i && j >= off) {
                s[j] = __expf(__fsub_rn(s[j], m));
                l = __fadd_rn(l, s[j]);
            }
        const float inv = __frcp_rn(l);
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < TMAX; ++j)
            if (j <= i && j >= off) {
                const float2 v = unpack_bf16x2(vc[j][lane]);
                const float p = bf16_round(__fmul_rn(s[j], inv));   // probabilities enter P@V as bf16
                acc.x = __fmaf_rn(p, v.x, acc.x);
                acc.y = __fmaf_rn(p, v.y, acc.y);
            }
        const size_t row = (static_cast<size_t>(b) * T + i) * P + pos;
        *reinterpret_cast<uint32_t*>(out + row * D + head * 64 + 2 * lane) = pack_bf16x2(acc.x, acc.y);
    }
}

// Last frame against tc (run-time, <= TMAX) cached frames: attn_temporal_last_kernel with the cache length as an argument.
// Same loads and the same temporal_last_core, so the same bits as row tc of the dense kernel.  RAGGED: rollout b attends to
// the trailing ragged_valid(lens, b, tc) of its tc cached slots, as attn_temporal_last_kernel<TC, true>.
template <int TMAX, bool RAGGED = false>
__global__ void __launch_bounds__(TL_WARPS * 32)
attn_temporal_last_long_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int B, int tc, int P, int heads,
                               const float2* __restrict__ rot, const bf16* __restrict__ kv_cache, TemporalLens lens) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const long wg = static_cast<long>(blockIdx.x) * TL_WARPS + (threadIdx.x >> 5);
    if (wg >= static_cast<long>(B) * P * heads) return;
    const int head = static_cast<int>(wg % heads);
    const int pos = static_cast<int>((wg / heads) % P);
    const int b = static_cast<int>(wg / (static_cast<long>(heads) * P));
    const int D = heads * 64;

    const size_t qrow = static_cast<size_t>(b) * P + pos;
    const bf16* base = qkv + qrow * (3 * D) + head * 64 + 2 * lane;
    const bf16* cache = kv_cache + (static_cast<size_t>(b) * tc * P + pos) * (2 * D) + head * 64 + 2 * lane;
    if (RAGGED) {                           // the trailing n of the tc cached slots
        const int n = ragged_valid(lens, b, tc);
        cache += static_cast<size_t>(tc - n) * P * (2 * D);
        tc = n;
    }
    uint32_t kc[TMAX], vc[TMAX];
    temporal_cache_load(kc, vc, tc, cache, static_cast<size_t>(P) * 2 * D, D);
    const float2 qx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base));
    const float2 kx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base + D));
    const float2 vx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base + 2 * D));
    *reinterpret_cast<uint32_t*>(out + qrow * D + head * 64 + 2 * lane) = temporal_last_core(tc, qx, kx, vx, kc, vc, rot[tc * 32 + lane]);
}

int launch_attention_temporal_long(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                                   bf16* kv_cache, const TemporalLens* lens, cudaStream_t s) {
    if (T < 9 || T > TL_MAX_FRAMES) {
        set_error("temporal attention: window of %d frames unsupported (1..32)", T);
        return -1;
    }
    const long problems = static_cast<long>(B) * positions * heads;
    if (problems <= 0) return 0;
    const int grid = static_cast<int>((problems + TLD_WARPS - 1) / TLD_WARPS);
    if (lens != nullptr) {
        GTAV_CUDA_OK(launch_k(attn_temporal_long_kernel<TL_MAX_FRAMES, true>, dim3(grid), dim3(TLD_WARPS * 32), 0, s, qkv, out, B,
                              T, positions, heads, rot, kv_cache, *lens));
        return 0;
    }
    GTAV_CUDA_OK(launch_k(attn_temporal_long_kernel<TL_MAX_FRAMES>, dim3(grid), dim3(TLD_WARPS * 32), 0, s, qkv, out, B, T,
                          positions, heads, rot, kv_cache, TemporalLens{}));
    return 0;
}

int launch_attention_temporal_last_long(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                        const float2* rot, const bf16* kv_cache, const TemporalLens* lens, cudaStream_t s) {
    if (ctx_frames < 8 || ctx_frames > TL_MAX_FRAMES - 1) {
        set_error("temporal attention (last frame): %d cached frames unsupported (0..31)", ctx_frames);
        return -1;
    }
    const long problems = static_cast<long>(B) * positions * heads;
    if (problems <= 0) return 0;
    if (kv_cache == nullptr) {
        set_error("temporal attention (last frame): missing K/V cache");
        return -1;
    }
    const int grid = static_cast<int>((problems + TL_WARPS - 1) / TL_WARPS);
    if (lens != nullptr) {
        GTAV_CUDA_OK(launch_k(attn_temporal_last_long_kernel<TL_MAX_FRAMES - 1, true>, dim3(grid), dim3(TL_WARPS * 32), 0, s, qkv,
                              out, B, ctx_frames, positions, heads, rot, kv_cache, *lens));
        return 0;
    }
    GTAV_CUDA_OK(launch_k(attn_temporal_last_long_kernel<TL_MAX_FRAMES - 1>, dim3(grid), dim3(TL_WARPS * 32), 0, s, qkv, out,
                          B, ctx_frames, positions, heads, rot, kv_cache, TemporalLens{}));
    return 0;
}

}  // namespace gtav
