// Causal attention over the (<= 8) frames of a short sliding window, one problem per (rollout, spatial
// position, head), with the 1-D rotary embedding on the frame index fused.
//
// Replaces TemporalAxialAttention's rearrange + rotate_queries_or_keys + causal SDPA (reference
// model/attention.py:52-66; rotary_embedding_torch.py:186-209: positions are window-relative
// arange(T), theta 1e4).  T x T scores with T <= 5 are far too small for tensor cores: this kernel
// is L2/HBM-bound (reads the 3*D-wide qkv rows once, writes D), one warp per problem, each lane owns
// one rotary pair (2 of the 64 head dims), dot products reduced with shuffles.  Windows of 9..32 frames
// (8..31 cached) run the kernels of attn_temporal_long.cu, which the launchers below dispatch to.
#include "attn_temporal_core.cuh"
#include "common.cuh"
#include "kernels.h"

namespace gtav {

static constexpr int TA_WARPS = 8;

// RAGGED: rollout b's window holds ragged_valid(lens, b, T) valid frames in its trailing slots (kernels.h, TemporalLens);
// the padded slots before them are neither keys nor queries, and their output and cache rows are 0.  A valid slot t sits
// at rotary position t - off, and its row runs the arithmetic, in the order, of row t - off of attn_temporal_kernel<T - off>:
// same bits.
template <int T, bool RAGGED = false>
__global__ void __launch_bounds__(TA_WARPS * 32)
attn_temporal_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int B, int P, int heads,
                     const float2* __restrict__ rot, bf16* __restrict__ kv_cache, TemporalLens lens) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const long wg = static_cast<long>(blockIdx.x) * TA_WARPS + (threadIdx.x >> 5);
    if (wg >= static_cast<long>(B) * P * heads) return;
    const int head = static_cast<int>(wg % heads);
    const int pos = static_cast<int>((wg / heads) % P);
    const int b = static_cast<int>(wg / (static_cast<long>(heads) * P));
    const int D = heads * 64;
    const int ld = 3 * D;

    const int off = RAGGED ? T - ragged_valid(lens, b, T) : 0;      // padded slots of this rollout

    float2 q[T], k[T], v[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
        const size_t row = (static_cast<size_t>(b) * T + t) * P + pos;
        const bf16* base = qkv + row * ld + head * 64 + 2 * lane;
        const uint32_t qu = *reinterpret_cast<const uint32_t*>(base);
        const uint32_t ku = *reinterpret_cast<const uint32_t*>(base + D);
        const uint32_t vu = *reinterpret_cast<const uint32_t*>(base + 2 * D);
        const float2 cs = rot[(t >= off ? t - off : 0) * 32 + lane];     // (a padded slot's values are never used)
        const float2 qx = unpack_bf16x2(qu), kx = unpack_bf16x2(ku);
        // rotate in fp32, round once to bf16 (apply_rotary_emb casts back to the input dtype)
        q[t] = rotary_pair_rn(qx, cs);
        k[t] = rotary_pair_rn(kx, cs);
        v[t] = unpack_bf16x2(vu);
        if (kv_cache != nullptr) {
            // rotated K (already rounded to bf16) and V of every frame, row-for-row like qkv: [row][k | v][D]
            bf16* c = kv_cache + row * (2 * D) + head * 64 + 2 * lane;
            const bool pad = RAGGED && t < off;
            *reinterpret_cast<uint32_t*>(c) = pad ? 0u : pack_bf16x2(k[t].x, k[t].y);
            *reinterpret_cast<uint32_t*>(c + D) = pad ? 0u : vu;
        }
    }
#pragma unroll
    for (int i = 0; i < T; ++i) {
        if (RAGGED && i < off) {
            const size_t row = (static_cast<size_t>(b) * T + i) * P + pos;
            *reinterpret_cast<uint32_t*>(out + row * D + head * 64 + 2 * lane) = 0u;
            continue;
        }
        float s[T];
        float m = -INFINITY;
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            if (RAGGED && j < off) continue;
            s[j] = __fmul_rn(warp_sum(dot_pair_rn(q[i], k[j])), 0.125f);
            m = fmaxf(m, s[j]);
        }
        float l = 0.f;
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            if (RAGGED && j < off) continue;
            s[j] = __expf(__fsub_rn(s[j], m));
            l = __fadd_rn(l, s[j]);
        }
        const float inv = __frcp_rn(l);
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            if (RAGGED && j < off) continue;
            const float p = bf16_round(__fmul_rn(s[j], inv));   // probabilities enter P@V as bf16
            acc.x = __fmaf_rn(p, v[j].x, acc.x);
            acc.y = __fmaf_rn(p, v[j].y, acc.y);
        }
        const size_t row = (static_cast<size_t>(b) * T + i) * P + pos;
        *reinterpret_cast<uint32_t*>(out + row * D + head * 64 + 2 * lane) = pack_bf16x2(acc.x, acc.y);
    }
}

// Last frame only: the query is the frame being denoised (window position TC = number of cached context
// frames), keys/values are the TC cached context frames (rotated K and V written by attn_temporal_kernel
// with kv_cache set) followed by the frame's own k/v.  Same arithmetic, in the same order, as row T-1 of
// attn_temporal_kernel<TC+1>, so the cached step reproduces the dense step bit for bit.
// qkv [B*P, 3D] (last-frame rows only), out [B*P, D], kv_cache [B*TC*P, 2D].
// RAGGED: rollout b attends to the trailing tc = ragged_valid(lens, b, TC) of its TC cached slots and its query sits at
// rotary position tc - the bits of attn_temporal_last_kernel<tc> (temporal_last_core takes a run-time tc).
template <int TC, bool RAGGED = false>
__global__ void __launch_bounds__(TA_WARPS * 32)
attn_temporal_last_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int B, int P, int heads,
                          const float2* __restrict__ rot, const bf16* __restrict__ kv_cache, TemporalLens lens) {
    pdl_trigger();
    pdl_wait();
    const int lane = threadIdx.x & 31;
    const long wg = static_cast<long>(blockIdx.x) * TA_WARPS + (threadIdx.x >> 5);
    if (wg >= static_cast<long>(B) * P * heads) return;
    const int head = static_cast<int>(wg % heads);
    const int pos = static_cast<int>((wg / heads) % P);
    const int b = static_cast<int>(wg / (static_cast<long>(heads) * P));
    const int D = heads * 64;

    const size_t qrow = static_cast<size_t>(b) * P + pos;
    const bf16* base = qkv + qrow * (3 * D) + head * 64 + 2 * lane;
    const bf16* cache = kv_cache + (static_cast<size_t>(b) * TC * P + pos) * (2 * D) + head * 64 + 2 * lane;
    int tc = TC;
    if (RAGGED) {                           // the trailing tc cached slots
        tc = ragged_valid(lens, b, TC);
        cache += static_cast<size_t>(TC - tc) * P * (2 * D);
    }
    const float2 qx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base));
    const float2 kx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base + D));
    const float2 vx = unpack_bf16x2(*reinterpret_cast<const uint32_t*>(base + 2 * D));
    uint32_t kc[TC > 0 ? TC : 1], vc[TC > 0 ? TC : 1];
    temporal_cache_load(kc, vc, tc, cache, static_cast<size_t>(P) * 2 * D, D);
    *reinterpret_cast<uint32_t*>(out + qrow * D + head * 64 + 2 * lane) = temporal_last_core(tc, qx, kx, vx, kc, vc, rot[tc * 32 + lane]);
}

int launch_attention_temporal_last(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                   const float2* rot, const bf16* kv_cache, cudaStream_t s) {
    const long problems = static_cast<long>(B) * positions * heads;
    if (problems <= 0) return 0;
    if (ctx_frames > 0 && kv_cache == nullptr) {
        set_error("temporal attention (last frame): missing K/V cache");
        return -1;
    }
    const int grid = static_cast<int>((problems + TA_WARPS - 1) / TA_WARPS);
#define GTAV_TL(TT)                                                                                          \
    case TT:                                                                                                 \
        GTAV_CUDA_OK(launch_k(attn_temporal_last_kernel<TT>, dim3(grid), dim3(TA_WARPS * 32), 0, s, qkv, out, B, positions, heads, \
                              rot, kv_cache, TemporalLens{}));                                              \
        break;
    switch (ctx_frames) {
        GTAV_TL(0) GTAV_TL(1) GTAV_TL(2) GTAV_TL(3) GTAV_TL(4) GTAV_TL(5) GTAV_TL(6) GTAV_TL(7)
        default:   // 8..31 cached frames (attn_temporal_long.cu); refuses anything else
            return launch_attention_temporal_last_long(qkv, out, B, ctx_frames, positions, heads, rot, kv_cache, nullptr, s);
    }
#undef GTAV_TL
    return 0;
}

int launch_attention_temporal_last_ragged(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                          const float2* rot, const bf16* kv_cache, TemporalLens lens, cudaStream_t s) {
    if (lens.len == nullptr) {
        set_error("temporal attention (last frame, ragged): missing window lengths");
        return -1;
    }
    // no cached frame: nothing is ragged, every rollout attends to its own key only
    if (ctx_frames == 0) return launch_attention_temporal_last(qkv, out, B, 0, positions, heads, rot, kv_cache, s);
    const long problems = static_cast<long>(B) * positions * heads;
    if (ctx_frames < 0 || ctx_frames > 7) {
        return launch_attention_temporal_last_long(qkv, out, B, ctx_frames, positions, heads, rot, kv_cache, &lens, s);
    }
    if (problems <= 0) return 0;
    if (kv_cache == nullptr) {
        set_error("temporal attention (last frame): missing K/V cache");
        return -1;
    }
    const int grid = static_cast<int>((problems + TA_WARPS - 1) / TA_WARPS);
#define GTAV_TL(TT)                                                                                          \
    case TT:                                                                                                 \
        GTAV_CUDA_OK(launch_k(attn_temporal_last_kernel<TT, true>, dim3(grid), dim3(TA_WARPS * 32), 0, s, qkv, out, B, positions, \
                              heads, rot, kv_cache, lens));                                                  \
        break;
    switch (ctx_frames) {
        GTAV_TL(1) GTAV_TL(2) GTAV_TL(3) GTAV_TL(4) GTAV_TL(5) GTAV_TL(6) GTAV_TL(7)
    }
#undef GTAV_TL
    return 0;
}

int launch_attention_temporal(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                              bf16* kv_cache, cudaStream_t s) {
    const long problems = static_cast<long>(B) * positions * heads;
    if (problems <= 0) return 0;
    const int grid = static_cast<int>((problems + TA_WARPS - 1) / TA_WARPS);
#define GTAV_TA(TT)                                                                                       \
    case TT:                                                                                              \
        GTAV_CUDA_OK(launch_k(attn_temporal_kernel<TT>, dim3(grid), dim3(TA_WARPS * 32), 0, s, qkv, out, B, positions, heads, rot, \
                              kv_cache, TemporalLens{}));                                                 \
        break;
    switch (T) {
        GTAV_TA(1) GTAV_TA(2) GTAV_TA(3) GTAV_TA(4) GTAV_TA(5) GTAV_TA(6) GTAV_TA(7) GTAV_TA(8)
        default:   // 9..32 frames (attn_temporal_long.cu); refuses anything else
            return launch_attention_temporal_long(qkv, out, B, T, positions, heads, rot, kv_cache, nullptr, s);
    }
#undef GTAV_TA
    return 0;
}

int launch_attention_temporal_ragged(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                                     bf16* kv_cache, TemporalLens lens, cudaStream_t s) {
    if (lens.len == nullptr) {
        set_error("temporal attention (ragged): missing window lengths");
        return -1;
    }
    if (T < 1 || T > 8) return launch_attention_temporal_long(qkv, out, B, T, positions, heads, rot, kv_cache, &lens, s);
    const long problems = static_cast<long>(B) * positions * heads;
    if (problems <= 0) return 0;
    const int grid = static_cast<int>((problems + TA_WARPS - 1) / TA_WARPS);
#define GTAV_TA(TT)                                                                                       \
    case TT:                                                                                              \
        GTAV_CUDA_OK(launch_k(attn_temporal_kernel<TT, true>, dim3(grid), dim3(TA_WARPS * 32), 0, s, qkv, out, B, positions, heads, \
                              rot, kv_cache, lens));                                                      \
        break;
    switch (T) {
        GTAV_TA(1) GTAV_TA(2) GTAV_TA(3) GTAV_TA(4) GTAV_TA(5) GTAV_TA(6) GTAV_TA(7) GTAV_TA(8)
    }
#undef GTAV_TA
    return 0;
}

}  // namespace gtav
