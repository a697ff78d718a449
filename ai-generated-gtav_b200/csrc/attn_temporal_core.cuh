// Temporal attention of ONE (rollout, position, head) problem for the frame being denoised: the query is the last
// frame's, keys/values are the TC cached context frames (rotated K and V, reference model/attention.py:52-66)
// followed by the frame's own.  One warp, lane = one rotary pair (2 of the 64 head dims).  Shared by
// attn_temporal_last_kernel (attn_temporal.cu) and the attention fused into the weight-streaming to_qkv GEMM's
// reduce (gemm_skinny.cu), so both produce the same bits from the same q / k / v.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace gtav {

// Valid frames of rollout b in a ragged pass over `frames` slots (kernels.h, TemporalLens); warp-uniform.
__device__ __forceinline__ int ragged_valid(const TemporalLens& r, int b, int frames) {
    return min(max(r.len[b], r.lo), frames + r.sub) - r.sub;
}

// Every fp32 operation below is an explicit round-to-nearest intrinsic: the same source compiled into different kernels
// must not be contracted into FMAs differently (the fused and the stand-alone paths are tested for equal bits), and
// the rotation is the reference's unfused t * cos + rotate_half(t) * sin (rotary_embedding_torch.py:46-73).
__device__ __forceinline__ float2 rotary_pair_rn(float2 x, float2 cs) {
    return make_float2(bf16_round(__fsub_rn(__fmul_rn(x.x, cs.x), __fmul_rn(x.y, cs.y))),
                       bf16_round(__fadd_rn(__fmul_rn(x.y, cs.x), __fmul_rn(x.x, cs.y))));
}
__device__ __forceinline__ float dot_pair_rn(float2 a, float2 b) { return __fmaf_rn(a.x, b.x, __fmul_rn(a.y, b.y)); }

// This lane's pairs of the cached rotated K and V of context frames 0 .. tc-1 (packed bf16x2), TMAX >= tc.
// cache: kv_cache + (first context row of this (b, pos)) * 2D + head*64 + 2*lane, consecutive frames frame_stride
// elements apart.  Separate from the core so that callers can issue the loads early.
template <int TMAX>
__device__ __forceinline__ void temporal_cache_load(uint32_t (&kc)[TMAX], uint32_t (&vc)[TMAX], int tc, const bf16* cache,
                                                    size_t frame_stride, int D) {
#pragma unroll
    for (int t = 0; t < TMAX; ++t) {
        kc[t] = 0u;
        vc[t] = 0u;
        if (t < tc) {
            const bf16* c = cache + static_cast<size_t>(t) * frame_stride;
            kc[t] = *reinterpret_cast<const uint32_t*>(c);
            vc[t] = *reinterpret_cast<const uint32_t*>(c + D);
        }
    }
}

// qx, kx, vx: this lane's un-rotated q / k pair and v pair of the last frame (bf16 values as floats); kc / vc: the
// first tc entries are the cached context pairs (temporal_cache_load); cs: (cos, sin) of window position tc for this
// lane's pair.  tc (<= TMAX, warp-uniform) is a run-time value: the loops are unrolled to TMAX + 1 keys and predicated,
// which executes exactly the operations, in the order, of a loop over the tc + 1 real keys - one copy of the code for
// every window length (a compile-time tc folds the predicates away).  Returns the packed bf16 output pair.
template <int TMAX>
__device__ __forceinline__ uint32_t temporal_last_core(int tc, float2 qx, float2 kx, float2 vx, const uint32_t (&kc)[TMAX],
                                                       const uint32_t (&vc)[TMAX], float2 cs) {
    // rotate in fp32, round once to bf16 (apply_rotary_emb casts back to the input dtype)
    const float2 q = rotary_pair_rn(qx, cs);
    const float2 kn = rotary_pair_rn(kx, cs);
    // Scores of all TMAX + 1 key slots at once: the dot products' warp reductions are five dependent shuffles each, and
    // reduced one key after the other (behind a branch per key) they were a chain of 5 (tc + 1) shuffle latencies in the
    // fused reduce of every temporal to_qkv launch.  Here each butterfly step issues the shuffles of all slots back to back
    // (slots beyond tc reduce a copy of the frame's own key and are ignored); per key the additions are warp_sum's, in its
    // order - same bits.
    float s[TMAX + 1];
#pragma unroll
    for (int j = 0; j <= TMAX; ++j) {
        float2 k = kn;
        if (j < TMAX && j < tc) k = unpack_bf16x2(kc[j < TMAX ? j : 0]);
        s[j] = dot_pair_rn(q, k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int j = 0; j <= TMAX; ++j) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
    }
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j <= TMAX; ++j) {
        if (j <= tc) {                                       // key j: cached frame j, or (j == tc) the frame's own
            s[j] = __fmul_rn(s[j], 0.125f);
            m = fmaxf(m, s[j]);
        } else {
            s[j] = 0.f;
        }
    }
    float l = 0.f;
#pragma unroll
    for (int j = 0; j <= TMAX; ++j)
        if (j <= tc) {
            s[j] = __expf(__fsub_rn(s[j], m));
            l = __fadd_rn(l, s[j]);
        }
    const float inv = __frcp_rn(l);
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int j = 0; j <= TMAX; ++j)
        if (j <= tc) {
            float2 v = vx;
            if (j < TMAX && j < tc) v = unpack_bf16x2(vc[j < TMAX ? j : 0]);
            const float p = bf16_round(__fmul_rn(s[j], inv));   // probabilities enter P@V as bf16
            acc.x = __fmaf_rn(p, v.x, acc.x);
            acc.y = __fmaf_rn(p, v.y, acc.y);
        }
    return pack_bf16x2(acc.x, acc.y);
}

}  // namespace gtav
