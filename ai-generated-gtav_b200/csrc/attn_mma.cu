// Non-causal multi-head attention over short sequences with the rotary embedding fused on load.
//
// Replaces SpatialAxialAttention's rearrange + get_axial_freqs + apply_rotary_emb + SDPA
// (reference model/attention.py:111-129, S = 144 tokens, rotary on all 64 head dims) and the VAE
// Attention (model/vae.py:83-107, S = 576, rotary on head dims 0..31 only).  Head dim is 64.
//
// This is 1.2 % (DiT) / 8.5 % (VAE) of the step's FLOPs, so round 1 keeps it on warp-level
// mma.sync m16n8k16 tiles (flash-style: scores stay in registers, online softmax across key
// blocks, P rounded to bf16 before P@V like the reference's fused SDPA backends).  q/k are rotated
// as apply_rotary_emb does (rotary_embedding_torch.py:46-73): two fp32 products and their fp32 sum,
// each rounded to nearest (no FMA contraction), then one rounding to bf16.
#include <stdlib.h>

#include "attn_seq.cuh"

namespace gtav {

// grid: (SEQ / (WARPS*16), heads, groups).  qkv rows of one group are consecutive.
template <int SEQ, int KB, int WARPS, int ROT_PAIRS>
__global__ void __launch_bounds__(WARPS * 32)
attn_seq_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int heads, const float2* __restrict__ rot) {
    __shared__ __align__(16) bf16 sK[KB * SROW];
    __shared__ __align__(16) bf16 sV[KB * SROW];
    pdl_trigger();
    pdl_wait();
    attn_seq_body<SEQ, KB, WARPS, ROT_PAIRS, false>(qkv, out, heads, rot, sK, sV, blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, 0);
}

// DiT spatial attention (144 tokens, rotary on all 32 pairs): the rotary table [144][32] (cos, sin) is a CONSTANT of the
// model, so every CTA copies it into shared memory with cp.async BEFORE griddepcontrol.wait - as global loads issued when
// the K / V rows arrive, it was a second dependent L2 round trip in a ~5 us kernel of the latency-bound last-frame chain.
static constexpr int ROT144_BYTES = 144 * 32 * 8;
static constexpr int ATTN144_SMEM = 2 * 144 * SROW * 2 + ROT144_BYTES;
__global__ void __launch_bounds__(3 * 32)
attn_seq144_kernel(const bf16* __restrict__ qkv, bf16* __restrict__ out, int heads, const float2* __restrict__ rot) {
    extern __shared__ __align__(16) uint8_t smem144[];
    bf16* sK = reinterpret_cast<bf16*>(smem144);
    bf16* sV = sK + 144 * SROW;
    float2* sRot = reinterpret_cast<float2*>(smem144 + 2 * 144 * SROW * 2);
    for (int i = threadIdx.x; i < ROT144_BYTES / 16; i += 3 * 32)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(reinterpret_cast<uint8_t*>(sRot) + i * 16)),
                     "l"(reinterpret_cast<const uint8_t*>(rot) + i * 16) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
    pdl_trigger();
    pdl_wait();
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    attn_seq_body<144, 144, 3, 32, false>(qkv, out, heads, sRot, sK, sV, blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, 0);
}

// Which implementation runs (measured on B200, scripts/bench_attn.py, profiles/r02/bench_attn_*.log):
//   S = 576 (VAE): the tcgen05 kernel (attn_tc.cu) from 4 frames up (64 CTAs): 128 us against 222 us for 32 frames; below
//                  that one CTA per head leaves most SMs idle and the mma.sync kernel's 9 CTAs per head win (23 vs 31 us);
//   S = 144 (DiT): the tcgen05 kernel from 96 frames up (context passes and dense windows of >= 20 rollouts), where it is
//                  2-3 % ahead (120 vs 123 us at 160 frames, 233 vs 238 us at 320; cross-over at ~96: 76.6 vs 77.1 us); below
//                  that the mma.sync kernel's 3 CTAs per head win, most clearly in the latency-bound last-frame steps of few
//                  rollouts (5 us against 11 us per launch at one frame, 35 vs 38 us at 40 frames).
// GTAV_ATTN = "tc" / "mma" forces one of them for every size (parity tests, A/B measurements).
static int attn_use_tc(int seq, int groups) {
    const char* e = getenv("GTAV_ATTN");          // read per call: launches are captured into graphs, tests flip it
    if (e != nullptr && e[0] == 't') return 1;
    if (e != nullptr && e[0] == 'm') return 0;
    return seq == 576 ? groups >= 4 : groups >= 96;
}

int launch_attention_seq(const bf16* qkv, bf16* out, int groups, int seq, int heads, const float2* rot, int rot_pairs,
                         cudaStream_t s) {
    if (groups <= 0) return 0;
    if (((seq == 144 && rot_pairs == 32) || (seq == 576 && rot_pairs == 16)) && attn_use_tc(seq, groups))
        return launch_attention_tc(qkv, out, groups, seq, heads, rot, rot_pairs, s);
    if (seq == 144 && rot_pairs == 32) {
        // all 144 keys of a head staged in one pass (every global load of the block in flight at once); the queries
        // are split over 3 CTAs of 3 warps so that 48 SMs share the loads at B = 1
        if (groups * heads * 3 <= 2 * 148) {
            // few frames (last-frame steps of up to 6 rollouts, context passes): latency matters, every CTA has an SM
            // (almost) to itself - the variant with the rotary table staged in its 78 KB of shared memory
            static bool configured = false;
            if (!configured) {
                GTAV_CUDA_OK(cudaFuncSetAttribute(attn_seq144_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTN144_SMEM));
                configured = true;
            }
            GTAV_CUDA_OK(launch_k(attn_seq144_kernel, dim3(3, heads, groups), dim3(3 * 32), ATTN144_SMEM, s, qkv, out, heads, rot));
        } else {
            GTAV_CUDA_OK(launch_k(attn_seq_kernel<144, 144, 3, 32>, dim3(3, heads, groups), dim3(3 * 32), 0, s, qkv, out, heads, rot));
        }
    } else if (seq == 576 && rot_pairs == 16) {
        GTAV_CUDA_OK(launch_k(attn_seq_kernel<576, 64, 4, 16>, dim3(9, heads, groups), dim3(4 * 32), 0, s, qkv, out, heads, rot));
    } else {
        set_error("attention: unsupported (seq=%d, rot_pairs=%d); built for (144,32) and (576,16)", seq, rot_pairs);
        return -1;
    }
    return 0;
}

}  // namespace gtav
