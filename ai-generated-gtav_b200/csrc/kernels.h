// Internal host-side interface between the engines (dit_engine.cu, vae_engine.cu, sampler.cu) and
// the kernel translation units.  Nothing here is exported; the C ABI lives in include/gtav_b200.h.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace gtav {

typedef __nv_bfloat16 bf16;

// thread-local error text returned by gtav_last_error()
void set_error(const char* fmt, ...);
const char* get_error();
#define GTAV_CUDA_OK(expr)                                                                     \
    do {                                                                                       \
        cudaError_t e__ = (expr);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            gtav::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return -2;                                                                         \
        }                                                                                      \
    } while (0)

// Launch with the programmatic-dependent-launch attribute (see common.cuh: pdl_wait / pdl_trigger).
// GTAV_PDL=0 in the environment turns the attribute off (plain stream order) for A/B measurements.
bool pdl_enabled();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- GEMM (gemm_sm100.cu)
enum Epilogue : int {
    EPI_STORE = 0,           // out = bf16(acc)
    EPI_BIAS = 1,            // out = bf16(acc + b)
    EPI_BIAS_GELU_TANH = 2,  // out = bf16(gelu_tanh(bf16(acc + b)))
    EPI_BIAS_GELU_ERF = 3,   // out = bf16(gelu_erf(bf16(acc + b)))
    EPI_BIAS_SILU = 4,       // out = bf16(silu(bf16(acc + b)))
    EPI_BIAS_GATE_RES = 5,   // out = bf16(res + bf16(gate * bf16(acc + b)))
    EPI_BIAS_RES = 6,        // out = bf16(res + bf16(acc + b))
    EPI_BIAS_RES_SILU = 7,   // out = bf16(silu(bf16(res + bf16(acc + b))))   (res may be null)
    EPI_COUNT = 8
};

struct GemmParams {
    bf16* out; int ldo;
    const bf16* bias;
    const bf16* res; int ldr;
    const bf16* gate; int gate_ld;      // gate vector of row r: gate + frame_row[r / rows_per_frame] * gate_ld
    const int* frame_row;               // null => identity
    int rows_per_frame;
    int M, N, K;
    // Weights of the NEXT GEMM in the stream (or null): every CTA asks the TMA unit to pull its share into L2 at
    // kernel start, so the next kernel's first loads are L2 hits instead of ~2 us HBM round trips.
    const void* prefetch;
    size_t prefetch_bytes;
};

struct GemmOp {
    CUtensorMap tmA, tmB;
    CUtensorMap tmB2;   // CTA-pair kernel (gemm_sm100_2cta.cu): boxes of 128 weight rows (each CTA loads half of a 256-wide tile)
    int two_cta;        // 1: run the cta_group::2 kernel
    int split_k;        // 1: run the split-K pair kernel (gemm_sm100_splitk.cu): few tiles, long K
    GemmParams p;
    int bn;      // tile width chosen at prepare time (64 / 128 / 256)
    int kc;      // 64-wide K chunks per TMA instruction / pipeline stage (1: 2-D maps, any K; 2: 3-D maps, K % 64 == 0)
    int epi;
};

// out[M,N] = epilogue(A[M,K] @ W[N,K]^T); A, W row-major bf16 with leading dimensions lda / ldw
// (elements, multiples of 8; base pointers 16-byte aligned).  bn_override = 0 picks the tile width.
int gemm_prepare(GemmOp* op, const bf16* A, int lda, const bf16* W, int ldw, const GemmParams& p, int epi,
                 int bn_override = 0);
int gemm_run(const GemmOp* op, cudaStream_t stream);
// CTA-pair variant (tcgen05.mma.cta_group::2, 256 x 256 tiles): M >= 256, N % 256 == 0, K % 128 == 0
bool gemm2_eligible(int M, int N, int K);
int gemm2_run(const GemmOp* op, cudaStream_t stream);
// Split-K variant (two CTAs of a cluster share a 128 x 128 tile, half of K each, DSMEM reduce): K >= 2048, K % 256 == 0,
// N % 128 == 0 and 2 x tiles <= SMs
bool gemm_splitk_eligible(int M, int N, int K, int sms);
int gemm_splitk_run(const GemmOp* op, cudaStream_t stream);

// [rows, cols] bf16 row-major (leading dimension ld) viewed as [64 | rows | cols/64]: boxes of
// box_rows x (box_chunks * 64) land in shared memory as box_chunks consecutive 128-byte-swizzled
// (box_rows x 64) tiles - one TMA instruction per multi-chunk slab.
int make_tmap_3d(CUtensorMap* out, const bf16* ptr, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                 uint32_t box_chunks);

// ---------------------------------------------------------------- weight-streaming GEMM (gemm_skinny.cu)
// Same contract as the GEMM above for M = 144 * {1,2,3} token rows (last-frame DiT step): operands swapped
// (weights on the UMMA M side), K split over CTAs with an in-kernel deterministic reduction.
// Row-wise work fused into the split-K reduce (every CTA then owns whole token rows, see gemm_skinny.cu):
//   SK_FUSE_LN    (N = 1024, EPI_BIAS_GATE_RES): besides out (the new residual stream), ln_out [M, 1024] receives
//                 LN(out row) * (1 + scale) + shift with shift / scale at ln_mod + frame * ln_mod_ld + {ln_shift_off, ln_scale_off}
//                 (frame from the GEMM's frame_row / rows_per_frame) - the launch_ln_modulate that would follow;
//   SK_FUSE_TATTN (N = 3072, EPI_STORE, 4 splits): out [M, 1024] receives the last-frame temporal attention of the q|k|v
//                 row against kv_cache (launch_attention_temporal_last's arguments) instead of the row itself.
enum SkinnyFuse : int { SK_FUSE_NONE = 0, SK_FUSE_LN = 1, SK_FUSE_TATTN = 2 };
struct SkinnyFuseParams {
    int mode;
    bf16* ln_out;
    const bf16* ln_mod;
    int ln_mod_ld, ln_shift_off, ln_scale_off;
    const bf16* kv_cache;
    const float2* rot;
    int ctx_frames, positions;
};
struct SkinnyOp {
    CUtensorMap tmW, tmA;
    GemmParams p;
    SkinnyFuseParams f;
    int grid;         // CTAs launched: (N/128) * splits, or more in the fused modes (reduce-only CTAs)
    int epi, splits, chunks, tiles;
    float* ws;        // fp32 partial-sum workspace, skinny_workspace_bytes(M)
    int* counters;    // 512 ints, zero before the first launch (rendezvous groups of 4 ints, maintained by the kernel)
    int tag;          // 0 (skinny_prepare's default): CTAs meet on `counters`.  2 | parity: tagged partial sums, no rendezvous -
                      // the caller owns the protocol: `ws` is used by launches of THIS shape and split only, was zeroed once,
                      // and consecutive launches on it alternate the parity starting with 1 (gemm_skinny.cu, SkTag)
    long long* trace; // optional phase time stamps [CTAs][8] (profiling aid), normally null
};
bool skinny_supported(int M, int N, int K, int epi);
int skinny_pick_splits(int M, int N, int K);
size_t skinny_workspace_bytes(int M);
int skinny_prepare(SkinnyOp* op, const bf16* A, int lda, const bf16* W, int ldw, const GemmParams& p, int epi, float* ws,
                   int* counters, int splits_override = 0, const SkinnyFuseParams* fuse = nullptr);
int skinny_run(const SkinnyOp* op, cudaStream_t stream);

// ---------------------------------------------------------------- row kernels (norm_mod.cu)
// out = bf16( LN(x) * bf16(1 + bf16(scale + 1e-6)) + shift ), LN without affine, eps 1e-6.
// shift/scale of row r live at mod + frame_row[r / rows_per_frame] * mod_ld + {shift_off, scale_off}.
int launch_ln_modulate(const bf16* x, bf16* out, int M, int D, const bf16* mod, int mod_ld, int shift_off,
                       int scale_off, const int* frame_row, int rows_per_frame, cudaStream_t s);
// out = bf16( LN(x) * w + b ), fp32 affine parameters (VAE).
int launch_ln_affine(const bf16* x, bf16* out, int M, int D, const float* w, const float* b, cudaStream_t s);

// ---------------------------------------------------------------- attention (attn_mma.cu, attn_temporal.cu)
// qkv [rows, 3*H*64] (q | k | v, head-major inside each), out [rows, H*64].  One problem per
// (group of `seq` consecutive rows, head).  rot: float2 (cos, sin) [seq][rot_pairs] applied to the
// first 2*rot_pairs features of q and k.  seq must be 144 (DiT spatial) or 576 (VAE).
int launch_attention_seq(const bf16* qkv, bf16* out, int groups, int seq, int heads, const float2* rot, int rot_pairs,
                         cudaStream_t s);
// The same op on tcgen05 tensor cores (attn_tc.cu): S = Q K^T and O = P V as UMMA tiles with TMEM accumulators.
int launch_attention_tc(const bf16* qkv, bf16* out, int groups, int seq, int heads, const float2* rot, int rot_pairs,
                        cudaStream_t s);
// Causal attention over the T frames of each (b, spatial position, head); rows ordered (b, t, pos).
// rot: float2 [T][32] window-relative angles.  kv_cache (optional) [B*T*positions, 2*H*64]: receives the rotated
// K and the V of every row, for later last-frame-only steps.
int launch_attention_temporal(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                              bf16* kv_cache, cudaStream_t s);
// The same attention for the LAST frame of a (ctx_frames + 1)-frame window only: qkv / out hold the last-frame
// rows [B*positions, ...], the context frames' K/V come from kv_cache [B*ctx_frames*positions, 2*H*64].
int launch_attention_temporal_last(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                   const float2* rot, const bf16* kv_cache, cudaStream_t s);
// Ragged windows: rollout b of a pass over `frames` slots has valid frames only in its trailing slots, at rotary positions
// 0, 1, ... from the first valid slot; the slots before are padding.  The count is read on the device at launch time:
// valid(b) = min(max(len[b], lo), frames + sub) - sub, so a bad length gives wrong numbers, never an out-of-range access.
// A DiT plan passes its window lengths with lo = 1 and sub = the window frames the pass does not cover (0 for a full
// window, 1 for the context and last-frame passes); the stand-alone entry points pass per-rollout counts with lo = sub = 0.
struct TemporalLens {
    const int* len;   // device int32 [B]
    int lo, sub;
};
// Long windows (attn_temporal_long.cu), reached through the launchers above and below: T = 9..32, ctx_frames = 8..31;
// lens == nullptr: every window full.
int launch_attention_temporal_long(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                                   bf16* kv_cache, const TemporalLens* lens, cudaStream_t s);
int launch_attention_temporal_last_long(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                        const float2* rot, const bf16* kv_cache, const TemporalLens* lens, cudaStream_t s);
// launch_attention_temporal with rollout b's valid frames in its trailing valid(b) slots (attending to valid keys only,
// rotated at rot[slot - first valid slot]); padded rows get output 0 and, with kv_cache, cache rows 0.  T = 1..32.
int launch_attention_temporal_ragged(const bf16* qkv, bf16* out, int B, int T, int positions, int heads, const float2* rot,
                                     bf16* kv_cache, TemporalLens lens, cudaStream_t s);
// launch_attention_temporal_last against the trailing valid(b) of the ctx_frames cached slots of rollout b, the query at
// rotary position valid(b).  ctx_frames = 0..31.
int launch_attention_temporal_last_ragged(const bf16* qkv, bf16* out, int B, int ctx_frames, int positions, int heads,
                                          const float2* rot, const bf16* kv_cache, TemporalLens lens, cudaStream_t s);

// ---------------------------------------------------------------- conditioning / patches / sampler (elementwise.cu)
// temb[r, 0:128] = cos(t_r f), temb[r,128:256] = sin(t_r f) (bf16); aemb[r,:] = bf16(act_r @ Wa^T + ba) if actions.
int launch_cond_prep(const int64_t* t, const float* actions, int act_dim, int R, const float* freqs, const bf16* Wa,
                     const bf16* ba, bf16* temb, bf16* aemb, int D, cudaStream_t s);
// x [F, C, H, W] (fp32 or bf16) -> patches [F*(H/p)*(W/p), ldo] bf16, k = c*p*p + ph*p + pw, zero padded to ldo.
// Frames come in groups of frames_per_group contiguous frames whose starts are group_stride elements apart
// (a sub-window of every rollout of a [B, T, C, H, W] tensor); frames_per_group <= 0 = all F frames contiguous.
int launch_patchify(const void* x, int x_is_bf16, bf16* out, int ldo, int F, int C, int H, int W, int p,
                    int frames_per_group, long group_stride, cudaStream_t s);
// DiT un-patchify: y [F*gh*gw, p*p*C] -> v [F, C, gh*p, gw*p] bf16, feature = ph*(p*C) + pw*C + c.
int launch_dit_unpatchify(const bf16* y, bf16* out, int F, int C, int gh, int gw, int p, cudaStream_t s);
// VAE un-patchify: y [F*sh*sw, 3*p*p] -> img [F,3,sh*p,sw*p] bf16 (feature = c*p*p + ph*p + pw), or, with
// to_u8, the fused pixel epilogue of generate.py:241-244 -> uint8 [F, sh*p, sw*p, 3].
int launch_vae_unpatchify(const bf16* y, void* out, int to_u8, int F, int sh, int sw, int p, cudaStream_t s);
// z [rows, C] float (scaled by `scale`) -> bf16 [rows, ldo] zero padded.
int launch_cast_pad(const float* z, bf16* out, int rows, int C, int ldo, float scale, cudaStream_t s);
// moments [rows, ldm] bf16 -> mean [rows, C] float (= first C columns), times `scale` rounded to bf16 if round_bf16.
int launch_take_mean(const bf16* moments, int ldm, float* out, int rows, int C, float scale, int round_bf16,
                     cudaStream_t s);
// v-prediction DDIM update (train_dit.py:110-123) over F frames of n elements (frame f at ptr + f*stride);
// abar_t / abar_next per frame; *final_flag selects the x0 return of noise_idx <= 0.
int launch_ddim(const float* x, long x_stride, const bf16* v, long v_stride, float* out, long out_stride, int F, int n,
                const float* abar_t, const float* abar_next, const int* final_flag, cudaStream_t s);
// Sampler bookkeeping for one DDIM step, read from / written to device memory so a captured graph can be
// replayed: k = *counter; frame_row [B*T], last_row [B] (conditioning row of each rollout's last frame), abar_t,
// abar_next, final_flag for step k; *counter = k - 1.
int launch_step_prep(int* counter, const int* levels, const float* abar, int B, int T, int steps, int* frame_row,
                     int* last_row, float* abar_t, float* abar_next, int* final_flag, cudaStream_t s);
int launch_set_int(int* dst, int value, cudaStream_t s);
// x[f*stride + i] = clamp(noise[f*n + i], -amax, amax)  (generate.py:201-203)
int launch_noise_clamp(const float* noise, float* x, long x_stride, int F, int n, float amax, cudaStream_t s);

}  // namespace gtav
