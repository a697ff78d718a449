/* gtav_b200 - C ABI of the B200-native inference hot path of AI-Generated-GTAV.
 *
 * The reference has no plugin / FFI layer: its "API" is the Python surface
 *   model/dit.py:343   DiT.forward(x, t, external_cond)
 *   model/vae.py:306   AutoencoderKL.encode(x) / :324 decode(z)
 *   train_dit.py:31    denoise_step(...)
 *   generate.py:200    the autoregressive sampling loop
 * so this header DEFINES the boundary one level below those signatures (SURVEY.md section 8(b)).
 * Each entry point names the reference code it stands in for.  Conventions:
 *   - plain C types only; device pointers are raw addresses owned by the caller (PyTorch's
 *     allocator in the shipped binding) and must stay valid until the stream has consumed them;
 *   - every call only ENQUEUES work on the given cudaStream_t (no host synchronisation, so calls
 *     are capturable into CUDA graphs) unless documented otherwise;
 *   - return value 0 = ok, negative = error; gtav_last_error() returns the thread-local message;
 *   - all matrices are row-major bf16 unless stated; weights are the reference's fp32 parameters
 *     rounded to bf16 (round-to-nearest-even, what torch.autocast's cast produces).
 * There is no CPU fallback: without an sm_100a device every compute call fails.
 */
#ifndef GTAV_B200_H
#define GTAV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

typedef struct CUstream_st* gtav_stream_t; /* == cudaStream_t */

const char* gtav_last_error(void);
/* ABI version; bumped on any signature change or new entry point (4: gtav_gemm_skinny_tagged_bf16, larger DiT plan workspace;
 * 5: gtav_gemm_skinny_fused_bf16). */
int gtav_abi_version(void);

/* ------------------------------------------------------------------------------------------
 * Stand-alone kernels (exported for parity tests and for callers that compose their own graph)
 * ------------------------------------------------------------------------------------------ */
enum gtav_epilogue {
    GTAV_EPI_STORE = 0,          /* out = bf16(acc)                                   to_qkv (attention.py:27,86) */
    GTAV_EPI_BIAS = 1,           /* out = bf16(acc + b)                               any nn.Linear with bias */
    GTAV_EPI_BIAS_GELU_TANH = 2, /* out = bf16(gelu_tanh(bf16(acc + b)))              DiT Mlp.fc1 (dit.py:161,171) */
    GTAV_EPI_BIAS_GELU_ERF = 3,  /* out = bf16(gelu(bf16(acc + b)))                   VAE Mlp.fc1 (vae.py:128,147) */
    GTAV_EPI_BIAS_SILU = 4,      /* out = bf16(silu(bf16(acc + b)))                   t_embedder.mlp[0:2] (dit.py:86-90) */
    GTAV_EPI_BIAS_GATE_RES = 5,  /* out = bf16(res + bf16(gate * bf16(acc + b)))      x + gate(f(x), g) (dit.py:207-223) */
    GTAV_EPI_BIAS_RES = 6,       /* out = bf16(res + bf16(acc + b))                   VAE residuals (vae.py:155-156) */
    GTAV_EPI_BIAS_RES_SILU = 7   /* out = bf16(silu(bf16(res + bf16(acc + b))))       c = t_emb + cond; SiLU(c) (dit.py:362-364,177) */
};

/* out[M,N] = epilogue(A[M,K] @ W[N,K]^T) on the tcgen05 GEMM.  lda/ldw/ldo/ldr/gate_ld in elements
 * (multiples of 8).  gate row of output row r is gate + frame_row[r / rows_per_frame] * gate_ld
 * (frame_row NULL = identity).  bn = 0 lets the library pick the tile width (64/128/256) and, for multi-round
 * shapes with N % 256 == 0 and K % 128 == 0, the CTA-pair kernel (tcgen05.mma.cta_group::2, 256x256 tile pairs);
 * both produce the same bits. */
int gtav_gemm_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                   int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                   const int* frame_row, int rows_per_frame, int bn, gtav_stream_t stream);

/* The same contract on the weight-streaming kernel used for last-frame steps: M = 144, 288 or 432 rows, N a
 * multiple of 128, K of 64; epilogues STORE / BIAS / BIAS_GELU_TANH / BIAS_GATE_RES (rows_per_frame must be 144).
 * workspace: fp32 scratch of gtav_gemm_skinny_workspace_bytes(M) bytes; counters: 512 ints, zero before the first
 * call (rendezvous state the kernel maintains itself from then on; do not share between concurrent streams).  splits = 0 lets the library pick the K split. */
size_t gtav_gemm_skinny_workspace_bytes(int M);
int gtav_gemm_skinny_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                          int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                          const int* frame_row, int rows_per_frame, int splits, void* workspace, int* counters,
                          gtav_stream_t stream);
/* The same GEMM with the split-K exchange the DiT engine uses for its last-frame passes (csrc/gemm_skinny.cu, SkTag): the
 * partial sums carry the launch's parity in their last mantissa bit and the reducing CTAs accept an element once it shows
 * it - no fence, counter or poll between the two halves of the kernel.  The caller owns the protocol: `workspace` is used
 * by launches of ONE (M, N, K, splits) shape only, was zeroed before the first of them, and parity alternates 1, 0, 1, 0 ...
 * from launch to launch on it (a captured graph must hold an even number of them).  A parity out of step fails the launch
 * (trap after a bounded spin) instead of hanging.  Results differ from gtav_gemm_skinny_bf16 by that cleared bit of
 * each fp32 partial sum only. */
int gtav_gemm_skinny_tagged_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                                 int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                                 const int* frame_row, int rows_per_frame, int splits, void* workspace, int parity,
                                 gtav_stream_t stream);
/* The same GEMM with the row-wise kernel that follows it in a last-frame DiT pass folded into its split-K reduce, as the
 * engine runs to_out / fc2 and the temporal to_qkv.  The mode fixes the epilogue:
 *   mode 1 (LayerNorm): N = 1024, 4, 8 or 16 splits, epilogue BIAS_GATE_RES with 144 rows per frame (res may be out).  out
 *          receives the new residual stream; ln_out [M, 1024] (contiguous) receives gtav_ln_modulate of those rows with shift /
 *          scale at ln_mod + frame * ln_mod_ld + {ln_shift_off, ln_scale_off}, frame from frame_row as for the gate;
 *   mode 2 (temporal attention): N = 3072 (q | k | v of 16 heads), 4 splits, epilogue STORE.  out [M, 1024] receives
 *          gtav_attention_temporal_last of the q|k|v rows (B = M / positions) against kv_cache with ctx_frames (0..7) cached
 *          frames and rot [ctx_frames + 1][32] (cos, sin); the q|k|v rows themselves are not stored.
 * Both give the bits of the unfused launch followed by gtav_ln_modulate / gtav_attention_temporal_last.  parity -1: the CTAs
 * meet on `counters` (as gtav_gemm_skinny_bf16); 0 or 1: tagged exchange under the protocol of gtav_gemm_skinny_tagged_bf16
 * (counters unused).  All CTAs of a launch (one per token row, up to the SM count) must be co-resident. */
int gtav_gemm_skinny_fused_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                                const void* bias, const void* res, int ldr, const void* gate, int gate_ld, const int* frame_row,
                                int splits, void* workspace, int* counters, int mode, void* ln_out, const void* ln_mod,
                                int ln_mod_ld, int ln_shift_off, int ln_scale_off, const void* kv_cache, const float* rot,
                                int ctx_frames, int positions, int parity, gtav_stream_t stream);

/* modulate(LayerNorm(x), shift, scale) of dit.py:19-27 -> bf16 [M, D]; D = 1024. */
int gtav_ln_modulate(const void* x, void* out, int M, int D, const void* mod, int mod_ld, int shift_off, int scale_off,
                     const int* frame_row, int rows_per_frame, gtav_stream_t stream);
/* nn.LayerNorm(D, eps=1e-6) with fp32 affine parameters (vae.py:132,145,209,232) -> bf16. */
int gtav_ln_affine(const void* x, void* out, int M, int D, const float* w, const float* b, gtav_stream_t stream);
/* Non-causal attention with fused rotary over groups of `seq` consecutive rows (attention.py:99-129, vae.py:78-107).
 * qkv [groups*seq, 3*heads*64], out [groups*seq, heads*64], rot = (cos,sin) float pairs [seq][rot_pairs]. */
int gtav_attention_seq(const void* qkv, void* out, int groups, int seq, int heads, const float* rot, int rot_pairs,
                       gtav_stream_t stream);
/* Causal attention over T = 1..32 frames with fused rotary (attention.py:41-66); rows ordered (b, t, position);
 * rot = (cos,sin) [>= T][32].  Any other T is refused before a launch. */
int gtav_attention_temporal(const void* qkv, void* out, int B, int T, int positions, int heads, const float* rot,
                            gtav_stream_t stream);
/* The last frame of that attention only, against cached context K/V: qkv / out hold the last-frame rows
 * [B*positions, ...]; kv_cache [B*ctx_frames*positions, 2*heads*64] = (rotated K | V) of window frames
 * 0..ctx_frames-1, rows ordered (b, t, position); the query sits at window position ctx_frames.  ctx_frames = 0..31
 * (rot rows >= ctx_frames + 1); any other count is refused before a launch.  Same bits as row ctx_frames of
 * gtav_attention_temporal over ctx_frames + 1 frames. */
int gtav_attention_temporal_last(const void* qkv, void* out, int B, int ctx_frames, int positions, int heads,
                                 const float* rot, const void* kv_cache, gtav_stream_t stream);
/* DDIM update of train_dit.py:110-123 over F frames of n elements. */
int gtav_ddim_update(const float* x, const void* v_bf16, float* out, int F, int n, const float* abar_t,
                     const float* abar_next, const int* final_flag, gtav_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * DiT (stands in for model/dit.py:228-376 DiT + model/attention.py)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int depth;        /* number of SpatioTemporalDiTBlocks (16) */
    int hidden;       /* 1024 */
    int heads;        /* 16 (head dim 64) */
    int grid_h, grid_w; /* token grid: 9 x 16 */
    int patch;        /* 2 */
    int in_channels;  /* 16 */
    int act_dim;      /* external_cond_dim: 25, or 0 */
    int max_frames;   /* sliding-window length, 1..32: rows in rot_temporal */
} gtav_dit_config;

typedef struct {
    const void *qkv_w;            /* [3D, D]   blocks.N.{s,t}_attn.to_qkv.weight */
    const void *out_w, *out_b;    /* [D, D],[D]         ..._attn.to_out */
    const void *fc1_w, *fc1_b;    /* [4D, D],[4D]       ..._mlp.fc1 */
    const void *fc2_w, *fc2_b;    /* [D, 4D],[D]        ..._mlp.fc2 */
} gtav_dit_half;

typedef struct {
    const void *patch_w, *patch_b;   /* [D, C*p*p],[D]   x_embedder.proj (conv weight flattened) */
    const void *t0_w, *t0_b;         /* [D, 256],[D]     t_embedder.mlp.0 */
    const void *t2_w, *t2_b;         /* [D, D],[D]       t_embedder.mlp.2 */
    const void *act_w, *act_b;       /* [D, act_dim],[D] external_cond (NULL if act_dim == 0) */
    const void *ada_w, *ada_b;       /* [depth*2*6D + 2D, D] and bias: adaLN_modulation.1 of block0.s, block0.t, ..., final_layer */
    const void *final_w, *final_b;   /* [p*p*C, D],[p*p*C] final_layer.linear */
    const float* temb_freqs;         /* [128] exp(-ln(1e4) i/128) (dit.py:107-111) */
    const float* rot_spatial;        /* (cos,sin) [grid_h*grid_w][32] axial "pixel" angles (rotary...:290-317) */
    const float* rot_temporal;       /* (cos,sin) [max_frames][32], max_frames <= 32 rows (rotary...:186-209) */
    const gtav_dit_half* halves;     /* [2*depth]: block0.s, block0.t, block1.s, ... */
} gtav_dit_weights;

typedef struct gtav_dit_s* gtav_dit_t;
typedef struct gtav_dit_plan_s* gtav_dit_plan_t;

int gtav_dit_create(const gtav_dit_config* cfg, const gtav_dit_weights* w, gtav_dit_t* out);
void gtav_dit_destroy(gtav_dit_t h);
/* Width of one modulation row: depth*2*6*hidden + 2*hidden. */
int gtav_dit_mod_width(gtav_dit_t h);

/* A plan fixes (B, T) and owns the TMA descriptors for a caller-provided workspace.
 * cond_rows = rows of the conditioning table (B*T for a plain forward).
 * stream: the stream the plan's passes will be enqueued on - the split-K rendezvous counters inside the workspace are
 * cleared with a cudaMemsetAsync on it, i.e. ordered after whatever used that (possibly recycled) memory before and
 * before the plan's first kernel. */
size_t gtav_dit_workspace_bytes(gtav_dit_t h, int B, int T, int cond_rows);
int gtav_dit_plan_create(gtav_dit_t h, int B, int T, int cond_rows, void* workspace, size_t workspace_bytes,
                         gtav_stream_t stream, gtav_dit_plan_t* out);
void gtav_dit_plan_destroy(gtav_dit_plan_t p);

/* Conditioning table: SiLU(t_embedder(t) + external_cond(a)) -> all adaLN modulation vectors
 * (dit.py:359-364 and the adaLN_modulation of 137-139,177-179,196-198) for cond_rows rows.
 * t: int64 [cond_rows] on device; actions: fp32 [cond_rows, act_dim] on device or NULL. */
int gtav_dit_conditioning(gtav_dit_plan_t p, const int64_t* t, const float* actions, gtav_stream_t stream);
/* Backbone: patch-embed -> blocks -> final layer -> un-patchify.  x [B,T,C,H,W] fp32 (x_is_bf16=0) or
 * bf16; frame_row int32 [B*T] on device maps each frame to its conditioning-table row (NULL = identity);
 * out bf16 [B,T,C,H,W]. */
int gtav_dit_backbone(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, void* out,
                      gtav_stream_t stream);
/* The backbone split along the frame axis for the sampler's frame cache.  Spatial attention is per frame and
 * temporal attention is causal over frames (attention.py:62 is_causal=True), so frames 0..T-2 do not depend on
 * frame T-1:
 *   gtav_dit_context   runs frames 0..T-2 of every rollout of the window x [B,T,C,H,W] and stores, for every
 *                      temporal layer, their rotated K and V in the plan's cache (no output; frame_row int32
 *                      [B*(T-1)] or NULL = identity);
 *   gtav_dit_last_frame runs frame T-1 only (144*B rows) against that cache; frame_row int32 [B] (NULL =
 *                      identity); out bf16 [B,C,H,W] = the last frame of what gtav_dit_backbone returns. */
int gtav_dit_context(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, gtav_stream_t stream);
int gtav_dit_last_frame(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, void* out,
                        gtav_stream_t stream);
/* DiT.forward(x, t, external_cond) = conditioning + backbone with cond_rows == B*T. */
int gtav_dit_forward(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int64_t* t, const float* actions,
                     void* out, gtav_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * VAE (stands in for model/vae.py:160-338 AutoencoderKL encode / decode)
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int dim, heads, enc_depth, dec_depth, latent_dim, patch, seq_h, seq_w;
} gtav_vae_config;

typedef struct {
    const float *norm1_w, *norm1_b, *norm2_w, *norm2_b;  /* fp32 [D] */
    const void *qkv_w, *qkv_b, *proj_w, *proj_b, *fc1_w, *fc1_b, *fc2_w, *fc2_b;
} gtav_vae_block;

typedef struct {
    const void *patch_w, *patch_b;     /* [D, 3*p*p (ld padded to a multiple of 8)], [D] */
    const float *enc_norm_w, *enc_norm_b, *dec_norm_w, *dec_norm_b;
    const void *quant_w, *quant_b;     /* [2*latent, D] */
    const void *post_w, *post_b;       /* [D, 64] (K zero-padded from latent_dim to 64) */
    const void *pred_w, *pred_b;       /* [3*p*p, D] */
    const float* rot;                  /* (cos,sin) [seq_h*seq_w][16] */
    const gtav_vae_block* enc;         /* [enc_depth] */
    const gtav_vae_block* dec;         /* [dec_depth] */
} gtav_vae_weights;

typedef struct gtav_vae_s* gtav_vae_t;
typedef struct gtav_vae_plan_s* gtav_vae_plan_t;

int gtav_vae_create(const gtav_vae_config* cfg, const gtav_vae_weights* w, gtav_vae_t* out);
void gtav_vae_destroy(gtav_vae_t h);
size_t gtav_vae_workspace_bytes(gtav_vae_t h, int n_frames);
int gtav_vae_plan_create(gtav_vae_t h, int n_frames, void* workspace, size_t workspace_bytes, gtav_vae_plan_t* out);
void gtav_vae_plan_destroy(gtav_vae_plan_t p);
/* img [N,3,H,W] (fp32 or bf16, already in [-1,1]) -> mean_out fp32 [N, seq, latent] = bf16 mean * scale,
 * re-rounded to bf16 when round_bf16 (generate.py:56 multiplies a bf16 tensor). */
int gtav_vae_encode(gtav_vae_plan_t p, const void* img, int img_is_bf16, float* mean_out, float scale, int round_bf16,
                    gtav_stream_t stream);
/* Both halves of the posterior (DiagonalGaussianDistribution, model/vae.py:19-45: torch.chunk(moments, 2)): mean_out and
 * logvar_out fp32 [N, seq, latent] holding the bf16 values of quant_conv's output, unclamped. */
int gtav_vae_encode_moments(gtav_vae_plan_t p, const void* img, int img_is_bf16, float* mean_out, float* logvar_out,
                            gtav_stream_t stream);
/* z fp32 [N, seq, latent], divided by `divisor` first (generate.py:241) -> out: bf16 [N,3,H,W] (to_u8 = 0)
 * or uint8 [N,H,W,3] with the pixel epilogue of generate.py:241-244 fused (to_u8 = 1). */
int gtav_vae_decode(gtav_vae_plan_t p, const float* z, float divisor, void* out, int to_u8, gtav_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Sampler (stands in for the per-frame loop of generate.py:204-220 around train_dit.py:30-125)
 * ------------------------------------------------------------------------------------------ */
typedef struct gtav_sampler_s* gtav_sampler_t;

/* Rows of the per-frame conditioning table a sampler plan needs: B*(T-1) context rows (row b*(T-1)+j for
 * window frame j of rollout b, t = stabilisation level) followed by B*(steps+1) last-frame rows
 * (row B*(T-1) + b*(steps+1) + k for noise level k).  Create the DiT plan with this cond_rows and fill the
 * table with gtav_dit_conditioning once per generated frame. */
int gtav_sampler_cond_rows(int B, int T, int steps);
size_t gtav_sampler_scratch_bytes(int B, int T, int steps);
enum gtav_sampler_flags {
    GTAV_SAMPLER_GRAPH = 1,       /* capture the frame's steps into a CUDA graph (stream must not be the legacy default stream) */
    GTAV_SAMPLER_FRAME_CACHE = 2  /* context pass once per frame + last-frame-only steps (same results, ~4.8x fewer FLOPs) */
};
/* x_win: fp32 [B,T,frame_elems] window (caller loads context frames + clamped noise before each frame);
 * v_out: bf16 [B,T,frame_elems] scratch for the v-prediction; abar_dev: fp32 alphas_cumprod on device;
 * levels_host: int[steps+1] integer timesteps (linspace(0,999,steps+1) truncated); flags: gtav_sampler_flags.
 * This call synchronises `stream` once (copies levels). */
int gtav_sampler_create(gtav_dit_plan_t plan, int B, int T, int steps, int frame_elems, float* x_win, void* v_out,
                        const float* abar_dev, const int* levels_host, void* scratch, size_t scratch_bytes, int flags,
                        gtav_stream_t stream, gtav_sampler_t* out);
void gtav_sampler_destroy(gtav_sampler_t s);
/* Runs noise levels steps, steps-1, ..., down to (steps+1-n_steps) on the window (n_steps < 0: all steps+1).
 * With GTAV_SAMPLER_GRAPH the first call runs eagerly and captures (synchronising the stream once); later calls
 * replay one graph per frame (all steps) or per step (partial runs). */
int gtav_sampler_run_frame(gtav_sampler_t s, int n_steps, gtav_stream_t stream);
/* x[f*x_stride + i] = clamp(noise[f*n + i], -amax, +amax): the fresh frame of generate.py:201-203. */
int gtav_noise_clamp(const float* noise, float* x, long x_stride, int F, int n, float amax, gtav_stream_t stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* GTAV_B200_H */
