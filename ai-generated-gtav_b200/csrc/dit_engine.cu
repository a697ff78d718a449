// Host-side DiT engine: owns the per-(B,T) launch plan (TMA descriptors, workspace carve-up) and
// enqueues the kernel sequence that stands in for DiT.forward (reference model/dit.py:343-376) and
// SpatioTemporalDiTBlock.forward (model/dit.py:200-225).  No allocation, no host sync: everything is
// launched on the caller's stream so a whole step can be captured into a CUDA graph.
#include <stdlib.h>

#include <new>
#include <vector>

#include "../../include/gtav_b200.h"
#include "kernels.h"

using namespace gtav;

struct gtav_dit_s {
    gtav_dit_config cfg;
    gtav_dit_weights w;
    std::vector<gtav_dit_half> halves;
    int tokens;       // grid_h * grid_w
    int mod_width;    // depth*2*6D + 2D
    int patch_k;      // C*p*p
    int out_feat;     // p*p*C
};

// GEMM launch descriptors for one row count (B * frames * tokens rows) over the plan's shared workspace.
struct Shape {
    int frames = 0, M = 0;
    GemmOp g_patch, g_final;
    std::vector<GemmOp> g_qkv, g_out, g_fc1, g_fc2;
    // weight-streaming variants (last-frame shape only); sk[kind] says whether kind uses them
    std::vector<SkinnyOp> s_qkv, s_out, s_fc1, s_fc2;
    bool sk[4] = {false, false, false, false};
    // row-wise kernels folded into the weight-streaming GEMMs' reduce (gemm_skinny.cu): the LayerNorm + modulate after
    // to_out / fc2, the last-frame temporal attention after the temporal half's to_qkv
    bool fuse_ln = false, fuse_tattn = false;
};

enum BackboneMode { MODE_FULL = 0, MODE_CONTEXT = 1, MODE_LAST = 2 };

struct gtav_dit_plan_s {
    gtav_dit_t eng;
    int B, T, M, R;
    // workspace slices
    bf16 *xa, *h, *hn, *qkv, *att, *mlp, *yfin, *temb, *aemb, *h1, *cact, *mod;
    bf16* kv_cache;          // [depth][B*(T-1)*tokens][2*hidden]: rotated K and V of the context frames per temporal layer
    float* sk_ws;            // split-K partial sums of the weight-streaming GEMM: four regions of sk_ws_bytes, one per GEMM
    size_t sk_ws_bytes;      // kind (to_qkv, to_out, fc1, fc2), so that the tagged exchange sees only its own shape's data
    int* sk_counters;
    bool sk_out_of_step = false;   // a last-frame pass failed part-way: the tagged exchange's parities no longer line up
    GemmOp g_t0, g_t2, g_ada;
    Shape full, ctx, last;   // all T frames / the T-1 context frames / the last frame only
};

namespace {

struct Carver {
    uint8_t* base;
    size_t off = 0;
    explicit Carver(void* p) : base(static_cast<uint8_t*>(p)) {}
    bf16* take(size_t elems) {
        bf16* r = reinterpret_cast<bf16*>(base + off);
        off += (elems * sizeof(bf16) + 1023) & ~size_t(1023);
        return r;
    }
};

void carve(gtav_dit_plan_s* p, void* ws, size_t* total) {
    const gtav_dit_s* e = p->eng;
    const size_t M = p->M, R = p->R, D = e->cfg.hidden;
    Carver c(ws);
    p->xa = c.take(M * 64);
    p->h = c.take(M * D);
    p->hn = c.take(M * D);
    p->qkv = c.take(M * 3 * D);
    p->att = c.take(M * D);
    p->mlp = c.take(M * 4 * D);
    p->yfin = c.take(M * 64);
    p->temb = c.take(R * 256);
    p->aemb = c.take(R * D);
    p->h1 = c.take(R * D);
    p->cact = c.take(R * D);
    p->mod = c.take(R * static_cast<size_t>(e->mod_width));
    // every size in size_t: at 32 frames the K/V caches alone are depth * B * 31 * 144 * 2048 bf16 (2.3 GB for the
    // 16-block DiT at B = 8), past what an int counts in elements
    const size_t ctx_rows = static_cast<size_t>(p->B) * (p->T - 1) * e->tokens;
    p->kv_cache = c.take(static_cast<size_t>(e->cfg.depth) * ctx_rows * 2 * D);
    const int m_last = p->B * e->tokens;
    p->sk_ws_bytes = p->B <= 3 ? skinny_workspace_bytes(m_last) : 0;
    p->sk_ws = reinterpret_cast<float*>(c.take(4 * p->sk_ws_bytes / sizeof(bf16)));
    p->sk_counters = reinterpret_cast<int*>(c.take(1024));      // 512 ints: 4 per rendezvous group (gemm_skinny.cu)
    *total = c.off;
}

GemmParams gp(bf16* out, int ldo, const void* bias, int M, int N, int K) {
    GemmParams p{};
    p.out = out; p.ldo = ldo; p.bias = static_cast<const bf16*>(bias);
    p.M = M; p.N = N; p.K = K; p.rows_per_frame = 1;
    return p;
}

bool skinny_enabled() {
    const char* e = getenv("GTAV_SKINNY");
    return !(e != nullptr && e[0] == '0');
}

// GTAV_SK_TAG=0: the weight-streaming GEMMs' CTAs meet on counters instead of exchanging tagged partial sums (gemm_skinny.cu).
bool tag_enabled() {
    const char* e = getenv("GTAV_SK_TAG");
    return !(e != nullptr && e[0] == '0');
}

// GTAV_FUSE=0 keeps LayerNorm and temporal attention as kernels of their own (same results, bit for bit).
bool fuse_enabled() {
    const char* e = getenv("GTAV_FUSE");
    return !(e != nullptr && e[0] == '0');
}

// Descriptors of the backbone GEMMs for `frames` frames per rollout.  allow_skinny: use the weight-streaming
// kernel where the shape fits it (last-frame steps of at most 3 rollouts).
int build_shape(gtav_dit_plan_s* p, Shape* sh, int frames, bool allow_skinny) {
    const gtav_dit_s* h = p->eng;
    const int D = h->cfg.hidden, S = h->tokens, W = h->mod_width;
    const int M = p->B * frames * S;
    const gtav_dit_weights& w = h->w;
    sh->frames = frames;
    sh->M = M;
    int rc = 0;
    rc |= gemm_prepare(&sh->g_patch, p->xa, 64, static_cast<const bf16*>(w.patch_w), 64, gp(p->h, D, w.patch_b, M, D, 64), EPI_BIAS);
    const int nh = 2 * h->cfg.depth;
    sh->g_qkv.resize(nh); sh->g_out.resize(nh); sh->g_fc1.resize(nh); sh->g_fc2.resize(nh);
    // Measured in the real step (B200, B = 1, scripts/bench_graph.py --engine): weight-streaming split-K kernel for all
    // four GEMMs 1.55 ms per last-frame step, tiled kernel for the K = 1024 ones 1.69 ms, tiled everywhere 2.16 ms.
    // GTAV_SKINNY=0 turns the weight-streaming kernel off (tiled GEMM everywhere: bit-identical to the dense window).
    const bool sk_ok = allow_skinny && skinny_enabled() && p->sk_ws != nullptr;
    sh->sk[0] = sk_ok && skinny_pick_splits(M, 3 * D, D) > 0;
    sh->sk[1] = sk_ok && skinny_pick_splits(M, D, D) > 0;
    sh->sk[2] = sk_ok && skinny_pick_splits(M, 4 * D, D) > 0;
    sh->sk[3] = sk_ok && skinny_pick_splits(M, D, 4 * D) > 0;
    if (sh->sk[0]) sh->s_qkv.resize(nh);
    if (sh->sk[1]) sh->s_out.resize(nh);
    if (sh->sk[2]) sh->s_fc1.resize(nh);
    if (sh->sk[3]) sh->s_fc2.resize(nh);
    sh->fuse_ln = sh->sk[1] && sh->sk[3] && fuse_enabled();
    sh->fuse_tattn = sh->sk[0] && fuse_enabled() && skinny_pick_splits(M, 3 * D, D) == 4 && p->T - 1 <= 7;
    const size_t cache_layer = static_cast<size_t>(p->B) * (p->T - 1) * S * 2 * D;
    for (int i = 0; i < nh && rc == 0; ++i) {
        const gtav_dit_half& hw = h->halves[i];
        const bf16* modl = p->mod + static_cast<size_t>(i) * 6 * D;
        GemmParams pq = gp(p->qkv, 3 * D, nullptr, M, 3 * D, D);
        GemmParams po = gp(p->h, D, hw.out_b, M, D, D);
        po.res = p->h; po.ldr = D; po.gate = modl + 2 * D; po.gate_ld = W; po.rows_per_frame = S;
        GemmParams p1 = gp(p->mlp, 4 * D, hw.fc1_b, M, 4 * D, D);
        GemmParams p2 = gp(p->h, D, hw.fc2_b, M, D, 4 * D);
        p2.res = p->h; p2.ldr = D; p2.gate = modl + 5 * D; p2.gate_ld = W; p2.rows_per_frame = S;
        // Each tiled GEMM pulls the next one's weights into L2 while it runs (weights: 2 bytes per element).  Not the
        // weight-streaming kernel: measured in the real step (scripts/bench_graph.py --engine), a prefetch issued at its
        // start competes with its own slab loads (1.208 vs 1.191 ms per step, round 1), and one issued after its MMAs -
        // when HBM is idle - still costs 2 % (1.191 vs 1.169 ms, round 2): the next launch's slab request is not what its
        // critical path waits for.
        const size_t DD = static_cast<size_t>(D) * D * 2;
        if (!sh->sk[0]) { pq.prefetch = hw.out_w; pq.prefetch_bytes = DD; }
        if (!sh->sk[1]) { po.prefetch = hw.fc1_w; po.prefetch_bytes = 4 * DD; }
        if (!sh->sk[2]) { p1.prefetch = hw.fc2_w; p1.prefetch_bytes = 4 * DD; }
        if (!sh->sk[3] && i + 1 < nh) { p2.prefetch = h->halves[i + 1].qkv_w; p2.prefetch_bytes = 3 * DD; }
        // fused reduces: LN2 of this half after to_out, LN1 of the next half (or the final layer's norm) after fc2,
        // temporal attention after the temporal half's to_qkv
        SkinnyFuseParams f_out{}, f_fc2{}, f_qkv{};
        f_out.mode = f_fc2.mode = SK_FUSE_LN;
        f_out.ln_out = f_fc2.ln_out = p->hn;
        f_out.ln_mod = f_fc2.ln_mod = p->mod;
        f_out.ln_mod_ld = f_fc2.ln_mod_ld = W;
        f_out.ln_shift_off = i * 6 * D + 3 * D; f_out.ln_scale_off = i * 6 * D + 4 * D;
        f_fc2.ln_shift_off = (i + 1) * 6 * D; f_fc2.ln_scale_off = (i + 1) * 6 * D + D;      // i + 1 == nh: final layer
        f_qkv.mode = SK_FUSE_TATTN;
        f_qkv.kv_cache = p->kv_cache + static_cast<size_t>(i >> 1) * cache_layer;
        f_qkv.rot = reinterpret_cast<const float2*>(w.rot_temporal);
        f_qkv.ctx_frames = p->T - 1;
        f_qkv.positions = S;
        const bool ta = sh->fuse_tattn && (i & 1);
        if (ta) { pq.out = p->att; pq.ldo = D; }
        // Tagged exchange of the split-K partial sums: every GEMM kind has its own workspace region (zeroed at plan creation)
        // and the 2 * depth launches of a pass alternate the parity on it, 1 first - an even count, so every pass leaves the
        // region at parity 0 and the next pass, or a replay of the captured graph, starts from the same state.
        float* ws4[4];
        for (int k = 0; k < 4; ++k) ws4[k] = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(p->sk_ws) + k * p->sk_ws_bytes);
        const int tag = tag_enabled() ? (2 | ((i & 1) ^ 1)) : 0;
        if (sh->sk[0]) { rc |= skinny_prepare(&sh->s_qkv[i], p->hn, D, static_cast<const bf16*>(hw.qkv_w), D, pq, EPI_STORE, ws4[0], p->sk_counters, 0, ta ? &f_qkv : nullptr); sh->s_qkv[i].tag = tag; }
        else rc |= gemm_prepare(&sh->g_qkv[i], p->hn, D, static_cast<const bf16*>(hw.qkv_w), D, pq, EPI_STORE);
        if (sh->sk[1]) { rc |= skinny_prepare(&sh->s_out[i], p->att, D, static_cast<const bf16*>(hw.out_w), D, po, EPI_BIAS_GATE_RES, ws4[1], p->sk_counters, 0, sh->fuse_ln ? &f_out : nullptr); sh->s_out[i].tag = tag; }
        else rc |= gemm_prepare(&sh->g_out[i], p->att, D, static_cast<const bf16*>(hw.out_w), D, po, EPI_BIAS_GATE_RES);
        if (sh->sk[2]) { rc |= skinny_prepare(&sh->s_fc1[i], p->hn, D, static_cast<const bf16*>(hw.fc1_w), D, p1, EPI_BIAS_GELU_TANH, ws4[2], p->sk_counters); sh->s_fc1[i].tag = tag; }
        else rc |= gemm_prepare(&sh->g_fc1[i], p->hn, D, static_cast<const bf16*>(hw.fc1_w), D, p1, EPI_BIAS_GELU_TANH);
        if (sh->sk[3]) { rc |= skinny_prepare(&sh->s_fc2[i], p->mlp, 4 * D, static_cast<const bf16*>(hw.fc2_w), 4 * D, p2, EPI_BIAS_GATE_RES, ws4[3], p->sk_counters, 0, sh->fuse_ln ? &f_fc2 : nullptr); sh->s_fc2[i].tag = tag; }
        else rc |= gemm_prepare(&sh->g_fc2[i], p->mlp, 4 * D, static_cast<const bf16*>(hw.fc2_w), 4 * D, p2, EPI_BIAS_GATE_RES);
    }
    rc |= gemm_prepare(&sh->g_final, p->hn, D, static_cast<const bf16*>(w.final_w), D, gp(p->yfin, 64, w.final_b, M, h->out_feat, D), EPI_BIAS);
    return rc == 0 ? 0 : (rc < 0 ? rc : -1);
}

// The kernel sequence of DiT.forward's backbone on the rows of `sh`.  x: the [B, T, C, H, W] window; the frames
// processed are first_frame .. first_frame + sh->frames - 1 of every rollout.  out == nullptr skips the final
// layer (context pass: only the K/V caches are wanted).
int run_backbone(gtav_dit_plan_s* p, const Shape* sh, int mode, const void* x, int x_is_bf16, int first_frame,
                 const int* frame_row, void* out, cudaStream_t stream) {
    const gtav_dit_s* e = p->eng;
    const gtav_dit_config& c = e->cfg;
    const int D = c.hidden, M = sh->M, S = e->tokens, W = e->mod_width, F = p->B * sh->frames;
    const long frame_elems = static_cast<long>(c.in_channels) * c.grid_h * c.patch * c.grid_w * c.patch;
    const char* x0 = static_cast<const char*>(x) + first_frame * frame_elems * (x_is_bf16 ? 2 : 4);
    int rc = launch_patchify(x0, x_is_bf16, p->xa, 64, F, c.in_channels, c.grid_h * c.patch, c.grid_w * c.patch, c.patch,
                             sh->frames, static_cast<long>(p->T) * frame_elems, stream);
    if (rc) return rc;
    if ((rc = gemm_run(&sh->g_patch, stream))) return rc;
    const float2* rot_s = reinterpret_cast<const float2*>(e->w.rot_spatial);
    const float2* rot_t = reinterpret_cast<const float2*>(e->w.rot_temporal);
    const size_t cache_layer = static_cast<size_t>(p->B) * (p->T - 1) * S * 2 * D;
    bool hn_ready = false;                  // the previous fc2's reduce already wrote this half's LN1 output
    // GTAV_ENGINE_TRACE=<device address>: phase time stamps of every weight-streaming GEMM of this pass, [launch][160][8]
    // int64 globaltimer ns (scripts/trace_step.py); profiling aid, unset in production
    long long* trace_base = nullptr;
    if (const char* tr = getenv("GTAV_ENGINE_TRACE")) trace_base = reinterpret_cast<long long*>(strtoull(tr, nullptr, 0));
    int trace_k = 0;
    auto run_skinny = [&](const SkinnyOp& op0) {
        SkinnyOp o = op0;
        o.p.frame_row = frame_row;
        if (trace_base != nullptr) o.trace = trace_base + static_cast<size_t>(trace_k++) * 160 * 8;
        return skinny_run(&o, stream);
    };
    for (int i = 0; i < 2 * c.depth; ++i) {
        const int off = i * 6 * D;          // shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp
        if (!hn_ready && (rc = launch_ln_modulate(p->h, p->hn, M, D, p->mod, W, off, off + D, frame_row, S, stream))) return rc;
        if (sh->sk[0]) rc = run_skinny(sh->s_qkv[i]);
        else rc = gemm_run(&sh->g_qkv[i], stream);
        if (rc) return rc;
        if (sh->s_qkv.size() && sh->sk[0] && sh->s_qkv[i].f.mode == SK_FUSE_TATTN) {
            // temporal attention ran inside to_qkv's reduce
        } else if ((i & 1) == 0) {
            rc = launch_attention_seq(p->qkv, p->att, F, S, c.heads, rot_s, 32, stream);
        } else {
            bf16* cache = p->kv_cache + static_cast<size_t>(i >> 1) * cache_layer;
            if (mode == MODE_LAST) rc = launch_attention_temporal_last(p->qkv, p->att, p->B, p->T - 1, S, c.heads, rot_t, cache, stream);
            else rc = launch_attention_temporal(p->qkv, p->att, p->B, sh->frames, S, c.heads, rot_t, mode == MODE_CONTEXT ? cache : nullptr, stream);
        }
        if (rc) return rc;
        if (sh->sk[1]) {
            rc = run_skinny(sh->s_out[i]);
        } else {
            GemmOp o = sh->g_out[i];
            o.p.frame_row = frame_row;
            rc = gemm_run(&o, stream);
        }
        if (rc) return rc;
        if (!sh->fuse_ln && (rc = launch_ln_modulate(p->h, p->hn, M, D, p->mod, W, off + 3 * D, off + 4 * D, frame_row, S, stream))) return rc;
        if (sh->sk[2]) rc = run_skinny(sh->s_fc1[i]);
        else rc = gemm_run(&sh->g_fc1[i], stream);
        if (rc) return rc;
        if (sh->sk[3]) {
            rc = run_skinny(sh->s_fc2[i]);
        } else {
            GemmOp o = sh->g_fc2[i];
            o.p.frame_row = frame_row;
            rc = gemm_run(&o, stream);
        }
        if (rc) return rc;
        hn_ready = sh->fuse_ln;
    }
    if (out == nullptr) return 0;
    const int foff = 2 * c.depth * 6 * D;   // final layer: shift, scale
    if (!hn_ready && (rc = launch_ln_modulate(p->h, p->hn, M, D, p->mod, W, foff, foff + D, frame_row, S, stream))) return rc;
    if ((rc = gemm_run(&sh->g_final, stream))) return rc;
    return launch_dit_unpatchify(p->yfin, static_cast<bf16*>(out), F, c.in_channels, c.grid_h, c.grid_w, c.patch, stream);
}

}  // namespace

extern "C" {

const char* gtav_last_error(void) { return get_error(); }
int gtav_abi_version(void) { return 5; }

int gtav_dit_create(const gtav_dit_config* cfg, const gtav_dit_weights* w, gtav_dit_t* out) {
    if (!cfg || !w || !out) { set_error("dit_create: null argument"); return -1; }
    if (cfg->hidden != 1024 || cfg->heads != 16 || cfg->grid_h * cfg->grid_w != 144 ||
        cfg->in_channels * cfg->patch * cfg->patch != 64 || cfg->depth < 1 || cfg->max_frames < 1 || cfg->max_frames > 32) {
        set_error("dit_create: unsupported geometry (hidden=%d heads=%d grid=%dx%d patch=%d C=%d depth=%d max_frames=%d); "
                  "kernels are built for hidden 1024, 16 heads of 64, 144 tokens, 64 patch features, windows of 1..32 frames",
                  cfg->hidden, cfg->heads, cfg->grid_h, cfg->grid_w, cfg->patch, cfg->in_channels, cfg->depth, cfg->max_frames);
        return -1;
    }
    if (cfg->act_dim < 0 || cfg->act_dim > 64 || (cfg->act_dim > 0 && (!w->act_w || !w->act_b))) {
        set_error("dit_create: bad external_cond configuration (act_dim=%d)", cfg->act_dim);
        return -1;
    }
    gtav_dit_s* e = new (std::nothrow) gtav_dit_s();
    if (!e) { set_error("dit_create: out of host memory"); return -4; }
    e->cfg = *cfg;
    e->w = *w;
    e->halves.assign(w->halves, w->halves + 2 * cfg->depth);
    e->w.halves = e->halves.data();
    e->tokens = cfg->grid_h * cfg->grid_w;
    e->mod_width = cfg->depth * 2 * 6 * cfg->hidden + 2 * cfg->hidden;
    e->patch_k = cfg->in_channels * cfg->patch * cfg->patch;
    e->out_feat = e->patch_k;
    *out = e;
    return 0;
}

void gtav_dit_destroy(gtav_dit_t h) { delete h; }
int gtav_dit_mod_width(gtav_dit_t h) { return h ? h->mod_width : 0; }

size_t gtav_dit_workspace_bytes(gtav_dit_t h, int B, int T, int cond_rows) {
    if (!h || B <= 0 || T <= 0 || cond_rows <= 0) return 0;
    gtav_dit_plan_s tmp{};
    tmp.eng = h; tmp.B = B; tmp.T = T; tmp.M = B * T * h->tokens; tmp.R = cond_rows;
    size_t total = 0;
    carve(&tmp, nullptr, &total);
    return total;
}

int gtav_dit_plan_create(gtav_dit_t h, int B, int T, int cond_rows, void* workspace, size_t workspace_bytes,
                         gtav_stream_t stream, gtav_dit_plan_t* out) {
    if (!h || !workspace || !out) { set_error("dit_plan_create: null argument"); return -1; }
    if (B <= 0 || T <= 0 || T > h->cfg.max_frames || cond_rows <= 0) {
        set_error("dit_plan_create: B=%d T=%d cond_rows=%d out of range (T <= max_frames=%d)", B, T, cond_rows, h->cfg.max_frames);
        return -1;
    }
    if (reinterpret_cast<uintptr_t>(workspace) & 1023) { set_error("dit_plan_create: workspace must be 1024-byte aligned"); return -1; }
    gtav_dit_plan_s* p = new (std::nothrow) gtav_dit_plan_s();
    if (!p) { set_error("dit_plan_create: out of host memory"); return -4; }
    p->eng = h; p->B = B; p->T = T; p->M = B * T * h->tokens; p->R = cond_rows;
    size_t need = 0;
    carve(p, workspace, &need);
    if (need > workspace_bytes) {
        set_error("dit_plan_create: workspace too small (%zu < %zu)", workspace_bytes, need);
        delete p;
        return -1;
    }
    const int D = h->cfg.hidden, R = p->R, W = h->mod_width;
    const gtav_dit_weights& w = h->w;
    int rc = 0;
    // conditioning chain (rows = R)
    rc |= gemm_prepare(&p->g_t0, p->temb, 256, static_cast<const bf16*>(w.t0_w), 256, gp(p->h1, D, w.t0_b, R, D, 256), EPI_BIAS_SILU);
    {
        GemmParams q = gp(p->cact, D, w.t2_b, R, D, D);
        if (h->cfg.act_dim > 0) { q.res = p->aemb; q.ldr = D; }
        rc |= gemm_prepare(&p->g_t2, p->h1, D, static_cast<const bf16*>(w.t2_w), D, q, EPI_BIAS_RES_SILU);
    }
    rc |= gemm_prepare(&p->g_ada, p->cact, D, static_cast<const bf16*>(w.ada_w), D, gp(p->mod, W, w.ada_b, R, W, D), EPI_BIAS);
    // backbone: one set of descriptors per row count
    if (rc == 0) rc = build_shape(p, &p->full, T, false);
    if (rc == 0 && T >= 2) rc = build_shape(p, &p->ctx, T - 1, false);
    if (rc == 0) rc = build_shape(p, &p->last, 1, true);
    // on the caller's stream: the workspace may be a recycled block of a stream-ordered allocator (torch's), and the
    // plan's kernels run on that stream too - a memset on the legacy stream would order with neither
    if (rc == 0 && cudaMemsetAsync(p->sk_counters, 0, 2048, stream) != cudaSuccess) { set_error("dit_plan_create: clearing the split-K counters failed"); rc = -2; }
    if (rc == 0 && p->sk_ws_bytes > 0 && cudaMemsetAsync(p->sk_ws, 0, 4 * p->sk_ws_bytes, stream) != cudaSuccess) { set_error("dit_plan_create: clearing the split-K workspace failed"); rc = -2; }
    if (rc) { delete p; return rc < 0 ? rc : -1; }
    *out = p;
    return 0;
}

void gtav_dit_plan_destroy(gtav_dit_plan_t p) { delete p; }

int gtav_dit_conditioning(gtav_dit_plan_t p, const int64_t* t, const float* actions, gtav_stream_t stream) {
    if (!p || !t) { set_error("dit_conditioning: null argument"); return -1; }
    const gtav_dit_s* e = p->eng;
    const bool use_act = e->cfg.act_dim > 0 && actions != nullptr;
    int rc = launch_cond_prep(t, use_act ? actions : nullptr, e->cfg.act_dim, p->R, e->w.temb_freqs,
                              static_cast<const bf16*>(e->w.act_w), static_cast<const bf16*>(e->w.act_b), p->temb,
                              p->aemb, e->cfg.hidden, stream);
    if (rc) return rc;
    if ((rc = gemm_run(&p->g_t0, stream))) return rc;
    // `c += external_cond(a)` only when an action tensor is passed (dit.py:363): toggle the residual
    GemmOp t2 = p->g_t2;
    if (!use_act) t2.p.res = nullptr;
    if ((rc = gemm_run(&t2, stream))) return rc;
    return gemm_run(&p->g_ada, stream);
}

int gtav_dit_backbone(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, void* out,
                      gtav_stream_t stream) {
    if (!p || !x || !out) { set_error("dit_backbone: null argument"); return -1; }
    return run_backbone(p, &p->full, MODE_FULL, x, x_is_bf16, 0, frame_row, out, stream);
}

int gtav_dit_context(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, gtav_stream_t stream) {
    if (!p || !x) { set_error("dit_context: null argument"); return -1; }
    if (p->T < 2) return 0;                  // a one-frame window has no context
    return run_backbone(p, &p->ctx, MODE_CONTEXT, x, x_is_bf16, 0, frame_row, nullptr, stream);
}

int gtav_dit_last_frame(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int* frame_row, void* out,
                        gtav_stream_t stream) {
    if (!p || !x || !out) { set_error("dit_last_frame: null argument"); return -1; }
    if (p->sk_out_of_step) {
        set_error("dit_last_frame: an earlier last-frame pass on this plan failed part-way, which leaves the split-K exchange's "
                  "parities out of step; create a new plan");
        return -3;
    }
    const int rc = run_backbone(p, &p->last, MODE_LAST, x, x_is_bf16, p->T - 1, frame_row, out, stream);
    if (rc != 0 && tag_enabled()) p->sk_out_of_step = true;      // (get_error() still holds the failing launch's message)
    return rc;
}

int gtav_dit_forward(gtav_dit_plan_t p, const void* x, int x_is_bf16, const int64_t* t, const float* actions,
                     void* out, gtav_stream_t stream) {
    if (!p) { set_error("dit_forward: null plan"); return -1; }
    if (p->R != p->B * p->T) {
        set_error("dit_forward: plan was created with cond_rows=%d, need B*T=%d", p->R, p->B * p->T);
        return -1;
    }
    int rc = gtav_dit_conditioning(p, t, actions, stream);
    if (rc) return rc;
    return gtav_dit_backbone(p, x, x_is_bf16, nullptr, out, stream);
}

// ---------------------------------------------------------------------------- stand-alone kernels
int gtav_gemm_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                   int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                   const int* frame_row, int rows_per_frame, int bn, gtav_stream_t stream) {
    GemmParams p{};
    p.out = static_cast<bf16*>(out); p.ldo = ldo; p.bias = static_cast<const bf16*>(bias);
    p.res = static_cast<const bf16*>(res); p.ldr = ldr; p.gate = static_cast<const bf16*>(gate); p.gate_ld = gate_ld;
    p.frame_row = frame_row; p.rows_per_frame = rows_per_frame > 0 ? rows_per_frame : 1;
    p.M = M; p.N = N; p.K = K;
    GemmOp op;
    int rc = gemm_prepare(&op, static_cast<const bf16*>(A), lda, static_cast<const bf16*>(W), ldw, p, epilogue, bn);
    if (rc) return rc;
    return gemm_run(&op, stream);
}

size_t gtav_gemm_skinny_workspace_bytes(int M) { return skinny_workspace_bytes(M); }

namespace {
int skinny_standalone(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K, int epilogue,
                      const void* bias, const void* res, int ldr, const void* gate, int gate_ld, const int* frame_row,
                      int rows_per_frame, int splits, void* workspace, int* counters, int tag, gtav_stream_t stream,
                      const SkinnyFuseParams* fuse = nullptr) {
    GemmParams p{};
    p.out = static_cast<bf16*>(out); p.ldo = ldo; p.bias = static_cast<const bf16*>(bias);
    p.res = static_cast<const bf16*>(res); p.ldr = ldr; p.gate = static_cast<const bf16*>(gate); p.gate_ld = gate_ld;
    p.frame_row = frame_row; p.rows_per_frame = rows_per_frame > 0 ? rows_per_frame : 1;
    p.M = M; p.N = N; p.K = K;
    SkinnyOp op;
    int rc = skinny_prepare(&op, static_cast<const bf16*>(A), lda, static_cast<const bf16*>(W), ldw, p, epilogue,
                            static_cast<float*>(workspace), counters, splits, fuse);
    if (rc) return rc;
    op.tag = tag;
    if (const char* t = getenv("GTAV_SKINNY_TRACE")) op.trace = reinterpret_cast<long long*>(strtoull(t, nullptr, 0));
    return skinny_run(&op, stream);
}
}  // namespace

int gtav_gemm_skinny_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                          int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                          const int* frame_row, int rows_per_frame, int splits, void* workspace, int* counters,
                          gtav_stream_t stream) {
    if (!workspace || !counters) { set_error("gemm_skinny: workspace and counters are required"); return -1; }
    return skinny_standalone(A, lda, W, ldw, out, ldo, M, N, K, epilogue, bias, res, ldr, gate, gate_ld, frame_row, rows_per_frame,
                             splits, workspace, counters, 0, stream);
}

int gtav_gemm_skinny_tagged_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                                 int epilogue, const void* bias, const void* res, int ldr, const void* gate, int gate_ld,
                                 const int* frame_row, int rows_per_frame, int splits, void* workspace, int parity,
                                 gtav_stream_t stream) {
    if (!workspace) { set_error("gemm_skinny_tagged: workspace is required"); return -1; }
    if (parity != 0 && parity != 1) { set_error("gemm_skinny_tagged: parity must be 0 or 1, got %d", parity); return -1; }
    return skinny_standalone(A, lda, W, ldw, out, ldo, M, N, K, epilogue, bias, res, ldr, gate, gate_ld, frame_row, rows_per_frame,
                             splits, workspace, nullptr, 2 | parity, stream);
}

int gtav_gemm_skinny_fused_bf16(const void* A, int lda, const void* W, int ldw, void* out, int ldo, int M, int N, int K,
                                const void* bias, const void* res, int ldr, const void* gate, int gate_ld, const int* frame_row,
                                int splits, void* workspace, int* counters, int mode, void* ln_out, const void* ln_mod,
                                int ln_mod_ld, int ln_shift_off, int ln_scale_off, const void* kv_cache, const float* rot,
                                int ctx_frames, int positions, int parity, gtav_stream_t stream) {
    if (!workspace) { set_error("gemm_skinny_fused: workspace is required"); return -1; }
    if (parity < -1 || parity > 1) { set_error("gemm_skinny_fused: parity must be -1, 0 or 1, got %d", parity); return -1; }
    if (parity == -1 && !counters) { set_error("gemm_skinny_fused: counters are required with parity -1"); return -1; }
    if (mode != SK_FUSE_LN && mode != SK_FUSE_TATTN) { set_error("gemm_skinny_fused: mode must be 1 or 2, got %d", mode); return -1; }
    SkinnyFuseParams f{};
    f.mode = mode;
    f.ln_out = static_cast<bf16*>(ln_out);
    f.ln_mod = static_cast<const bf16*>(ln_mod);
    f.ln_mod_ld = ln_mod_ld; f.ln_shift_off = ln_shift_off; f.ln_scale_off = ln_scale_off;
    f.kv_cache = static_cast<const bf16*>(kv_cache);
    f.rot = reinterpret_cast<const float2*>(rot);
    f.ctx_frames = ctx_frames; f.positions = positions;
    // the mode fixes the epilogue (skinny_prepare checks every other argument against it)
    const int epi = mode == SK_FUSE_LN ? EPI_BIAS_GATE_RES : EPI_STORE;
    return skinny_standalone(A, lda, W, ldw, out, ldo, M, N, K, epi, bias, res, ldr, gate, gate_ld, frame_row, 144, splits,
                             workspace, parity == -1 ? counters : nullptr, parity == -1 ? 0 : 2 | parity, stream, &f);
}

int gtav_ln_modulate(const void* x, void* out, int M, int D, const void* mod, int mod_ld, int shift_off, int scale_off,
                     const int* frame_row, int rows_per_frame, gtav_stream_t stream) {
    return launch_ln_modulate(static_cast<const bf16*>(x), static_cast<bf16*>(out), M, D, static_cast<const bf16*>(mod),
                              mod_ld, shift_off, scale_off, frame_row, rows_per_frame, stream);
}
int gtav_ln_affine(const void* x, void* out, int M, int D, const float* w, const float* b, gtav_stream_t stream) {
    return launch_ln_affine(static_cast<const bf16*>(x), static_cast<bf16*>(out), M, D, w, b, stream);
}
int gtav_attention_seq(const void* qkv, void* out, int groups, int seq, int heads, const float* rot, int rot_pairs,
                       gtav_stream_t stream) {
    return launch_attention_seq(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), groups, seq, heads,
                                reinterpret_cast<const float2*>(rot), rot_pairs, stream);
}
int gtav_attention_temporal(const void* qkv, void* out, int B, int T, int positions, int heads, const float* rot,
                            gtav_stream_t stream) {
    return launch_attention_temporal(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), B, T, positions, heads,
                                     reinterpret_cast<const float2*>(rot), nullptr, stream);
}
int gtav_attention_temporal_last(const void* qkv, void* out, int B, int ctx_frames, int positions, int heads,
                                 const float* rot, const void* kv_cache, gtav_stream_t stream) {
    return launch_attention_temporal_last(static_cast<const bf16*>(qkv), static_cast<bf16*>(out), B, ctx_frames, positions,
                                          heads, reinterpret_cast<const float2*>(rot), static_cast<const bf16*>(kv_cache), stream);
}
int gtav_ddim_update(const float* x, const void* v_bf16, float* out, int F, int n, const float* abar_t,
                     const float* abar_next, const int* final_flag, gtav_stream_t stream) {
    return launch_ddim(x, n, static_cast<const bf16*>(v_bf16), n, out, n, F, n, abar_t, abar_next, final_flag, stream);
}

}  // extern "C"
