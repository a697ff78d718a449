"""Sliding windows of 9..32 frames on the GPU: the long-window temporal attention kernels (csrc/attn_temporal_long.cu)
against float64 and against each other, and the DiT, Sampler and FrameStream at windows longer than 8 frames.

Kernel references are float64 from the same bf16 inputs with the kernels' rounding points written out (the rotated q / k
and the softmax probabilities), as in test_last_frame_kernels_gpu.py, whose input and cache helpers are reused here."""
import math

import pytest
import torch

from oracle import reference_port as rp
from oracle.cases import seeded_randn
from oracle.weights import DiTConfig, dummy_prompt, make_dit_state, make_vae_state, VAEConfig, w_key_actions
from parity64 import assert_within, r16, round_diff
from test_last_frame_kernels_gpu import D, H, P, attention_last, dense_attention, kv_cache_of, rot_table, rotate_rn, \
    temporal_inputs, to_rows

pytestmark = pytest.mark.gpu

TOL_FP32 = (6e-2, 1.2e-2)       # test_model_gpu.py: DiT forward vs the fp32 reference (max-abs, mean-abs)
TOL_BF16 = (4e-2, 4e-3)         # ... vs the bf16-rounding oracle


@pytest.fixture(scope="module")
def lib():
    import gtav_b200._native as N
    return N.load()


def _N():
    import gtav_b200._native as N
    return N


def temporal_ref_long(q, k, v, rot):
    """float64 causal attention over the T <= 32 frames of q, k, v [B, T, P, H, 64] (bf16 values), and a bound for every
    frame's output, [B, T, P, H, 64].
    Scores: an fp32 dot product of 64 terms per lane pair (a product and an fma) reduced by 5 shuffle additions, so within
    2^-21 sum|q k| / 8 = es, whatever the window length.
    Probabilities before rounding: s - max uses two scores (2 es); __expf adds 2^-21 relative plus |s - max| 2^-24, and
    |s - max| <= 60 for the inputs here (2^-18).  The fp32 sum of at most 32 exponentials is off by at most 31 * 2^-24 < 2^-19
    relative, and the correctly rounded reciprocal and product add 2^-23.  All of these but the scores' share stay below
    2^-15, so the relative error is at most eps = 4 max(es) + 2^-15 and the bf16 p is off by at most round_diff(p_ref, eps p).
    Output: an fp32 fma chain of at most 32 terms, each rounding off by 2^-24 of the running sum, so 32 * 2^-24 = 2^-19
    sum p|v|, plus the p errors times |v|, then the final bf16 rounding."""
    T = q.shape[1]
    qr, kr = rotate_rn(q, rot), rotate_rn(k, rot)
    qr, kr, vv = (z.double().permute(0, 2, 3, 1, 4) for z in (qr, kr, v))            # [B, P, H, T, 64]
    causal = torch.ones(T, T, dtype=torch.bool, device=q.device).triu(1)
    s = (qr @ kr.transpose(-1, -2) / 8).masked_fill(causal, -math.inf)
    es = (2.0 ** -21 * (qr.abs() @ kr.abs().transpose(-1, -2)) / 8).masked_fill(causal, 0.0)
    e = torch.exp(s - s.amax(-1, keepdim=True))
    pex = e / e.sum(-1, keepdim=True)
    p = r16(pex)
    eps = 4 * es.amax(-1, keepdim=True) + 2.0 ** -15
    dp = round_diff(p, eps * pex).masked_fill(causal, 0.0)
    va = vv.abs()
    ref = r16(p @ vv)
    tol = round_diff(ref, dp @ va + 2.0 ** -19 * (p @ va))
    return ref.permute(0, 3, 1, 2, 4), tol.permute(0, 3, 1, 2, 4)


# ------------------------------------------------------------------------------------------ kernels
LONG_WINDOWS = [(T, B, "random") for T in (9, 12, 16, 24, 32) for B in (1, 3)] + \
               [(32, 1, "far"), (32, 1, "uniform"), (24, 1, "pairs")]


@pytest.mark.parametrize("T,B,kind", LONG_WINDOWS)
def test_dense_long_window_float64(lib, T, B, kind):
    """gtav_attention_temporal at 9..32 frames against float64 with the kernel's rounding points."""
    rot = rot_table(32)
    q, k, v = temporal_inputs(B, T, kind, 900 + 10 * T + B)
    _, out = dense_attention(lib, q, k, v, rot)
    ref, tol = temporal_ref_long(q, k, v, rot)
    assert_within(out, to_rows(ref), to_rows(tol), f"dense temporal attention T={T} B={B} {kind}")


@pytest.mark.parametrize("B", (1, 3))
@pytest.mark.parametrize("ctx", range(8, 32))
def test_last_frame_long_equals_dense(lib, ctx, B):
    """gtav_attention_temporal_last with 8..31 cached frames against the cache the context pass writes: the same bits as
    row ctx of the dense kernel over ctx + 1 frames."""
    T = ctx + 1
    rot = rot_table(32)
    q, k, v = temporal_inputs(B, T, "random", 1100 + 10 * T + B)
    qkv, dense = dense_attention(lib, q, k, v, rot)
    last_qkv = qkv.view(B, T, P, 3 * D)[:, T - 1].reshape(B * P, 3 * D).contiguous()
    out = attention_last(lib, last_qkv, ctx, rot, kv_cache_of(k[:, :ctx], v[:, :ctx], rot))
    ref = dense.view(B, T, P, D)[:, T - 1].reshape(B * P, D)
    assert torch.equal(out, ref), f"last-frame kernel differs from the dense kernel's last row: max-abs {float((out.float() - ref.float()).abs().max())}"


def plan_buffers(model, B, T):
    """The q|k|v rows and the K/V cache inside the workspace of model's (B, T) plan (dit_engine.cu carve(): slices in this
    order, each rounded up to 1024 bytes)."""
    plan, ws = model._plans[(B, T, B * T)]
    base = (ws.data_ptr() + 1023) & ~1023
    M, R = B * T * P, B * T
    W = model.depth * 2 * 6 * D + 2 * D
    elems = [M * 64, M * D, M * D, M * 3 * D, M * D, M * 4 * D, M * 64, R * 256, R * D, R * D, R * D, R * W]
    off = [0]
    for n in elems:
        off.append(off[-1] + ((2 * n + 1023) & ~1023))
    flat = ws[base - ws.data_ptr():].view(torch.bfloat16)
    qkv = flat[off[3] // 2: off[3] // 2 + M * 3 * D].view(M, 3 * D)
    cache_layer = B * (T - 1) * P * 2 * D
    cache = flat[off[12] // 2: off[12] // 2 + model.depth * cache_layer].view(model.depth, B * (T - 1) * P, 2 * D)
    return qkv, cache


def model_rot(model):
    """The temporal (cos, sin) table DiT._pack hands the engine, built by the same torch expressions on the same device."""
    tf = model.temporal_rotary_emb.freqs.detach().to(device="cuda", dtype=torch.float32)
    pos = torch.arange(model.max_frames, device="cuda", dtype=torch.bfloat16).to(torch.float32)
    ang = pos[:, None] * tf[None]
    return torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()


@pytest.mark.parametrize("B,T", [(1, 16), (2, 12), (1, 32)])
def test_context_pass_writes_the_cache_of_its_qkv(B, T):
    """The dense kernel with a cache pointer, as the context pass runs it over T - 1 >= 9 frames: the K/V cache of the last
    temporal layer equals kv_cache_of the q|k|v rows that layer attended over (still in the plan's qkv buffer after the
    pass), bit for bit."""
    from gtav_b200.model.dit import DiT
    N = _N()
    lib = N.load()
    model = DiT(depth=2, max_frames=T)
    model.load_state_dict(make_dit_state(DiTConfig(depth=2), seed=0), strict=True)
    model = model.cuda().eval()
    x = seeded_randn((B, T, 16, 18, 32), 1300 + T).cuda()
    t = torch.randint(0, 1000, (B, T), generator=torch.Generator().manual_seed(T)).cuda().reshape(-1)
    model.forward_last_frame(x, t.view(B, T))                 # packs and creates the plan
    ctx_rows = torch.arange(B * T, dtype=torch.int32, device="cuda").reshape(B, T)[:, :-1].contiguous()
    plan = model._plan(B, T)
    s = N.current_stream()
    N.check(lib.gtav_dit_conditioning(plan, t.data_ptr(), None, s), "conditioning")
    N.check(lib.gtav_dit_context(plan, x.data_ptr(), 0, ctx_rows.data_ptr(), s), "context")
    torch.cuda.synchronize()
    qkv, cache = plan_buffers(model, B, T)
    F = B * (T - 1) * P
    rows = qkv[:F].float().view(B, T - 1, P, 3, H, 64)
    k, v = rows[:, :, :, 1], rows[:, :, :, 2]
    ref = kv_cache_of(k, v, model_rot(model))
    assert torch.isfinite(ref.float()).all()
    assert torch.equal(cache[model.depth - 1], ref), "K/V cache differs from the rotated K | V of the q|k|v rows"


# ------------------------------------------------------------------------------------------ DiT
def dit(max_frames, depth=2, seed=0):
    from gtav_b200.model.dit import DiT
    m = DiT(depth=depth, max_frames=max_frames)
    m.load_state_dict(make_dit_state(DiTConfig(depth=depth), seed=seed), strict=True)
    return m.cuda().eval()


def check(out, ref, tol, what):
    err = (out.float().cpu() - ref).abs()
    mx, mean = float(err.max()), float(err.mean())
    print(f"{what}: max-abs {mx:.4f} mean-abs {mean:.5f} (ref std {float(ref.std()):.3f})")
    assert mx <= tol[0] and mean <= tol[1], (what, mx, mean)


def test_dit_forward_16_frames_vs_oracle():
    """DiT.forward over a 16-frame window (depth 2, non-degenerate weights) against the reference port in fp32 and in
    bf16-rounding mode, with the bounds test_model_gpu.py applies at 5 frames."""
    sd = make_dit_state(DiTConfig(depth=2), seed=0)
    model = dit(16)
    x = seeded_randn((1, 16, 16, 18, 32), 1401)
    t = torch.tensor([[15] * 15 + [749]])
    a = w_key_actions(1, 16)
    v = model(x.cuda(), t.cuda(), a.cuda())
    assert v.dtype == torch.bfloat16 and v.shape == x.shape
    cfg = DiTConfig(depth=2, max_frames=16)
    check(v, rp.dit_forward(sd, cfg, x, t, a, rp.FP32), TOL_FP32, "T=16 vs fp32 oracle")
    check(v, rp.dit_forward(sd, cfg, x, t, a, rp.BF16), TOL_BF16, "T=16 vs bf16-rounding oracle")


@pytest.mark.parametrize("mode", ["tiled", "default"])
def test_dit_last_frame_long_window_equals_dense(monkeypatch, mode):
    """Context pass + last-frame pass over windows of 9, 16 and 32 frames == the last frame of the dense forward: bit for
    bit with the tiled GEMMs everywhere, within test_dit_last_frame_split_equals_dense's 2e-2 on the default path (the
    weight-streaming GEMM sums its K splits in another order)."""
    if mode == "tiled":
        monkeypatch.setenv("GTAV_SKINNY", "0")
        monkeypatch.setenv("GTAV_GEMM_SPLITK", "0")
    model = dit(32)
    for B, T, seed, actions in ((1, 16, 1501, True), (2, 9, 1502, False), (1, 32, 1503, True), (3, 12, 1504, True)):
        x = seeded_randn((B, T, 16, 18, 32), seed).cuda()
        t = torch.randint(0, 1000, (B, T), generator=torch.Generator().manual_seed(seed)).cuda()
        a = w_key_actions(B, T).cuda() if actions else None
        dense = model(x, t, a)[:, -1:]
        split = model.forward_last_frame(x, t, a)
        err = float((dense.float() - split.float()).abs().max())
        print(f"{mode} B={B} T={T}: last-frame split vs dense max-abs {err:.5f} equal={torch.equal(dense, split)}")
        assert torch.isfinite(split.float()).all()
        if mode == "tiled":
            assert torch.equal(dense, split), err
        else:
            assert err <= 2e-2, err
        assert torch.equal(split, model.forward_last_frame(x, t, a)), "last-frame pass is not deterministic"


# ------------------------------------------------------------------------------------------ Sampler / FrameStream
@pytest.fixture(scope="module")
def vae():
    from gtav_b200.model.vae import AutoencoderKL
    m = AutoencoderKL(latent_dim=16, patch_size=20, enc_dim=1024, enc_depth=1, enc_heads=16, dec_dim=1024, dec_depth=1,
                      dec_heads=16, input_height=360, input_width=640)
    m.load_state_dict(make_vae_state(VAEConfig(enc_depth=1, dec_depth=1), seed=0), strict=True)
    return m.cuda().eval()


def test_sampler_12_frames_equals_stepwise_dropin_loop():
    """max_frames = 12, frame cache off: graph == no graph, and both == the reference-shaped loop over denoise_step, bit
    for bit, while the window grows from 3 to 12 frames and then slides."""
    from gtav_b200.sampler import Sampler
    from gtav_b200.train_dit import denoise_step
    model = dit(12)
    steps, total, n_prompt = 2, 15, 2
    prompt = torch.randn((2, n_prompt, 16, 18, 32), generator=torch.Generator().manual_seed(1601)).cuda()
    noise = torch.randn((2, total - n_prompt, 16, 18, 32), generator=torch.Generator().manual_seed(1602)).cuda()
    acts = torch.zeros(2, total, 25, device="cuda")
    acts[0, :, 3] = 1.0
    acts[1, :, 7] = 1.0
    acts[1, 9:, 2] = 1.0
    outs = []
    for use_graph in (True, False):
        s = Sampler(model, None, noise_steps=steps, use_graph=use_graph, frame_cache=False)
        outs.append(s.sample_latents(prompt, acts, total, noise=noise))
        s.close()
    assert torch.equal(outs[0], outs[1])
    abar = rp.alphas_cumprod_table().cuda().reshape(-1, 1, 1, 1)
    noise_range = torch.linspace(0, 999, steps + 1)
    x = prompt.float()
    for i in range(n_prompt, total):
        x = torch.cat([x, noise[:, i - n_prompt: i - n_prompt + 1].clamp(-20, 20)], dim=1)
        start = max(0, i + 1 - model.max_frames)
        for k in reversed(range(steps + 1)):
            xp, _ = denoise_step(dit_model=model, x_noisy=x, actions=acts, noise_idx=k, stabilization_level=15,
                                 noise_range=noise_range, alphas_cumprod=abar, start_frame=start)
            x[:, -1:] = xp[:, -1:]
    assert torch.equal(outs[0], x), float((outs[0] - x).abs().max())


def test_sampler_12_frames_frame_cache_equals_dense():
    """max_frames = 12: context pass + last-frame steps against dense sampling, within the bounds of
    test_frame_cache_equals_dense_sampling."""
    from gtav_b200.sampler import Sampler
    model = dit(12)
    steps, total, n_prompt = 3, 15, 2
    prompt = torch.randn((2, n_prompt, 16, 18, 32), generator=torch.Generator().manual_seed(1701)).cuda()
    noise = torch.randn((2, total - n_prompt, 16, 18, 32), generator=torch.Generator().manual_seed(1702)).cuda()
    acts = torch.zeros(2, total, 25, device="cuda")
    acts[:, :, 3] = 1.0
    acts[1, 6:, 9] = 1.0
    res = {}
    for name, kw in (("dense", dict(frame_cache=False)), ("cache", dict(frame_cache=True)),
                     ("cache_nograph", dict(frame_cache=True, use_graph=False))):
        s = Sampler(model, None, noise_steps=steps, **kw)
        res[name] = s.sample_latents(prompt, acts, total, noise=noise)
        s.close()
    assert torch.equal(res["cache"], res["cache_nograph"])
    err = (res["cache"] - res["dense"]).abs()
    print(f"max_frames 12, frame cache vs dense sampling: max-abs {float(err.max()):.5f} mean-abs {float(err.mean()):.6f}")
    assert float(err.max()) < 3e-2 and float(err.mean()) < 2e-3


def test_sampler_12_frames_growing_window_vs_oracle():
    """One prompt frame, max_frames = 12: the window grows 2, 3, ..., 11 frames, past the 8 of the short-window kernels,
    against the bf16-rounding oracle's rollout with DiTConfig(max_frames=12), within the bounds of
    test_sampler_without_actions_and_growing_window."""
    from gtav_b200.sampler import Sampler
    model = dit(12)
    total = 11
    s = Sampler(model, None, noise_steps=2)
    prompt = torch.randn((1, 1, 16, 18, 32), generator=torch.Generator().manual_seed(1801)).cuda()
    noise = torch.randn((1, total - 1, 16, 18, 32), generator=torch.Generator().manual_seed(1802))
    x = s.sample_latents(prompt, None, total, noise=noise.cuda())
    cfg = DiTConfig(depth=2, max_frames=12)
    it = iter(range(total - 1))
    ref = rp.rollout(make_dit_state(DiTConfig(depth=2), seed=0), cfg, prompt.cpu(), None, total, 2,
                     lambda i: noise[:, next(it)][:, None], rd=rp.BF16)
    err = (x.cpu() - ref).abs()
    print(f"max_frames 12, growing window vs bf16 oracle: max-abs {float(err.max()):.4f} mean-abs {float(err.mean()):.5f}")
    assert float(err.max()) < 1e-1 and float(err.mean()) < 1e-2


def test_frame_stream_16_frames_equals_batch_generate(vae):
    """max_frames = 16: FrameStream keeps the last 15 latents and slides; its latents equal Sampler.generate's bit for bit."""
    from gtav_b200.sampler import Sampler
    model = dit(16)
    steps, total, n_prompt, B = 1, 19, 2, 1
    video = dummy_prompt(5)[None, :n_prompt].expand(B, -1, -1, -1, -1).contiguous().cuda()
    noise = torch.randn((B, total - n_prompt, 16, 18, 32), generator=torch.Generator().manual_seed(1901)).cuda()
    acts = torch.zeros(B, total, 25, device="cuda")
    acts[:, :, 3] = 1.0
    acts[:, 10:, 9] = 1.0
    s = Sampler(model, vae, noise_steps=steps)
    _, lat = s.generate(video, acts, total, noise=noise)
    st = s.stream(video, prompt_actions=acts[:, :n_prompt])
    for i in range(n_prompt, total):
        _, z = st.next(action=acts[:, i], noise=noise[:, i - n_prompt], decode=False)
        assert torch.equal(z, lat[:, i]), f"frame {i}: streamed latent differs from the batch rollout"
    assert st.window.shape[1] == 15


def test_changing_max_frames_after_a_forward():
    """max_frames set from 5 to 16 on a module that has already run: the next call re-packs (engine, temporal rotary table,
    plans).  A 16-frame forward then equals a freshly built max_frames = 16 module's, and a Sampler created before the
    change gives the new module's results, bit for bit."""
    from gtav_b200.sampler import Sampler
    model = dit(5)
    x5 = seeded_randn((1, 5, 16, 18, 32), 2001).cuda()
    t5 = torch.tensor([[15, 15, 15, 15, 500]]).cuda()
    model(x5, t5)
    prompt = seeded_randn((1, 2, 16, 18, 32), 2002).cuda()
    noise = seeded_randn((1, 12, 16, 18, 32), 2003).cuda()
    s = Sampler(model, None, noise_steps=1)
    before = s.sample_latents(prompt, None, 14, noise=noise)
    with pytest.raises(RuntimeError, match="max_frames"):
        model(seeded_randn((1, 16, 16, 18, 32), 2004).cuda(), torch.full((1, 16), 15).cuda())
    model.max_frames = 16
    fresh = dit(16)
    x = seeded_randn((1, 16, 16, 18, 32), 2004).cuda()
    t = torch.tensor([[15] * 15 + [300]]).cuda()
    assert torch.equal(model(x, t), fresh(x, t))
    after = s.sample_latents(prompt, None, 14, noise=noise)
    ref = Sampler(fresh, None, noise_steps=1).sample_latents(prompt, None, 14, noise=noise)
    assert torch.equal(after, ref)
    assert not torch.equal(after, before), "the sampler kept the 5-frame window"
    assert torch.equal(model(x5, t5), fresh(x5, t5))
