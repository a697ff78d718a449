"""Ragged windows on the GPU: the ragged temporal attention kernels against the existing kernels run on each rollout alone,
a DiT plan with per-rollout window lengths against each rollout's own window, and StreamPool sessions against B = 1
FrameStreams.  Every "equal" below is torch.equal."""
import pytest
import torch

from oracle.cases import seeded_randn
from oracle.weights import DiTConfig, VAEConfig, dummy_prompt, make_dit_state, make_vae_state
from test_last_frame_kernels_gpu import D, H, P, attention_last, dense_attention, kv_cache_of, rot_table, temporal_inputs, \
    to_rows

pytestmark = pytest.mark.gpu


def _N():
    import gtav_b200._native as N
    return N


@pytest.fixture(scope="module")
def lib():
    return _N().load()


def ragged_dense(lib, q, k, v, rot, valid):
    N = _N()
    B, T = q.shape[:2]
    qkv = torch.cat([to_rows(z) for z in (q, k, v)], dim=1).to(torch.bfloat16).contiguous()
    out = torch.full((B * T * P, D), float("nan"), dtype=torch.bfloat16, device="cuda")
    cache = torch.full((B * T * P, 2 * D), float("nan"), dtype=torch.bfloat16, device="cuda")
    lens = torch.tensor(valid, dtype=torch.int32, device="cuda")
    N.check(lib.gtav_attention_temporal_ragged(qkv.data_ptr(), out.data_ptr(), B, T, P, H, rot.data_ptr(), lens.data_ptr(),
                                               cache.data_ptr(), N.current_stream()), "ragged dense")
    return qkv, out.view(B, T, P, D), cache.view(B, T, P, 2 * D)


def ragged_last(lib, qkv, ctx, rot, valid, cache):
    N = _N()
    out = torch.full((qkv.shape[0], D), float("nan"), dtype=torch.bfloat16, device="cuda")
    lens = torch.tensor(valid, dtype=torch.int32, device="cuda")
    N.check(lib.gtav_attention_temporal_last_ragged(qkv.data_ptr(), out.data_ptr(), qkv.shape[0] // P, ctx, P, H, rot.data_ptr(),
                                                    lens.data_ptr(), N.ptr(cache), N.current_stream()), "ragged last")
    return out


# ------------------------------------------------------------------------------------------ kernels
DENSE = [(2, [2, 1, 0]), (5, [5, 1, 3, 2]), (8, [1, 8, 4, 7, 0]), (9, [9, 1, 8, 5]), (16, [16, 1, 9, 8, 3]),
         (32, [1, 32, 17, 31, 9])]


@pytest.mark.parametrize("T,valid", DENSE)
def test_ragged_dense_equals_each_rollout_alone(lib, T, valid):
    """Each rollout's valid rows and cache rows equal gtav_attention_temporal (and the cache the context pass writes) run on
    its valid frames alone; padded rows and padded cache rows are 0; with every length T the output is the existing
    kernel's."""
    B = len(valid)
    rot = rot_table(32)
    q, k, v = temporal_inputs(B, T, "random", 3000 + 10 * T + B)
    _, out, cache = ragged_dense(lib, q, k, v, rot, valid)
    for b, L in enumerate(valid):
        pad = T - L
        assert not out[b, :pad].any() and not cache[b, :pad].any(), f"T={T} rollout {b}: padded rows are not 0"
        if L == 0:
            continue
        _, solo = dense_attention(lib, q[b:b + 1, pad:], k[b:b + 1, pad:], v[b:b + 1, pad:], rot)
        assert torch.equal(out[b, pad:].reshape(-1, D), solo), f"T={T} rollout {b} (L={L}) differs from its window alone"
        assert torch.equal(cache[b, pad:].reshape(-1, 2 * D), kv_cache_of(k[b:b + 1, pad:], v[b:b + 1, pad:], rot)), \
            f"T={T} rollout {b} (L={L}): cache rows"
    _, full, _ = ragged_dense(lib, q, k, v, rot, [T] * B)
    _, ref = dense_attention(lib, q, k, v, rot)
    assert torch.equal(full.reshape(-1, D), ref)


@pytest.mark.parametrize("ctx", range(1, 32))
def test_ragged_last_equals_each_rollout_alone(lib, ctx):
    """On the cache the ragged dense kernel writes for the context frames (as the context pass does), the ragged last-frame
    kernel gives each rollout the bits of gtav_attention_temporal_last at ctx_frames = its valid count, and of the last row
    of the dense kernel over its window alone."""
    T = ctx + 1
    valid = [ctx, 0, (ctx + 1) // 2, 1]
    B = len(valid)
    rot = rot_table(32)
    q, k, v = temporal_inputs(B, T, "random", 3500 + T)
    _, _, cache = ragged_dense(lib, q[:, :ctx], k[:, :ctx], v[:, :ctx], rot, valid)
    qkv = torch.cat([to_rows(z) for z in (q, k, v)], dim=1).to(torch.bfloat16).view(B, T, P, 3 * D)
    last_qkv = qkv[:, T - 1].reshape(B * P, 3 * D).contiguous()
    out = ragged_last(lib, last_qkv, ctx, rot, valid, cache.reshape(-1, 2 * D)).view(B, P, D)
    for b, c in enumerate(valid):
        mine = last_qkv.view(B, P, 3 * D)[b].contiguous()
        solo_cache = cache[b, ctx - c:].reshape(-1, 2 * D).contiguous() if c else None
        ref = attention_last(lib, mine, c, rot, solo_cache)
        assert torch.equal(out[b], ref), f"ctx={ctx} rollout {b} ({c} valid cached frames)"
        _, dense = dense_attention(lib, q[b:b + 1, T - 1 - c:], k[b:b + 1, T - 1 - c:], v[b:b + 1, T - 1 - c:], rot)
        assert torch.equal(out[b], dense.view(c + 1, P, D)[c])


# ------------------------------------------------------------------------------------------ DiT plan with lengths
def dit(max_frames, depth=2, seed=0):
    from gtav_b200.model.dit import DiT
    m = DiT(depth=depth, max_frames=max_frames)
    m.load_state_dict(make_dit_state(DiTConfig(depth=depth), seed=seed), strict=True)
    return m.cuda().eval()


def ragged_plan_last_frame(model, x, t, a, lengths, owner):
    """Last-frame v [B, C, H, W] of every rollout through a plan with `lengths` attached: (context pass + last frame,
    full forward)."""
    N = _N()
    lib = N.load()
    B, T = x.shape[:2]
    model._pack()
    plan = model._plan(B, T, owner=owner)
    lens = torch.tensor(lengths, dtype=torch.int32, device="cuda")
    N.check(lib.gtav_dit_plan_set_window_lengths(plan, lens.data_ptr()), "set_window_lengths")
    x = x.contiguous()
    tr = t.reshape(-1).contiguous()
    act = a.reshape(B * T, -1).contiguous()
    rows = torch.arange(B * T, dtype=torch.int32, device="cuda").reshape(B, T)
    ctx_rows, last_rows = rows[:, :-1].contiguous(), rows[:, -1].contiguous()
    split = torch.empty((B, 16, 18, 32), dtype=torch.bfloat16, device="cuda")
    full = torch.empty((B, T, 16, 18, 32), dtype=torch.bfloat16, device="cuda")
    s = N.current_stream()
    N.check(lib.gtav_dit_conditioning(plan, tr.data_ptr(), act.data_ptr(), s), "conditioning")
    N.check(lib.gtav_dit_context(plan, x.data_ptr(), 0, ctx_rows.data_ptr(), s), "context")
    N.check(lib.gtav_dit_last_frame(plan, x.data_ptr(), 0, last_rows.data_ptr(), split.data_ptr(), s), "last frame")
    N.check(lib.gtav_dit_forward(plan, x.data_ptr(), 0, tr.data_ptr(), act.data_ptr(), full.data_ptr(), s), "forward")
    torch.cuda.synchronize()
    model._drop_plans(owner)
    return split, full[:, -1]


@pytest.mark.parametrize("mode", ["tiled", "default"])
def test_dit_plan_with_window_lengths(monkeypatch, mode):
    """B = 4 plans with lengths [5, 1, 3, 2] (T = 5) and [16, 9, 8, 1] (T = 16): each rollout's last-frame v, through context
    pass + last frame and through the full forward, equals forward_last_frame of its own window - bit for bit with the
    tiled GEMMs, within the split-vs-dense bound of 1 bf16 ulp of the output range (2^-6 = 0.0156) on the default path (GEMM
    kernels there depend on the row count)."""
    if mode == "tiled":
        monkeypatch.setenv("GTAV_SKINNY", "0")
        monkeypatch.setenv("GTAV_GEMM_SPLITK", "0")
    model = dit(16)
    for T, lengths, seed in ((5, [5, 1, 3, 2], 3101), (16, [16, 9, 8, 1], 3102)):
        B = len(lengths)
        x = seeded_randn((B, T, 16, 18, 32), seed).cuda()
        t = torch.randint(0, 1000, (B, T), generator=torch.Generator().manual_seed(seed)).cuda()
        a = torch.randn((B, T, 25), generator=torch.Generator().manual_seed(seed + 1)).cuda()
        for b, L in enumerate(lengths):           # padding: zero latents, as the pool loads them
            x[b, :T - L] = 0
        split, full = ragged_plan_last_frame(model, x, t, a, lengths, ("test", mode, T))
        for b, L in enumerate(lengths):
            ref = model.forward_last_frame(x[b:b + 1, T - L:], t[b:b + 1, T - L:], a[b:b + 1, T - L:])[:, 0]
            for name, got in (("context + last frame", split[b:b + 1]), ("full forward", full[b:b + 1])):
                err = float((got.float() - ref.float()).abs().max())
                print(f"{mode} T={T} rollout {b} (L={L}) {name}: max-abs {err:.5f}")
                assert torch.isfinite(got.float()).all()
                if mode == "tiled":
                    assert torch.equal(got, ref), (T, b, L, name, err)
                else:
                    assert err <= 2.0 ** -6, (T, b, L, name, err)


def test_b1_plan_with_full_lengths_equals_plan_without():
    """Default path, B = 1: the plan without lengths fuses the temporal attention into the weight-streaming to_qkv GEMM,
    the same plan with lengths [T] runs the ragged kernel; the last frame is the same bits, and detaching restores the
    fused path."""
    N = _N()
    lib = N.load()
    model = dit(5)
    x = seeded_randn((1, 5, 16, 18, 32), 3201).cuda()
    t = torch.tensor([[15, 15, 15, 15, 600]]).cuda()
    a = torch.randn((1, 5, 25), generator=torch.Generator().manual_seed(3202)).cuda()
    before = model.forward_last_frame(x, t, a)
    plan = model._plan(1, 5)
    lens = torch.tensor([5], dtype=torch.int32, device="cuda")
    N.check(lib.gtav_dit_plan_set_window_lengths(plan, lens.data_ptr()), "attach")
    with_lengths = model.forward_last_frame(x, t, a)
    N.check(lib.gtav_dit_plan_set_window_lengths(plan, None), "detach")
    after = model.forward_last_frame(x, t, a)
    assert torch.equal(with_lengths, before), float((with_lengths.float() - before.float()).abs().max())
    assert torch.equal(after, before)


# ------------------------------------------------------------------------------------------ StreamPool
@pytest.fixture(scope="module")
def vae():
    from gtav_b200.model.vae import AutoencoderKL
    m = AutoencoderKL(latent_dim=16, patch_size=20, enc_dim=1024, enc_depth=1, enc_heads=16, dec_dim=1024, dec_depth=1,
                      dec_heads=16, input_height=360, input_width=640)
    m.load_state_dict(make_vae_state(VAEConfig(enc_depth=1, dec_depth=1), seed=0), strict=True)
    return m.cuda().eval()


def prompt(n, seed):
    g = torch.Generator().manual_seed(seed)
    return (dummy_prompt(n) + 0.2 * torch.rand((n, 3, 360, 640), generator=g)).clamp(0, 1).cuda()


def action(seed, i):
    a = torch.zeros(25, device="cuda")
    a[(seed + i) % 25] = 1.0
    a[(3 * seed + 2 * i) % 25] += 0.5
    return a


# (step at which the session opens, prompt frames, step at which it closes or None); A's slot goes to D
SCENARIO = {"A": (0, 4, 4), "B": (2, 1, None), "C": (3, 2, None), "D": (5, 1, None)}
STEPS = 9


def run_pool(sampler, capacity=3):
    """Runs SCENARIO on a pool: {name: (latents [k, C, h, w], frames [k, H, W, 3])} per session."""
    pool = sampler.pool(capacity, use_actions=True)
    ids, got, done = {}, {}, {}
    for i in range(STEPS):
        for name, (start, n, end) in SCENARIO.items():
            if end == i:
                pool.close(ids[name])
                done[name] = ids.pop(name)
        for name, (start, n, end) in SCENARIO.items():
            if start == i:
                seed = ord(name)
                ids[name] = pool.open(prompt(n, seed), torch.stack([action(seed, j) for j in range(n)]),
                                      generator=torch.Generator(device="cuda").manual_seed(seed))
                got[name] = []
        res = pool.step(actions={name_id: action(ord(name), SCENARIO[name][1] + len(got[name])) for name, name_id in ids.items()})
        assert set(res) == set(ids.values())
        for name, sid in ids.items():
            got[name].append(res[sid])
    return {name: (torch.stack([z for _, z in r]), torch.stack([f for f, _ in r])) for name, r in got.items()}


def run_solo(sampler):
    """The same sessions as B = 1 FrameStreams, one after another."""
    out = {}
    for name, (start, n, end) in SCENARIO.items():
        seed = ord(name)
        st = sampler.stream(prompt(n, seed)[None], torch.stack([action(seed, j) for j in range(n)])[None],
                            generator=torch.Generator(device="cuda").manual_seed(seed))
        k = (end if end is not None else STEPS) - start
        frames, lats = [], []
        for j in range(k):
            f, z = st.next(action(seed, n + j)[None])
            frames.append(f[0])
            lats.append(z[0])
        out[name] = (torch.stack(lats), torch.stack(frames))
    return out


@pytest.mark.parametrize("max_frames", [5, 16])
@pytest.mark.parametrize("mode", ["tiled", "default"])
def test_pool_sessions_equal_solo_streams(monkeypatch, vae, max_frames, mode):
    """A opens with 4 prompt frames, B joins two frames later with 1, C later still, A closes and D takes its slot; all
    action-conditioned with seeded generators.  Each session's latents equal a B = 1 FrameStream's: bit for bit with the
    tiled GEMMs, and then the decoded pixels are within 4 LSB (decodes of different sizes may run different attention
    kernels); within test_frame_cache_equals_dense_sampling's bounds on the default path, where the latents themselves differ
    (the GEMM kernels depend on the row count), so the pixels are not held to the 4 LSB."""
    from gtav_b200.sampler import Sampler
    if mode == "tiled":
        monkeypatch.setenv("GTAV_SKINNY", "0")
        monkeypatch.setenv("GTAV_GEMM_SPLITK", "0")
    model = dit(max_frames)
    s = Sampler(model, vae, noise_steps=2)
    pool = run_pool(s)
    solo = run_solo(s)
    res = {}
    for name in SCENARIO:
        (zp, fp), (zs, fs) = pool[name], solo[name]
        assert zp.shape == zs.shape, name
        err = (zp - zs).abs()
        pix = int((fp.int() - fs.int()).abs().max())
        print(f"max_frames {max_frames} {mode} session {name}: latents max-abs {float(err.max()):.5f} "
              f"mean-abs {float(err.mean()):.6f}, pixels max {pix} LSB")
        res[name] = (torch.equal(zp, zs), float(err.max()), float(err.mean()), pix)
    for name, (equal, mx, mean, pix) in res.items():
        if mode == "tiled":
            assert equal and pix <= 4, (name, mx, pix)
        else:
            assert mx < 3e-2 and mean < 2e-3, (name, mx, mean)


def test_pool_graph_replay_reads_current_lengths(vae):
    """The pool without graphs equals the pool with graphs, bit for bit, across steps whose window lengths change: the
    replayed graph reads the lengths uploaded for its step."""
    from gtav_b200.sampler import Sampler
    model = dit(5)
    res = [run_pool(Sampler(model, vae, noise_steps=2, use_graph=g)) for g in (True, False)]
    for name in SCENARIO:
        assert torch.equal(res[0][name][0], res[1][name][0]), name
        assert torch.equal(res[0][name][1], res[1][name][1]), name


def test_pool_refusals(vae):
    from gtav_b200.sampler import Sampler
    model = dit(5)
    pool = Sampler(model, vae, noise_steps=1).pool(1, use_actions=True)
    with pytest.raises(RuntimeError, match="prompt_actions"):
        pool.open(prompt(1, 1))
    with pytest.raises(RuntimeError, match="prompt_video must be"):
        pool.open(prompt(1, 1)[None], torch.zeros(1, 25, device="cuda"))
    sid = pool.open(prompt(1, 1), torch.zeros(1, 25, device="cuda"))
    with pytest.raises(RuntimeError, match="slots are taken"):
        pool.open(prompt(1, 2), torch.zeros(1, 25, device="cuda"))
    with pytest.raises(RuntimeError, match="action is needed"):
        pool.step()
    with pytest.raises(RuntimeError, match="no open session"):
        pool.step(actions={sid: action(1, 0), sid + 1: action(1, 0)})
    pool.close(sid)
    with pytest.raises(RuntimeError, match="no open session"):
        pool.close(sid)
    plain = Sampler(model, vae, noise_steps=1).pool(1)
    sid = plain.open(prompt(1, 1))
    with pytest.raises(RuntimeError, match="without actions"):
        plain.step(actions={sid: action(1, 0)})
    frame, z = plain.step(decode=True)[sid]
    assert frame.shape == (360, 640, 3) and frame.dtype == torch.uint8 and z.shape == (16, 18, 32)
