"""Per-kernel parity on the GPU, called through the C ABI (ctypes), against plain torch fp32 math on
the same bf16 inputs with the reference's rounding points written out."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    import gtav_b200._native as N
    return N.load()


def _N():
    import gtav_b200._native as N
    return N


def r16(x):
    return x.to(torch.bfloat16).float()


def run_gemm(lib, A, W, epi, bias=None, res=None, gate=None, frame_row=None, rows_per_frame=1, bn=0, N_out=None, out=None):
    N = _N()
    M, K = A.shape
    Nn = W.shape[0] if N_out is None else N_out
    if out is None:
        out = torch.zeros((M, Nn), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_gemm_bf16(A.data_ptr(), A.stride(0), W.data_ptr(), W.stride(0), out.data_ptr(), out.stride(0), M, Nn, K,
                               epi, N.ptr(bias), N.ptr(res), 0 if res is None else res.stride(0), N.ptr(gate),
                               0 if gate is None else gate.stride(0), N.ptr(frame_row), rows_per_frame, bn,
                               N.current_stream()), "gemm")
    torch.cuda.synchronize()
    return out


def close_bf16(out, ref, ulps=2.0, atol=1e-3, mag=None):
    """|out - ref| within a couple of bf16 ulps of the fp32 reference (accumulation-order noise).
    `mag` = magnitude of the largest intermediate when the result is a sum that can cancel."""
    err = (out.float() - ref).abs()
    tol = ulps * (ref.abs() if mag is None else torch.maximum(ref.abs(), mag)) * 2 ** -8 + atol
    bad = err > tol
    assert not bool(bad.any()), (f"{int(bad.sum())}/{bad.numel()} elements off; max err {float(err.max()):.5f} "
                                 f"at {torch.nonzero(bad)[:5].tolist()}")


@pytest.mark.parametrize("M,N,K,bn", [
    (128, 128, 64, 128), (128, 256, 128, 256), (128, 64, 64, 64),        # single tile, 1-2 k-blocks
    (720, 3072, 1024, 0), (720, 1024, 4096, 0), (720, 4096, 1024, 0),    # DiT hot shapes at B=1
    (5760, 1024, 1024, 0), (5760, 4096, 1024, 256),                      # B=8
    (5, 2048, 1024, 0), (200, 64, 1024, 0), (576, 1200, 1024, 0), (576, 1024, 1200, 0), (576, 32, 1024, 0),
    (576, 1024, 64, 0), (1000, 1024, 256, 0),
])
def test_gemm_store(lib, M, N, K, bn):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    out = run_gemm(lib, A, W, _N().EPI_STORE, bn=bn)
    close_bf16(out, A.float() @ W.float().t())


def test_gemm_strided_operands(lib):
    """Leading dimensions larger than the logical width (views into wider buffers)."""
    g = torch.Generator(device="cuda").manual_seed(5)
    Abig = torch.randn((300, 1024 + 64), device="cuda", generator=g).to(torch.bfloat16)
    A = Abig[:, :1024]
    W = (torch.randn((256, 1024), device="cuda", generator=g) / 32).to(torch.bfloat16)
    out = run_gemm(lib, A, W, _N().EPI_STORE)
    close_bf16(out, A.float() @ W.float().t())


@pytest.mark.parametrize("epi_name", ["BIAS", "GELU_TANH", "GELU_ERF", "SILU", "GATE_RES", "RES", "RES_SILU", "RES_SILU_NORES"])
def test_gemm_epilogues(lib, epi_name):
    N = _N()
    M, Nn, K, S = 432, 1024, 1024, 144
    g = torch.Generator(device="cuda").manual_seed(17)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((Nn, K), device="cuda", generator=g) / 32).to(torch.bfloat16)
    bias = (torch.randn((Nn,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    res = torch.randn((M, Nn), device="cuda", generator=g).to(torch.bfloat16)
    modw = 3 * Nn
    gate_tab = torch.randn((5, modw), device="cuda", generator=g).to(torch.bfloat16)
    frame_row = torch.tensor([4, 0, 2], dtype=torch.int32, device="cuda")
    y = r16(A.float() @ W.float().t() + bias.float())
    kw = dict(bias=bias)
    mag = None
    if epi_name == "BIAS":
        epi, ref = N.EPI_BIAS, y
    elif epi_name == "GELU_TANH":
        epi, ref = N.EPI_BIAS_GELU_TANH, torch.nn.functional.gelu(y, approximate="tanh")
    elif epi_name == "GELU_ERF":
        epi, ref = N.EPI_BIAS_GELU_ERF, torch.nn.functional.gelu(y)
    elif epi_name == "SILU":
        epi, ref = N.EPI_BIAS_SILU, torch.nn.functional.silu(y)
    elif epi_name == "GATE_RES":
        epi = N.EPI_BIAS_GATE_RES
        gate = gate_tab[:, Nn:2 * Nn]
        grow = gate[frame_row.long()].float().repeat_interleave(S, dim=0)
        ref = res.float() + r16(grow * y)
        mag = res.float().abs() + (grow * y).abs()
        kw.update(res=res, gate=gate, frame_row=frame_row, rows_per_frame=S)
    elif epi_name == "RES":
        epi, ref = N.EPI_BIAS_RES, res.float() + y
        mag = res.float().abs() + y.abs()
        kw.update(res=res)
    elif epi_name == "RES_SILU":
        epi, ref = N.EPI_BIAS_RES_SILU, torch.nn.functional.silu(r16(res.float() + y))
        kw.update(res=res)
    else:
        epi, ref = N.EPI_BIAS_RES_SILU, torch.nn.functional.silu(y)
    out = run_gemm(lib, A, W, epi, **kw)
    close_bf16(out, ref, ulps=3.0, atol=4e-3, mag=mag)


def test_gemm_inplace_residual(lib):
    """The DiT residual update writes back into the residual stream buffer."""
    N = _N()
    g = torch.Generator(device="cuda").manual_seed(3)
    A = torch.randn((720, 1024), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((1024, 1024), device="cuda", generator=g) / 32).to(torch.bfloat16)
    bias = torch.zeros(1024, device="cuda", dtype=torch.bfloat16)
    x = torch.randn((720, 1024), device="cuda", generator=g).to(torch.bfloat16)
    xin = x.float().clone()
    ref = xin + r16(A.float() @ W.float().t())
    M = 720
    N.check(lib.gtav_gemm_bf16(A.data_ptr(), 1024, W.data_ptr(), 1024, x.data_ptr(), 1024, M, 1024, 1024, N.EPI_BIAS_RES,
                               bias.data_ptr(), x.data_ptr(), 1024, None, 0, None, 1, 0, N.current_stream()), "gemm")
    torch.cuda.synchronize()
    close_bf16(x, ref, ulps=3.0, atol=4e-3, mag=xin.abs() + (ref - xin).abs())


def test_gemm_rejects_bad_arguments(lib):
    N = _N()
    A = torch.zeros((16, 60), device="cuda", dtype=torch.bfloat16)
    W = torch.zeros((64, 60), device="cuda", dtype=torch.bfloat16)
    out = torch.zeros((16, 64), device="cuda", dtype=torch.bfloat16)
    rc = lib.gtav_gemm_bf16(A.data_ptr(), 60, W.data_ptr(), 60, out.data_ptr(), 64, 16, 64, 60, 0, None, None, 0, None, 0,
                            None, 1, 0, N.current_stream())
    assert rc != 0 and b"multiples of 8" in lib.gtav_last_error()
    rc = lib.gtav_gemm_bf16(A.data_ptr(), 64, W.data_ptr(), 64, out.data_ptr(), 64, 16, 64, 64, N.EPI_BIAS, None, None, 0,
                            None, 0, None, 1, 0, N.current_stream())
    assert rc != 0 and b"bias" in lib.gtav_last_error()


def test_ln_modulate(lib):
    N = _N()
    M, D, S = 720, 1024, 144
    g = torch.Generator(device="cuda").manual_seed(23)
    x = (torch.randn((M, D), device="cuda", generator=g) * 2 + 0.3).to(torch.bfloat16)
    mod = (torch.randn((7, 6 * D), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    mod[0, D:D + 8] = 0.0                                       # scale == 0: the +1e-6 survives in bf16
    frame_row = torch.tensor([3, 0, 6, 1, 5], dtype=torch.int32, device="cuda")
    out = torch.empty_like(x)
    N.check(lib.gtav_ln_modulate(x.data_ptr(), out.data_ptr(), M, D, mod.data_ptr(), 6 * D, 0, D, frame_row.data_ptr(), S,
                                 N.current_stream()), "ln_modulate")
    rows = frame_row.long().repeat_interleave(S)
    shift, scale = mod[rows, :D], mod[rows, D:2 * D]
    ln = torch.nn.functional.layer_norm(x.float(), (D,), eps=1e-6)
    ref = ln * (1 + (scale + 1e-6)).float() + shift.float()      # bf16 tensor ops, as in dit.py:26-27
    close_bf16(out, ref, ulps=1.5, atol=2e-3)
    # identity frame_row
    N.check(lib.gtav_ln_modulate(x.data_ptr(), out.data_ptr(), M, D, mod.data_ptr(), 6 * D, 3 * D, 4 * D, None, S,
                                 N.current_stream()), "ln_modulate")
    rows = torch.arange(5, device="cuda").repeat_interleave(S)
    ref = ln * (1 + (mod[rows, 4 * D:5 * D] + 1e-6)).float() + mod[rows, 3 * D:4 * D].float()
    close_bf16(out, ref, ulps=1.5, atol=2e-3)


def test_ln_affine(lib):
    N = _N()
    M, D = 576 + 3, 1024
    g = torch.Generator(device="cuda").manual_seed(29)
    x = (torch.randn((M, D), device="cuda", generator=g) * 3 - 1).to(torch.bfloat16)
    w = 1 + 0.1 * torch.randn(D, device="cuda", generator=g)
    b = 0.1 * torch.randn(D, device="cuda", generator=g)
    out = torch.empty_like(x)
    N.check(lib.gtav_ln_affine(x.data_ptr(), out.data_ptr(), M, D, w.data_ptr(), b.data_ptr(), N.current_stream()), "ln")
    close_bf16(out, torch.nn.functional.layer_norm(x.float(), (D,), w, b, eps=1e-6), ulps=1.5, atol=2e-3)


def _rot_table(ang):
    return torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()


def _rotate(x, ang):
    """x [..., S, d] fp32 (bf16 values); ang [S, n_pairs]; rotate the first 2*n_pairs features, round to bf16."""
    n = ang.shape[-1] * 2
    a = ang.repeat_interleave(2, dim=-1)
    head, tail = x[..., :n], x[..., n:]
    pair = head.reshape(*head.shape[:-1], n // 2, 2)
    sw = torch.stack((-pair[..., 1], pair[..., 0]), dim=-1).reshape(head.shape)
    return torch.cat([r16(head * a.cos() + sw * a.sin()), tail], dim=-1)


@pytest.mark.parametrize("impl", ["tc", "mma"])
@pytest.mark.parametrize("seq,pairs,groups", [(144, 32, 5), (576, 16, 2), (576, 16, 11), (144, 32, 1)])
def test_attention_seq(lib, monkeypatch, seq, pairs, groups, impl):
    """impl tc: the tcgen05 kernel (attn_tc.cu, the default); mma: the mma.sync kernel it replaced (GTAV_ATTN=mma)."""
    monkeypatch.setenv("GTAV_ATTN", impl)
    N = _N()
    H, d = 16, 64
    g = torch.Generator(device="cuda").manual_seed(seq)
    qkv = torch.randn((groups * seq, 3 * H * d), device="cuda", generator=g).to(torch.bfloat16)
    ang = torch.rand((seq, pairs), device="cuda", generator=g) * 20 - 10
    rot = _rot_table(ang)
    out = torch.empty((groups * seq, H * d), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_seq(qkv.data_ptr(), out.data_ptr(), groups, seq, H, rot.data_ptr(), pairs,
                                   N.current_stream()), "attention_seq")
    q, k, v = [z.float().reshape(groups, seq, H, d).permute(0, 2, 1, 3) for z in qkv.chunk(3, dim=-1)]
    q, k = _rotate(q, ang), _rotate(k, ang)
    p = torch.softmax(q @ k.transpose(-1, -2) / 8.0, dim=-1)
    ref = (p @ v).permute(0, 2, 1, 3).reshape(groups * seq, H * d)
    err = (out.float() - ref).abs()
    assert float(err.max()) < 2e-2 and float(err.mean()) < 2e-3, (float(err.max()), float(err.mean()))


def test_attention_seq_rescale_stress(lib, monkeypatch):
    """The tcgen05 attention under the conditions that once stalled it in a VAE decode: logits whose block maximum jumps by
    > 2^8 from key block to key block in half of the heads (the rare rescale path of the lazy online softmax runs in every
    tile there, never in the other heads, so the softmax groups of a CTA drift apart), many CTAs, many launches.  Every
    launch must give the same bits, and those must match the fp32 softmax."""
    monkeypatch.setenv("GTAV_ATTN", "tc")
    N = _N()
    H, d, seq, pairs, groups = 16, 64, 576, 16, 40
    g = torch.Generator(device="cuda").manual_seed(7)
    qkv = (torch.randn((groups, seq, 3, H, d), device="cuda", generator=g) * 0.5)
    pos = torch.arange(seq, device="cuda").float()
    step = torch.where(torch.arange(H, device="cuda") % 2 == 0, 1.0, -1.0)           # rising / falling block maxima per head
    c = 9.0 * torch.floor(pos / 96.0)[:, None] * step[None, :]                      # [seq, H]: +-9 logits per 96 keys
    qkv[:, :, 0, :, 40] = 8.0                                                        # q . k / 8 = c(key) (+ noise); dim 40 is not rotated
    qkv[:, :, 1, :, 40] = c[None]
    qkv = qkv.reshape(groups * seq, 3 * H * d).to(torch.bfloat16)
    ang = torch.rand((seq, pairs), device="cuda", generator=g) * 20 - 10
    rot = _rot_table(ang)
    outs = []
    for _ in range(12):
        out = torch.empty((groups * seq, H * d), dtype=torch.bfloat16, device="cuda")
        N.check(lib.gtav_attention_seq(qkv.data_ptr(), out.data_ptr(), groups, seq, H, rot.data_ptr(), pairs,
                                       N.current_stream()), "attention_seq")
        outs.append(out)
    torch.cuda.synchronize()
    for o in outs[1:]:
        assert torch.equal(o, outs[0])
    q, k, v = [z.float().reshape(groups, seq, H, d).permute(0, 2, 1, 3) for z in qkv.chunk(3, dim=-1)]
    q, k = _rotate(q, ang), _rotate(k, ang)
    p = torch.softmax(q @ k.transpose(-1, -2) / 8.0, dim=-1)
    ref = (p @ v).permute(0, 2, 1, 3).reshape(groups * seq, H * d)
    err = (outs[0].float() - ref).abs()
    assert float(err.max()) < 2e-2 and float(err.mean()) < 2e-3, (float(err.max()), float(err.mean()))


@pytest.mark.parametrize("B,T", [(1, 5), (2, 3), (1, 1)])
def test_attention_temporal(lib, B, T):
    N = _N()
    H, d, P = 16, 64, 144
    g = torch.Generator(device="cuda").manual_seed(T)
    qkv = torch.randn((B * T * P, 3 * H * d), device="cuda", generator=g).to(torch.bfloat16)
    base = 1.0 / (10000 ** (torch.arange(0, 64, 2, device="cuda").float() / 64))
    ang = torch.arange(5, device="cuda").float()[:, None] * base[None]
    rot = _rot_table(ang)
    out = torch.empty((B * T * P, H * d), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_temporal(qkv.data_ptr(), out.data_ptr(), B, T, P, H, rot.data_ptr(), N.current_stream()),
            "attention_temporal")
    q, k, v = [z.float().reshape(B, T, P, H, d).permute(0, 2, 3, 1, 4) for z in qkv.chunk(3, dim=-1)]   # B P H T d
    q, k = _rotate(q, ang[:T]), _rotate(k, ang[:T])
    s = q @ k.transpose(-1, -2) / 8.0
    s = s.masked_fill(torch.ones(T, T, dtype=torch.bool, device="cuda").triu(1), float("-inf"))
    ref = (torch.softmax(s, dim=-1) @ v).permute(0, 3, 1, 2, 4).reshape(B * T * P, H * d)
    err = (out.float() - ref).abs()
    assert float(err.max()) < 2e-2 and float(err.mean()) < 2e-3, (float(err.max()), float(err.mean()))


def test_ddim_update_bit_exact(lib):
    """fp32 elementwise chain == the reference's tensor expression (train_dit.py:110-123), bit for bit."""
    N = _N()
    from oracle.reference_port import alphas_cumprod_table, ddim_update
    F, n = 6, 16 * 18 * 32
    g = torch.Generator(device="cuda").manual_seed(31)
    x = torch.randn((F, n), device="cuda", generator=g)
    v = torch.randn((F, n), device="cuda", generator=g).to(torch.bfloat16)
    abar = alphas_cumprod_table().cuda()
    a_t = abar[torch.tensor([15, 15, 999, 509, 9, 0], device="cuda")].contiguous()
    a_n = abar[torch.tensor([15, 15, 989, 499, 0, 0], device="cuda")].contiguous()
    a_n[:2] = 1.0
    for fin in (0, 1):
        flag = torch.tensor([fin], dtype=torch.int32, device="cuda")
        out = torch.empty_like(x)
        N.check(lib.gtav_ddim_update(x.data_ptr(), v.data_ptr(), out.data_ptr(), F, n, a_t.data_ptr(), a_n.data_ptr(),
                                     flag.data_ptr(), N.current_stream()), "ddim")
        ref = ddim_update(x, v.float(), a_t[:, None], a_n[:, None], bool(fin))
        assert torch.equal(out, ref), float((out - ref).abs().max())


# ------------------------------------------------------------------------------------------ weight-streaming GEMM
def run_skinny(lib, A, W, epi, bias=None, res=None, gate=None, frame_row=None, rows_per_frame=144, splits=0, out=None, state=None):
    N = _N()
    M, K = A.shape
    Nn = W.shape[0]
    if out is None:
        out = torch.zeros((M, Nn), dtype=torch.bfloat16, device="cuda")
    if state is None:
        state = (torch.empty(lib.gtav_gemm_skinny_workspace_bytes(M), dtype=torch.uint8, device="cuda"),
                 torch.zeros(512, dtype=torch.int32, device="cuda"))
    ws, counters = state
    N.check(lib.gtav_gemm_skinny_bf16(A.data_ptr(), A.stride(0), W.data_ptr(), W.stride(0), out.data_ptr(), out.stride(0), M, Nn, K,
                                      epi, N.ptr(bias), N.ptr(res), 0 if res is None else res.stride(0), N.ptr(gate),
                                      0 if gate is None else gate.stride(0), N.ptr(frame_row), rows_per_frame, splits,
                                      ws.data_ptr(), counters.data_ptr(), N.current_stream()), "gemm_skinny")
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("M,N,K,splits", [
    (144, 128, 64, 1), (144, 128, 256, 1), (144, 128, 256, 2), (144, 256, 512, 4),       # small: no split, 2- and 4-way split
    (144, 3072, 1024, 0), (144, 1024, 1024, 0), (144, 4096, 1024, 0), (144, 1024, 4096, 0),   # last-frame shapes at B=1
    (288, 1024, 1024, 0), (288, 512, 1024, 8), (432, 1024, 1024, 0), (432, 256, 512, 8),       # B = 2, 3 (where the slab fits)
])
def test_skinny_gemm_store(lib, M, N, K, splits):
    g = torch.Generator(device="cuda").manual_seed(M + N * 3 + K * 5)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    out = run_skinny(lib, A, W, _N().EPI_STORE, splits=splits)
    close_bf16(out, A.float() @ W.float().t())


def test_skinny_gemm_epilogues_and_reuse(lib):
    """The fused epilogues, repeated calls on the same workspace/counters (they must reset themselves), in-place residual."""
    N = _N()
    M, Nn, K, S = 288, 1024, 1024, 144
    g = torch.Generator(device="cuda").manual_seed(23)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((Nn, K), device="cuda", generator=g) / 32).to(torch.bfloat16)
    bias = (torch.randn((Nn,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    res = torch.randn((M, Nn), device="cuda", generator=g).to(torch.bfloat16)
    gate_tab = torch.randn((5, 3 * Nn), device="cuda", generator=g).to(torch.bfloat16)
    gate = gate_tab[:, Nn:2 * Nn]
    frame_row = torch.tensor([3, 1], dtype=torch.int32, device="cuda")
    state = (torch.empty(lib.gtav_gemm_skinny_workspace_bytes(M), dtype=torch.uint8, device="cuda"),
             torch.zeros(512, dtype=torch.int32, device="cuda"))
    y = r16(A.float() @ W.float().t() + bias.float())
    for _ in range(3):
        out = run_skinny(lib, A, W, N.EPI_BIAS, bias=bias, state=state)
        close_bf16(out, y, ulps=3.0, atol=4e-3)
        out = run_skinny(lib, A, W, N.EPI_BIAS_GELU_TANH, bias=bias, state=state)
        close_bf16(out, torch.nn.functional.gelu(y, approximate="tanh"), ulps=3.0, atol=4e-3)
        grow = gate[frame_row.long()].float().repeat_interleave(S, dim=0)
        ref = res.float() + r16(grow * y)
        h = res.clone()
        run_skinny(lib, A, W, N.EPI_BIAS_GATE_RES, bias=bias, res=h, gate=gate, frame_row=frame_row, out=h, state=state)
        close_bf16(h, ref, ulps=3.0, atol=4e-3, mag=res.float().abs() + (grow * y).abs())
    # rendezvous state after 9 launches on 8 row blocks: each group {count A, count B, which} has one stale total and
    # one cleared counter, nothing else was touched
    st = state[1].cpu().view(-1, 4)
    assert int(st[8:].abs().sum()) == 0 and bool(((st[:8, 0] == 0) | (st[:8, 1] == 0)).all())


def test_skinny_tagged_exchange(lib):
    """gtav_gemm_skinny_tagged_bf16: partial sums tagged with the launch's parity instead of the counter rendezvous.  Four
    launches on one zeroed workspace with parity 1, 0, 1, 0 (fresh inputs each time, so a stale partial sum accepted by
    mistake would show) against the fp32 product and against the counter version, every split count and 1-3 frame tiles."""
    N = _N()
    for M, Nn, K, splits in ((144, 3072, 1024, 0), (144, 1024, 4096, 0), (288, 1024, 1024, 0), (432, 256, 512, 8), (144, 128, 256, 2)):
        ws = torch.zeros(lib.gtav_gemm_skinny_workspace_bytes(M), dtype=torch.uint8, device="cuda")
        g = torch.Generator(device="cuda").manual_seed(M + Nn + K)
        bias = (torch.randn((Nn,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
        for launch in range(4):
            A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
            W = (torch.randn((Nn, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
            out = torch.zeros((M, Nn), dtype=torch.bfloat16, device="cuda")
            N.check(lib.gtav_gemm_skinny_tagged_bf16(A.data_ptr(), K, W.data_ptr(), K, out.data_ptr(), Nn, M, Nn, K, N.EPI_BIAS,
                                                     bias.data_ptr(), None, 0, None, 0, None, 144, splits, ws.data_ptr(),
                                                     (launch & 1) ^ 1, N.current_stream()), "gemm_skinny_tagged")
            torch.cuda.synchronize()
            close_bf16(out, A.float() @ W.float().t() + bias.float())
            ref = run_skinny(lib, A, W, N.EPI_BIAS, bias=bias, splits=splits)
            d = (out.float() - ref.float()).abs()
            assert float((d > 0).float().mean()) < 1e-3 and float(d.max()) <= 2 ** -7 * float(ref.float().abs().max())
    with pytest.raises(RuntimeError, match="parity"):
        N.check(lib.gtav_gemm_skinny_tagged_bf16(A.data_ptr(), K, W.data_ptr(), K, out.data_ptr(), Nn, M, Nn, K, N.EPI_BIAS, bias.data_ptr(),
                                                 None, 0, None, 0, None, 144, splits, ws.data_ptr(), 2, N.current_stream()), "gemm_skinny_tagged")


def test_skinny_matches_tiled_gemm(lib):
    """Same inputs through both GEMM kernels: only the fp32 summation order differs."""
    N = _N()
    g = torch.Generator(device="cuda").manual_seed(29)
    A = torch.randn((144, 4096), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((1024, 4096), device="cuda", generator=g) / 64).to(torch.bfloat16)
    a = run_skinny(lib, A, W, N.EPI_STORE)
    b = run_gemm(lib, A, W, N.EPI_STORE)
    assert float((a.float() - b.float()).abs().max()) <= 2 ** -7 * float(b.float().abs().max())


def test_temporal_attention_last_frame_matches_dense(lib):
    """attn_temporal_last on cached K/V == the last-frame rows of the dense causal kernel, bit for bit."""
    N = _N()
    B, T, P, H = 2, 5, 144, 16
    D = H * 64
    g = torch.Generator(device="cuda").manual_seed(31)
    qkv = torch.randn((B * T * P, 3 * D), device="cuda", generator=g).to(torch.bfloat16)
    ang = torch.arange(T, device="cuda", dtype=torch.float32)[:, None] * (1.0 / (10000 ** (torch.arange(0, 64, 2, device="cuda").float() / 64)))[None]
    rot = torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()
    dense = torch.zeros((B * T * P, D), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_temporal(qkv.data_ptr(), dense.data_ptr(), B, T, P, H, rot.data_ptr(), N.current_stream()), "dense")
    # context pass on the first T-1 frames with the cache-writing variant is exercised through the engine
    # (test_model_gpu.py); here the cache is rebuilt by hand: rotated K (bf16) and V of frames 0..T-2
    q5 = qkv.view(B, T, P, 3, H, 64)
    k = q5[:, : T - 1, :, 1].float()
    kr = torch.empty_like(k)
    c, s = ang[: T - 1].cos()[None, :, None, None], ang[: T - 1].sin()[None, :, None, None]
    kr[..., 0::2] = k[..., 0::2] * c - k[..., 1::2] * s
    kr[..., 1::2] = k[..., 1::2] * c + k[..., 0::2] * s
    cache = torch.stack([kr.to(torch.bfloat16).reshape(B, T - 1, P, D), q5[:, : T - 1, :, 2].reshape(B, T - 1, P, D)], dim=3).contiguous()
    last_qkv = q5[:, T - 1].reshape(B * P, 3 * D).contiguous()
    out = torch.zeros((B * P, D), dtype=torch.bfloat16, device="cuda")
    import ctypes as C
    fn = lib.gtav_attention_temporal_last
    N.check(fn(last_qkv.data_ptr(), out.data_ptr(), B, T - 1, P, H, rot.data_ptr(), cache.data_ptr(), N.current_stream()), "last")
    torch.cuda.synchronize()
    ref = dense.view(B, T, P, D)[:, T - 1].reshape(B * P, D)
    assert torch.equal(out, ref), float((out.float() - ref.float()).abs().max())



@pytest.mark.parametrize("M,N,K", [(256, 256, 128), (512, 512, 256), (1152, 1024, 1024), (1000, 3072, 1024), (2304, 1024, 4096),
                                   (4608, 4096, 1024)])
def test_gemm_cta_pair_equals_single_cta(lib, monkeypatch, M, N, K):
    """tcgen05.mma.cta_group::2 on 256 x 256 tile pairs (gemm_sm100_2cta.cu) accumulates every output element over K in
    the same order as the single-CTA kernel: same bits, including the ragged last row pair."""
    Nmod = _N()
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = (torch.randn((N,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    outs = {}
    for mode in ("0", "1"):
        monkeypatch.setenv("GTAV_GEMM_2CTA", mode)
        outs[mode] = (run_gemm(lib, A, W, Nmod.EPI_STORE), run_gemm(lib, A, W, Nmod.EPI_BIAS_GELU_TANH, bias=bias))
    close_bf16(outs["1"][0], A.float() @ W.float().t())
    assert torch.equal(outs["0"][0], outs["1"][0]) and torch.equal(outs["0"][1], outs["1"][1])


@pytest.mark.parametrize("M,N,K", [(1152, 1024, 4096), (720, 1024, 4096), (144, 1024, 2048), (1000, 256, 2048), (576, 1024, 4096)])
def test_gemm_split_k_pair(lib, monkeypatch, M, N, K):
    """Split-K over the two CTAs of a cluster with the DSMEM reduce (gemm_sm100_splitk.cu; chosen for few tiles and K >= 2048,
    i.e. fc2 at M <= 1152): plain store, GELU and the gated in-place residual against the fp32 product, and within the
    rounding of the summation order of the single-CTA kernel (GTAV_GEMM_SPLITK=0)."""
    Nmod = _N()
    S = 144
    g = torch.Generator(device="cuda").manual_seed(M + N + K + 1)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = (torch.randn((N,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    res = torch.randn((M, N), device="cuda", generator=g).to(torch.bfloat16)
    frames = (M + S - 1) // S
    gate = torch.randn((frames + 1, N), device="cuda", generator=g).to(torch.bfloat16)
    frame_row = torch.arange(frames, 0, -1, dtype=torch.int32, device="cuda")
    outs = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("GTAV_GEMM_SPLITK", mode)
        h = res.clone()
        run_gemm(lib, A, W, Nmod.EPI_BIAS_GATE_RES, bias=bias, res=h, gate=gate, frame_row=frame_row, rows_per_frame=S, out=h)
        outs[mode] = (run_gemm(lib, A, W, Nmod.EPI_STORE), run_gemm(lib, A, W, Nmod.EPI_BIAS_GELU_TANH, bias=bias), h)
    prod = A.float() @ W.float().t()
    y = r16(prod + bias.float())
    grow = gate[frame_row.long()].float().repeat_interleave(S, dim=0)[:M]
    close_bf16(outs["1"][0], prod)
    # (y itself may sit one bf16 ulp away from the fp32 product's rounding at K = 4096; the gate multiplies that)
    close_bf16(outs["1"][1], torch.nn.functional.gelu(y, approximate="tanh"), ulps=3.0)
    close_bf16(outs["1"][2], res.float() + r16(grow * y), ulps=4.0, mag=res.float().abs() + (grow * y).abs())
    for a, b in zip(outs["1"], outs["0"]):
        d = (a.float() - b.float()).abs()
        assert float(d.max()) <= 0.07 and float((d > 0).float().mean()) < 0.05, (float(d.max()), float((d > 0).float().mean()))


def test_gemm_cta_pair_gated_residual_in_place(lib, monkeypatch):
    """The CTA-pair kernel with the adaLN gate + in-place residual epilogue and a frame_row indirection (B = 8 shape)."""
    Nmod = _N()
    monkeypatch.setenv("GTAV_GEMM_2CTA", "1")
    M, N, K, S = 1152, 1024, 1024, 144
    g = torch.Generator(device="cuda").manual_seed(77)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((N, K), device="cuda", generator=g) / 32).to(torch.bfloat16)
    bias = (torch.randn((N,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    res = torch.randn((M, N), device="cuda", generator=g).to(torch.bfloat16)
    gate = torch.randn((9, N), device="cuda", generator=g).to(torch.bfloat16)
    frame_row = torch.tensor([3, 1, 4, 1, 5, 8, 2, 6], dtype=torch.int32, device="cuda")
    y = r16(A.float() @ W.float().t() + bias.float())
    grow = gate[frame_row.long()].float().repeat_interleave(S, dim=0)
    ref = res.float() + r16(grow * y)
    h = res.clone()
    Nn = _N()
    Nn.check(lib.gtav_gemm_bf16(A.data_ptr(), K, W.data_ptr(), K, h.data_ptr(), N, M, N, K, Nn.EPI_BIAS_GATE_RES, bias.data_ptr(),
                                h.data_ptr(), N, gate.data_ptr(), N, frame_row.data_ptr(), S, 0, Nn.current_stream()), "gemm")
    torch.cuda.synchronize()
    close_bf16(h, ref, ulps=3.0, atol=4e-3, mag=res.float().abs() + (grow * y).abs())
