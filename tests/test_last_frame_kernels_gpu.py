"""Kernel-level parity of the last-frame chain: the weight-streaming GEMM with the LayerNorm / temporal attention fused into
its split-K reduce, its tagged split-K exchange under every epilogue the engine runs it with, and the temporal attention at
every window length.

Every reference is computed in float64 from the same bf16 inputs with the kernels' bf16 rounding points written out: the
Linear's output, the gate product, the residual sum, the modulation factor, the rotated q / k and the softmax probabilities.
Between two rounding points the kernels work in fp32, so a kernel's value can only differ from the reference where an fp32
error moves a value across a bf16 rounding boundary.  Each bound below is that fp32 error, carried through the later
rounding points, plus one bf16 ulp for the final rounding. In practice that is one or two bf16 ulps of the output, not an
absolute 2e-2.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

D, H, P = 1024, 16, 144                    # hidden width, heads of 64, tokens per frame
MOD_LD = 16 * 2 * 6 * D + 2 * D            # modulation row width of the 16-block DiT (gtav_dit_mod_width)
LN, TATTN = 1, 2                           # modes of gtav_gemm_skinny_fused_bf16


@pytest.fixture(scope="module")
def lib():
    import gtav_b200._native as N
    return N.load()


def _N():
    import gtav_b200._native as N
    return N


# ------------------------------------------------------------------------------------------ float64 rounding model
def r16(x):
    """Round-to-nearest-even of float64 values to bf16 (8 significant bits), exact in float64."""
    m, e = torch.frexp(x)
    return torch.round(m * 256) * torch.exp2((e - 8).double())


def ulp(x):
    """Spacing of the bf16 numbers at |x| (float64)."""
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -120))
    return torch.exp2((e - 8).double())


def round_diff(ref, delta):
    """Bound on |bf16(a) - ref| when ref = bf16(b) and |a - b| <= delta.  Each rounding is off by at most half an ulp,
    taken at the larger magnitude (|a| <= |b| + delta and |b| <= 1.01 |ref|)."""
    return delta + ulp(ref.abs() * 1.01 + delta)


def assert_within(out, ref, tol, what):
    err = (out.double() - ref).abs()
    bad = err > tol
    if bool(bad.any()):
        worst = float((err / tol.clamp_min(1e-300)).max())
        raise AssertionError(f"{what}: {int(bad.sum())}/{bad.numel()} elements outside the bound (worst err / bound {worst:.2f}), "
                             f"first at {torch.nonzero(bad)[:4].tolist()}")


def assert_last_bit_close(out, ref, what):
    """Tagged vs counter exchange: the tag costs each fp32 partial sum its last mantissa bit (2^-24 relative), which flips
    an occasional bf16 rounding.  This is the same bound test_kernels_gpu.py::test_skinny_tagged_exchange uses."""
    d = (out.float() - ref.float()).abs()
    frac = float((d > 0).float().mean())
    assert frac < 1e-3 and float(d.max()) <= 2 ** -7 * float(ref.float().abs().max()), (what, frac, float(d.max()))


def linear_ref(A, W, bias, S):
    """float64 A @ W^T (+ bias), and a bound E on the distance of the kernel's fp32 pre-rounding value from it.  The fp32
    value passes through K / 16 tensor-core accumulation steps (16 exact bf16 products each) spread over the S splits, the
    split-order reduce of the S partial sums (each of which may also have lost its last bit to the tag) and the bias add.
    Each step errs by at most 2^-23 of a running sum bounded by sum |a w|, and the factor 2 covers the tensor core's own
    sum of a step's 16 products."""
    a, w = A.double(), W.double()
    acc = a @ w.t()
    if bias is not None:
        acc = acc + bias.double()
    K = A.shape[1]
    E = 2.0 ** -22 * (K / 16 + 2 * S) * (a.abs() @ w.abs().t()) + 2.0 ** -23 * acc.abs()
    return acc, E


def epilogue_ref(acc, E, epi, gate=None, res=None):
    """bf16 reference of the skinny epilogues (gemm_skinny.cu skinny_epi4) and the bound per element.
    y = bf16(acc + b): |y - y_ref| <= round_diff(y_ref, E).
    GELU_TANH: gelu' <= 1.13, and the kernel's gelu is within 2^-20 of tanh-GELU (common.cuh), so the bound is
    round_diff(gelu_ref, 1.13 dy + 2^-18 |gelu|).
    GATE_RES: bf16(g y) is off by at most round_diff(gy_ref, |g| dy).  The sum r + gy of two bf16 values is exact in fp32
    (or off by 2^-24), and bf16(r + gy) is off by round_diff of that."""
    N = _N()
    y = r16(acc)
    dy = round_diff(y, E)
    if epi in (N.EPI_STORE, N.EPI_BIAS):
        return y, dy
    if epi == N.EPI_BIAS_GELU_TANH:
        gl = 0.5 * y * (1 + torch.tanh(math.sqrt(2 / math.pi) * (y + 0.044715 * y ** 3)))
        ref = r16(gl)
        return ref, round_diff(ref, 1.13 * dy + 2.0 ** -18 * gl.abs())
    assert epi == N.EPI_BIAS_GATE_RES
    g, r = gate.double(), res.double()
    gy = r16(g * y)
    dgy = round_diff(gy, g.abs() * dy)
    ref = r16(r + gy)
    return ref, round_diff(ref, dgy + 2.0 ** -24 * (r + gy).abs())


def ln_modulate_ref(x, shift, scale):
    """float64 modulate(LayerNorm(x), shift, scale) of bf16 rows x [M, 1024] (dit.py:19-27).  The factor
    bf16(1 + bf16(scale + 1e-6)) is made of bf16 tensor ops in the reference, so it is computed as they are: an fp32 op,
    then rounding to bf16.  Kernel (ln_row.cuh): the fp32 mean and sum of squares are fixed trees of depth 10 over 1024
    terms, so the mean is within 2^-20 mean|x| and the variance within 2^-20 relative.  rsqrtf adds 2 ulps, so rstd is
    within 2^-19 relative.  Three more fp32 roundings follow before the bf16 one.  So the pre-rounding value is within
    2^-17 (|z m| + rstd |m| mean|x| + |shift|), where z = (x - mean) rstd."""
    xd = x.double()
    mean = xd.mean(-1, keepdim=True)
    xc = xd - mean
    rstd = 1.0 / torch.sqrt((xc * xc).mean(-1, keepdim=True) + 1e-6)
    m = (1 + (scale.float() + 1e-6).to(torch.bfloat16).float()).to(torch.bfloat16).double()
    zm = xc * rstd * m
    ref = r16(zm + shift.double())
    delta = 2.0 ** -17 * (zm.abs() + rstd * m.abs() * xd.abs().mean(-1, keepdim=True) + shift.double().abs())
    return ref, round_diff(ref, delta)


def rot_table(frames=8):
    """(cos, sin) [frames][32] of the temporal rotary embedding (theta 1e4, window-relative frame index)."""
    base = 1.0 / (10000 ** (torch.arange(0, 64, 2, dtype=torch.float64) / 64))
    ang = torch.arange(frames, dtype=torch.float64)[:, None] * base[None]
    return torch.stack([ang.cos(), ang.sin()], dim=-1).float().contiguous().cuda()


def rotate_rn(x, rot):
    """The kernels' rotation of x [B, T, P, H, 64] (bf16 values) at window positions 0..T-1.  Per pair this is two fp32
    products and an fp32 sum, each rounded to nearest (the reference's fp32 t * cos + rotate_half(t) * sin), then one
    rounding to bf16.  torch's separate fp32 elementwise ops round at the same places, so q and k come out exactly as the
    kernels have them."""
    T = x.shape[1]
    c, s = rot[:T, :, 0].view(1, T, 1, 1, 32), rot[:T, :, 1].view(1, T, 1, 1, 32)
    x0, x1 = x[..., 0::2].float(), x[..., 1::2].float()
    y = torch.stack((x0 * c - x1 * s, x1 * c + x0 * s), dim=-1).flatten(-2)
    return y.to(torch.bfloat16).float()


def temporal_ref(q, k, v, rot):
    """float64 causal attention over the frames of q, k, v [B, T, P, H, 64] (bf16 values): reference and bound for every
    frame's output, [B, T, P, H, 64].
    Scores: fp32 dot product of 64 terms (a product, an fma, 5 shuffle additions), so within 2^-21 sum|q k| / 8 = es.
    Probabilities before rounding: exp(s - max) uses two scores, __expf adds 2^-21 plus |s - max| 2^-24 (at most 2^-17 here),
    then the fp32 sum of at most 8 terms and a correctly rounded reciprocal.  So the relative error is at most
    eps = 4 max(es) + 2^-15, and the bf16 p is off by at most round_diff(p_ref, eps p).
    Output: fp32 fma chain of at most 8 terms (2^-20 sum p|v|) plus the p errors times |v|, then the final bf16 rounding."""
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
    tol = round_diff(ref, dp @ va + 2.0 ** -20 * (p @ va))
    return ref.permute(0, 3, 1, 2, 4), tol.permute(0, 3, 1, 2, 4)


def temporal_inputs(B, T, kind, seed):
    """q, k, v [B, T, P, H, 64] (bf16 values).  Kinds:
    random:  N(0, 1);
    far:     q and k scaled so that the logits q.k / 8 have a spread of +-30 (nearly one-hot softmax);
    uniform: every key is zero, so all scores are equal and the softmax is uniform over the frames;
    pairs:   q and k non-zero in rotary pairs 0 and 5 only, and k is q with the pair's features swapped (pair 0) or the second
             one negated (pair 5).  q . R(t_k - t_q) k then has a term in sin(t_k - t_q), so a rotation with the wrong
             sign or of the wrong pair changes every score.  With k = q that term would vanish."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    shape = (B, T, P, H, 64)
    q, k, v = (torch.randn(shape, device="cuda", generator=g) for _ in range(3))
    if kind == "far":
        q, k = q * math.sqrt(30), k * math.sqrt(30)
    elif kind == "uniform":
        k.zero_()
    elif kind == "pairs":
        u = 4 * torch.randn((B, 1, P, H, 4), device="cuda", generator=g).expand(B, T, P, H, 4)
        q.zero_()
        k.zero_()
        q[..., 0:2], q[..., 10:12] = u[..., 0:2], u[..., 2:4]
        k[..., 0], k[..., 1] = u[..., 1], u[..., 0]
        k[..., 10], k[..., 11] = u[..., 2], -u[..., 3]
    elif kind != "random":
        raise ValueError(kind)
    return tuple(z.to(torch.bfloat16).float() for z in (q, k, v))


def kv_cache_of(k, v, rot):
    """The K/V cache of frames 0..T-1 as the context pass writes it: rotated K (bf16) | V per row, rows (b, t, pos)."""
    B, T = k.shape[:2]
    kr = rotate_rn(k, rot).reshape(B, T, P, D)
    return torch.stack([kr, v.reshape(B, T, P, D)], dim=3).to(torch.bfloat16).reshape(B * T * P, 2 * D).contiguous()


def to_rows(x):
    """[B, T, P, H, 64] -> [B*T*P, H*64] rows ordered (b, t, pos)."""
    return x.reshape(-1, D)


# ------------------------------------------------------------------------------------------ launches
def workspace(lib, M):
    return torch.zeros(lib.gtav_gemm_skinny_workspace_bytes(M), dtype=torch.uint8, device="cuda")


def counters():
    return torch.zeros(512, dtype=torch.int32, device="cuda")


def skinny(lib, A, W, epi, out, splits, ws, cnt=None, parity=-1, bias=None, res=None, gate=None, frame_row=None):
    """gtav_gemm_skinny_bf16 (parity -1, counter rendezvous) or gtav_gemm_skinny_tagged_bf16; gate: a view into the
    modulation table (row stride MOD_LD)."""
    N = _N()
    M, K = A.shape
    args = (A.data_ptr(), K, W.data_ptr(), K, out.data_ptr(), out.stride(0), M, W.shape[0], K, epi, N.ptr(bias), N.ptr(res),
            0 if res is None else res.stride(0), N.ptr(gate), MOD_LD, N.ptr(frame_row), P, splits, ws.data_ptr())
    if parity < 0:
        N.check(lib.gtav_gemm_skinny_bf16(*args, cnt.data_ptr(), N.current_stream()), "gemm_skinny")
    else:
        N.check(lib.gtav_gemm_skinny_tagged_bf16(*args, parity, N.current_stream()), "gemm_skinny_tagged")
    return out


def skinny_fused(lib, mode, A, W, out, splits, ws, cnt=None, parity=-1, bias=None, res=None, gate=None, frame_row=None,
                 ln_out=None, mod=None, shift_off=0, scale_off=0, cache=None, rot=None, ctx=0):
    N = _N()
    M, K = A.shape
    N.check(lib.gtav_gemm_skinny_fused_bf16(
        A.data_ptr(), K, W.data_ptr(), K, out.data_ptr(), out.stride(0), M, W.shape[0], K, N.ptr(bias), N.ptr(res),
        0 if res is None else res.stride(0), N.ptr(gate), MOD_LD, N.ptr(frame_row), splits, ws.data_ptr(), N.ptr(cnt), mode,
        N.ptr(ln_out), N.ptr(mod), MOD_LD, shift_off, scale_off, N.ptr(cache), N.ptr(rot), ctx, P, parity,
        N.current_stream()), "gemm_skinny_fused")
    return out


def ln_modulate(lib, x, mod, shift_off, scale_off, frame_row):
    N = _N()
    out = torch.empty_like(x)
    N.check(lib.gtav_ln_modulate(x.data_ptr(), out.data_ptr(), x.shape[0], D, mod.data_ptr(), MOD_LD, shift_off, scale_off,
                                 N.ptr(frame_row), P, N.current_stream()), "ln_modulate")
    return out


def attention_last(lib, qkv, ctx, rot, cache):
    N = _N()
    out = torch.empty((qkv.shape[0], D), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_temporal_last(qkv.data_ptr(), out.data_ptr(), qkv.shape[0] // P, ctx, P, H, rot.data_ptr(),
                                             N.ptr(cache), N.current_stream()), "attention_temporal_last")
    return out


# ------------------------------------------------------------------------------------------ (a) fused LayerNorm
class LnCase:
    """Modulation table of the 16-block DiT and the engine's offsets.  For K = 1024 the offsets are to_out's of half 7:
    gate_msa, then shift_mlp / scale_mlp.  For K = 4096 they are fc2's of the last half: gate_mlp, then the final layer's
    shift / scale in the last 2048 columns of the row.  frame_row is non-identity and every frame has its own rows.  A few
    scales are exactly 0, where bf16(0 + 1e-6) survives as in test_ln_modulate."""

    def __init__(self, g, M, K):
        self.mod = (torch.randn((5, MOD_LD), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
        half = 7 if K == 1024 else 31
        if K == 1024:
            self.gate_off, self.shift_off, self.scale_off = half * 6 * D + 2 * D, half * 6 * D + 3 * D, half * 6 * D + 4 * D
        else:
            self.gate_off, self.shift_off, self.scale_off = half * 6 * D + 5 * D, (half + 1) * 6 * D, (half + 1) * 6 * D + D
        rows = [3, 0, 4][: M // P] if M > P else [2]
        self.frame_row = torch.tensor(rows, dtype=torch.int32, device="cuda")
        self.mod[rows[0], self.scale_off:self.scale_off + 8] = 0.0
        self.mod[rows[-1], self.scale_off + 1000:self.scale_off + 1008] = 0.0
        self.gate = self.mod[:, self.gate_off:]
        fr = self.frame_row.long().repeat_interleave(P)
        self.gate_rows = self.mod[fr, self.gate_off:self.gate_off + D]
        self.shift_rows = self.mod[fr, self.shift_off:self.shift_off + D]
        self.scale_rows = self.mod[fr, self.scale_off:self.scale_off + D]

    def fused(self, lib, A, W, bias, h, ln_out, S, ws, cnt=None, parity=-1):
        return skinny_fused(lib, LN, A, W, h, S, ws, cnt, parity, bias=bias, res=h, gate=self.gate, frame_row=self.frame_row,
                            ln_out=ln_out, mod=self.mod, shift_off=self.shift_off, scale_off=self.scale_off)

    def two_kernels(self, lib, A, W, bias, h, S, ws, cnt=None, parity=-1):
        N = _N()
        skinny(lib, A, W, N.EPI_BIAS_GATE_RES, h, S, ws, cnt, parity, bias=bias, res=h, gate=self.gate, frame_row=self.frame_row)
        return ln_modulate(lib, h, self.mod, self.shift_off, self.scale_off, self.frame_row)

    def check_ref(self, A, W, bias, res, h, ln_out, S, what):
        acc, E = linear_ref(A, W, bias, S)
        ref, tol = epilogue_ref(acc, E, _N().EPI_BIAS_GATE_RES, self.gate_rows, res)
        assert_within(h, ref, tol, f"{what}: new residual")
        # LayerNorm of the row the kernel wrote: the one-ulp freedom of that row allowed above is not carried through
        ref, tol = ln_modulate_ref(h, self.shift_rows, self.scale_rows)
        assert_within(ln_out, ref, tol, f"{what}: LayerNorm + modulate")


@pytest.mark.parametrize("M,K,S", [
    (144, 1024, 4), (144, 4096, 16),      # the engine's to_out and fc2 at B = 1
    (144, 1024, 8),                       # explicit split override
    (288, 1024, 16), (432, 1024, 16),     # more token rows than CTAs: the reduce's token loop and next-token preload run
])
def test_fused_layernorm(lib, M, K, S):
    """SK_FUSE_LN with the residual updated in place (res == out, as in the engine): the new residual and the LayerNorm +
    modulate output against float64, and bit for bit against the skinny GATE_RES launch followed by gtav_ln_modulate."""
    g = torch.Generator(device="cuda").manual_seed(M + K + S)
    A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
    W = (torch.randn((D, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
    bias = (torch.randn((D,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    res = torch.randn((M, D), device="cuda", generator=g).to(torch.bfloat16)
    c = LnCase(g, M, K)
    h, ln_out = res.clone(), torch.full((M, D), float("nan"), dtype=torch.bfloat16, device="cuda")
    c.fused(lib, A, W, bias, h, ln_out, S, workspace(lib, M), counters())
    c.check_ref(A, W, bias, res, h, ln_out, S, f"fused LN M={M} K={K} S={S}")
    h2 = res.clone()
    ln2 = c.two_kernels(lib, A, W, bias, h2, S, workspace(lib, M), counters())
    assert torch.equal(h, h2), "fused LN: residual differs from the GATE_RES launch"
    assert torch.equal(ln_out, ln2), "fused LN: LayerNorm output differs from gtav_ln_modulate"


# ------------------------------------------------------------------------------------------ (b) fused temporal attention
ADVERSARIAL = [("far", 8), ("uniform", 7), ("pairs", 6)]          # (kind, frames in the window)


class TattnCase:
    """to_qkv of a temporal half (M = 144, N = 3072, K = 1024) on one rollout with ctx cached frames.  For the random kind
    the q|k|v row is the product of random A and W.  For the adversarial kinds A holds one-hot rows, so the GEMM passes W's
    columns through exactly and q|k|v is the constructed row."""

    def __init__(self, ctx, kind, seed):
        self.ctx, self.rot = ctx, rot_table(8)
        q, k, v = temporal_inputs(1, ctx + 1, kind, seed)
        self.ctx_qkv = (q[:, :ctx], k[:, :ctx], v[:, :ctx])
        self.cache = kv_cache_of(k[:, :ctx], v[:, :ctx], self.rot) if ctx > 0 else None
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        if kind == "random":
            self.A = torch.randn((P, D), device="cuda", generator=g).to(torch.bfloat16)
            self.W = (torch.randn((3 * D, D), device="cuda", generator=g) / 32).to(torch.bfloat16)
        else:
            self.A = torch.eye(P, D, device="cuda").to(torch.bfloat16)
            row = torch.cat([to_rows(z[:, ctx]) for z in (q, k, v)], dim=1)             # [P, 3D]
            self.W = torch.zeros((3 * D, D), device="cuda")
            self.W[:, :P] = row.t()
            self.W = self.W.to(torch.bfloat16)

    def new_operands(self, g):
        self.A = torch.randn((P, D), device="cuda", generator=g).to(torch.bfloat16)
        self.W = (torch.randn((3 * D, D), device="cuda", generator=g) / 32).to(torch.bfloat16)

    def fused(self, lib, ws, cnt=None, parity=-1):
        out = torch.full((P, D), float("nan"), dtype=torch.bfloat16, device="cuda")
        return skinny_fused(lib, TATTN, self.A, self.W, out, 4, ws, cnt, parity, cache=self.cache, rot=self.rot, ctx=self.ctx)

    def qkv(self, lib, ws, cnt=None, parity=-1):
        out = torch.empty((P, 3 * D), dtype=torch.bfloat16, device="cuda")
        return skinny(lib, self.A, self.W, _N().EPI_STORE, out, 4, ws, cnt, parity)

    def check_ref(self, qkv, out, what):
        acc, E = linear_ref(self.A, self.W, None, 4)
        ref, tol = epilogue_ref(acc, E, _N().EPI_STORE)
        assert_within(qkv, ref, tol, f"{what}: q|k|v")
        # attention of the q|k|v row the GEMM produced (bit-equal to the one inside the fused reduce), checked above
        last = [z.float().view(1, 1, P, H, 64) for z in qkv.split(D, dim=1)]
        q, k, v = (torch.cat([c, l], dim=1) for c, l in zip(self.ctx_qkv, last))
        ref, tol = temporal_ref(q, k, v, self.rot)
        assert_within(out, to_rows(ref[:, -1]), to_rows(tol[:, -1]), f"{what}: attention")


@pytest.mark.parametrize("ctx,kind", [(c, "random") for c in range(8)] + [(t - 1, kind) for kind, t in ADVERSARIAL])
def test_fused_temporal_attention(lib, ctx, kind):
    """SK_FUSE_TATTN at every cached window length 0..7 (rotary table of 8 rows, cache rebuilt by hand): the attention
    output against float64, and bit for bit against the skinny STORE launch followed by gtav_attention_temporal_last."""
    c = TattnCase(ctx, kind, 300 + 10 * ctx + len(kind))
    out = c.fused(lib, workspace(lib, P), counters())
    qkv = c.qkv(lib, workspace(lib, P), counters())
    c.check_ref(qkv, out, f"fused attention ctx={ctx} {kind}")
    assert torch.equal(out, attention_last(lib, qkv, ctx, c.rot, c.cache)), "fused attention differs from the two-kernel path"


# ------------------------------------------------------------------------------------------ (c) tagged exchange
TAGGED = [
    # (what, M, N, K, splits): each last-frame GEMM of the engine with the epilogue it runs there
    ("STORE", 144, 3 * D, D, 4),          # to_qkv, spatial half
    ("GATE_RES", 144, D, D, 4),           # to_out (unfused), in place
    ("GELU_TANH", 144, 4 * D, D, 4),      # fc1
    ("GATE_RES", 144, D, 4 * D, 16),      # fc2 (unfused), in place
    ("GATE_RES", 288, D, D, 16),          # to_out at B = 2
    ("GATE_RES", 432, D, D, 16),          # to_out at B = 3
    ("LN", 144, D, D, 4),                 # to_out + LayerNorm
    ("LN", 144, D, 4 * D, 16),            # fc2 + LayerNorm
    ("LN", 432, D, D, 16),                # to_out + LayerNorm at B = 3: token loop
    ("TATTN", 144, 3 * D, D, 4),          # temporal to_qkv + attention, 4 cached frames
]


@pytest.mark.parametrize("what,M,Nn,K,S", TAGGED)
def test_tagged_exchange_launch_sequence(lib, what, M, Nn, K, S):
    """Six consecutive tagged launches on one zeroed workspace with parity 1, 0, 1, 0, ... and new A, W and residual every
    time: a stale partial sum accepted by mistake would then give a wrong result instead of the same one.  Every launch
    against float64, and against the counter-rendezvous launch up to the tag's last-bit difference.  The fused modes are also
    compared bit for bit with the tagged two-kernel path, which runs on a workspace of its own."""
    N = _N()
    g = torch.Generator(device="cuda").manual_seed(M + Nn + K + S + len(what))
    ws_t, ws_u, ws_c, cnt = workspace(lib, M), workspace(lib, M), workspace(lib, M), counters()
    epi = {"STORE": N.EPI_STORE, "GATE_RES": N.EPI_BIAS_GATE_RES, "GELU_TANH": N.EPI_BIAS_GELU_TANH}.get(what)
    bias = None if what in ("STORE", "TATTN") else (torch.randn((Nn,), device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    ln = LnCase(g, M, K) if what in ("GATE_RES", "LN") else None
    ta = TattnCase(4, "random", 77) if what == "TATTN" else None
    for launch in range(6):
        parity = (launch & 1) ^ 1
        tag = f"{what} M={M} N={Nn} K={K} S={S} launch {launch}"
        A = torch.randn((M, K), device="cuda", generator=g).to(torch.bfloat16)
        W = (torch.randn((Nn, K), device="cuda", generator=g) / math.sqrt(K)).to(torch.bfloat16)
        res = torch.randn((M, Nn), device="cuda", generator=g).to(torch.bfloat16)
        if what == "LN":
            h_t, h_c, h_u = res.clone(), res.clone(), res.clone()
            ln_t, ln_c = (torch.full((M, D), float("nan"), dtype=torch.bfloat16, device="cuda") for _ in range(2))
            ln.fused(lib, A, W, bias, h_t, ln_t, S, ws_t, parity=parity)
            ln.fused(lib, A, W, bias, h_c, ln_c, S, ws_c, cnt)
            ln_u = ln.two_kernels(lib, A, W, bias, h_u, S, ws_u, parity=parity)
            assert torch.equal(h_t, h_u) and torch.equal(ln_t, ln_u), f"{tag}: fused differs from the two-kernel path"
            ln.check_ref(A, W, bias, res, h_t, ln_t, S, tag)
            assert_last_bit_close(h_t, h_c, tag)
            assert_last_bit_close(ln_t, ln_c, tag)
        elif what == "TATTN":
            ta.A, ta.W = A, W
            out_t, out_c = ta.fused(lib, ws_t, parity=parity), ta.fused(lib, ws_c, cnt)
            qkv = ta.qkv(lib, ws_u, parity=parity)
            assert torch.equal(out_t, attention_last(lib, qkv, ta.ctx, ta.rot, ta.cache)), f"{tag}: fused differs from the two-kernel path"
            ta.check_ref(qkv, out_t, tag)
            assert_last_bit_close(out_t, out_c, tag)
        else:
            gated = epi == N.EPI_BIAS_GATE_RES
            kw = dict(bias=bias, gate=ln.gate if gated else None, frame_row=ln.frame_row if gated else None)
            out_t = res.clone() if gated else torch.zeros((M, Nn), dtype=torch.bfloat16, device="cuda")
            out_c = out_t.clone()
            skinny(lib, A, W, epi, out_t, S, ws_t, parity=parity, res=out_t if gated else None, **kw)
            skinny(lib, A, W, epi, out_c, S, ws_c, cnt, res=out_c if gated else None, **kw)
            acc, E = linear_ref(A, W, bias, S)
            ref, tol = epilogue_ref(acc, E, epi, ln.gate_rows if gated else None, res)
            assert_within(out_t, ref, tol, tag)
            assert_last_bit_close(out_t, out_c, tag)


# ------------------------------------------------------------------------------------------ (d) temporal attention
def dense_attention(lib, q, k, v, rot):
    N = _N()
    B, T = q.shape[:2]
    qkv = torch.cat([to_rows(z) for z in (q, k, v)], dim=1).to(torch.bfloat16).contiguous()
    out = torch.full((B * T * P, D), float("nan"), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_temporal(qkv.data_ptr(), out.data_ptr(), B, T, P, H, rot.data_ptr(), N.current_stream()), "dense")
    return qkv, out


WINDOWS = [(T, B, "random") for T in range(1, 9) for B in (1, 3)] + [(T, 1, kind) for kind, T in ADVERSARIAL]


@pytest.mark.parametrize("T,B,kind", WINDOWS)
def test_temporal_attention_every_window(lib, T, B, kind):
    """gtav_attention_temporal at T = 1..8 frames against float64 with the kernel's rounding points."""
    rot = rot_table(8)
    q, k, v = temporal_inputs(B, T, kind, 500 + 10 * T + B)
    _, out = dense_attention(lib, q, k, v, rot)
    ref, tol = temporal_ref(q, k, v, rot)
    assert_within(out, to_rows(ref), to_rows(tol), f"dense temporal attention T={T} B={B} {kind}")


@pytest.mark.parametrize("T,B,kind", WINDOWS)
def test_temporal_attention_last_equals_dense_every_window(lib, T, B, kind):
    """gtav_attention_temporal_last with ctx_frames = T - 1 = 0..7 against the cache the context pass would write: the same
    bits as row T - 1 of the dense kernel (attn_temporal.cu promises the same arithmetic in the same order)."""
    rot = rot_table(8)
    q, k, v = temporal_inputs(B, T, kind, 700 + 10 * T + B)
    qkv, dense = dense_attention(lib, q, k, v, rot)
    last_qkv = qkv.view(B, T, P, 3 * D)[:, T - 1].reshape(B * P, 3 * D).contiguous()
    cache = kv_cache_of(k[:, : T - 1], v[:, : T - 1], rot) if T > 1 else None
    out = attention_last(lib, last_qkv, T - 1, rot, cache)
    ref = dense.view(B, T, P, D)[:, T - 1].reshape(B * P, D)
    assert torch.equal(out, ref), f"last-frame kernel differs from the dense kernel's last row: max-abs {float((out.float() - ref.float()).abs().max())}"
