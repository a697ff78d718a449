"""Kernel-level parity of the non-causal rotary attention behind gtav_attention_seq (DiT spatial attention at S = 144, VAE
attention at S = 576) on every kernel it dispatches to:
  attn_seq144_kernel           S = 144, groups * heads * 3 <= 296 (rotary table staged in shared memory)
  attn_seq_kernel<144,144,...> S = 144, larger launches below 96 groups (or GTAV_ATTN=mma)
  attn_tc_kernel<144,...>      S = 144, groups >= 96 (or GTAV_ATTN=tc): one 144-key block, query tiles 0..127, 128..143
  attn_seq_kernel<576,64,...>  S = 576, groups < 4 (or GTAV_ATTN=mma): nine key blocks of 64, running maximum
  attn_tc_kernel<576,...>      S = 576, groups >= 4 (or GTAV_ATTN=tc): four key blocks of 144, lazy rescale, three softmax
                               groups whose partial row sums meet in the epilogue, ragged query tile 512..575

The kernels' rounding points:
1. q and k are rotated pair by pair (pairs < rot_pairs only) with two fp32 products and an fp32 sum, each rounded to
   nearest, then rounded to bf16 - the reference's t * cos + rotate_half(t) * sin.  `rotate` computes this with torch fp32
   elementwise ops, which round at the same places, so the reference has the kernels' q and k bit for bit.
2. Scores are fp32 tensor-core sums of 64 exact bf16 products.
3. p~ = 2^((s - m) log2(e) / 8) relative to a per-row reference maximum m: the running maximum of the key blocks so far
   (mma.sync), or the lazily updated maximum (tcgen05, which keeps the previous maximum unless a block exceeds it by more
   than 2^8, so p~ can reach 2^8).  p~ is rounded to bf16 before P V; the row sum l is taken over the unrounded p~.
4. O is an fp32 tensor-core accumulation of bf16(p~) v.
5. out = bf16(O * (1 / l)).

The reference is o = sum_j p_j v_j in float64, p the float64 softmax of the float64 scores of the rotated q and k (`spatial_ref`
derives the bound).  Whatever m is, rounding p~ to bf16 moves a term by at most 2^-8 relative, and every other error is an
fp32 one, so the bound does not need to emulate the lazy schedule.  It comes to about one bf16 ulp of sum p |v|, where the
absolute bound of test_kernels_gpu.py allows 2e-2 (about 40 ulps of a typical output).  A biased rounding can still hide
inside it, so the random cases also bound the mean signed error (`assert_unbiased`).
"""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest
import torch

from parity64 import assert_within, r16, round_diff

gpu = pytest.mark.gpu
HD = 64                      # head dim
FLAT = 20                    # at S = 144 every dim is rotated: the controlled kinds turn rotary pair 20 (dims 40, 41) off
GUARD = 128                  # guard rows on either side of the output (the tcgen05 query tile of S = 144 spans 256 rows)
# Bound on the mean signed error of a random case, in units of the per-element bound (assert_unbiased).  On a B200 (1000 W
# power limit) the 40 random cases measured |mean| <= 4.5e-4; probabilities truncated to bf16 instead of rounded give
# several times this limit.
BIAS_MAX = 0.005


@pytest.fixture(scope="module")
def lib():
    import gtav_b200._native as N
    return N.load()


def _N():
    import gtav_b200._native as N
    return N


def pairs_of(seq):
    return {144: 32, 576: 16}[seq]


# ------------------------------------------------------------------------------------------ rotary tables, (cos, sin) [S, pairs, 2]
def random_table(seq, g):
    ang = torch.rand((seq, pairs_of(seq)), device="cuda", generator=g) * 20 - 10
    return torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()


def model_table(seq):
    """The models' own tables, rebuilt with the expressions of model/dit.py (spatial, 9 x 16 tokens, 16 row + 16 column
    pairs) and model/vae.py (18 x 32 tokens, 8 row + 8 column pairs, head dims 32..63 not rotated)."""
    if seq == 144:
        from oracle.weights import DiTConfig, spatial_rotary_base
        base, gh, gw = spatial_rotary_base(DiTConfig()).to(device="cuda", dtype=torch.float32), 9, 16
    else:
        base, gh, gw = (torch.linspace(1.0, 576 / 2, 8) * math.pi).to("cuda"), 18, 32
    ah = torch.linspace(-1, 1, steps=gh, device="cuda")[:, None] * base[None]
    aw = torch.linspace(-1, 1, steps=gw, device="cuda")[:, None] * base[None]
    ang = torch.cat([ah[:, None].expand(gh, gw, -1), aw[None].expand(gh, gw, -1)], dim=-1).reshape(gh * gw, -1)
    assert ang.shape[1] == pairs_of(seq)
    return torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous()


def rotate(x, tab):
    """The kernels' rotation of x [..., S, 64] (bf16 values, fp32) by tab [S, pairs, 2]: rounding point 1."""
    n = tab.shape[1]
    c, s = tab[:, :, 0], tab[:, :, 1]
    x0, x1 = x[..., 0:2 * n:2], x[..., 1:2 * n:2]
    y = torch.stack((x0 * c - x1 * s, x1 * c + x0 * s), dim=-1).flatten(-2)
    return torch.cat([y.to(torch.bfloat16).float(), x[..., 2 * n:]], dim=-1)


# ------------------------------------------------------------------------------------------ reference and bound
def key_blocks(seq, tc):
    return 1 if seq == 144 else (4 if tc else 9)


def spatial_ref(q, k, v, tab, nb):
    """float64 attention of q, k, v [G, H, S, 64] (bf16 values) with the rotation of `tab`, and the per-element bound of a
    kernel with nb key blocks.  Relative errors of p~ against exp((s - m) / 8) for the exact scores s of the rotated q, k:
      score: fp32 tensor-core sum of 64 exact products in 4 steps of 16, each step off by at most 2^-23 of the running
             sum of |q k| and twice that for the step's own sum: 2^-19 sum|q k| / 8 = es in natural-log units;
      exponent: s log2(e) / 8 - m log2(e) / 8 in fp32 (three roundings of values up to L log2(e), L = max |s| / 8 of the
             row, and the rounded constant) costs 4 L 2^-24; ex2.approx / exp2f 2^-21.  The block-to-block rescale factors
             of O and l (and, tcgen05, the factors that bring the groups' partial row sums to one maximum) are such
             exponentials too, at most nb + 1 of them on any term: eps = max es + (nb + 1)(2^-21 + 4 L 2^-24).
    Row sum l: fp32 sum of S positive terms, eps_l = S 2^-24.  O: fp32 tensor-core sum over S / 16 steps, up to nb
    rescales and the final O * (1 / l): acc = 2^-22 (S / 16 + 2 nb + 2) relative to sum p |v|.
    With p~_j = e_j (1 + eta_j), |eta_j| <= eps, and bf16(p~_j) = p~_j (1 + rho_j), |rho_j| <= 2^-8:
      |O / l - o| <= sum p |v| (2^-8 + eps + acc) + |o| (eps + eps_l), to first order (the factor 1.01 covers the rest),
    plus 2^-110 for probabilities that ex2.approx.ftz flushes to zero; then one bf16 rounding (round_diff)."""
    S = q.shape[-2]
    qr, kr = (rotate(z, tab).double() for z in (q, k))
    vv = v.double()
    s = qr @ kr.transpose(-1, -2) / 8
    es = 2.0 ** -19 * (qr.abs() @ kr.abs().transpose(-1, -2)) / 8
    L = s.abs().amax(-1, keepdim=True)
    e = torch.exp(s - s.amax(-1, keepdim=True))
    p = e / e.sum(-1, keepdim=True)
    o = p @ vv
    pv = p @ vv.abs()
    eps = es.amax(-1, keepdim=True) + (nb + 1) * (2.0 ** -21 + 4 * L * 2.0 ** -24)
    acc = 2.0 ** -22 * (S / 16 + 2 * nb + 2)
    delta = 1.01 * (pv * (2.0 ** -8 + eps + acc) + o.abs() * (eps + S * 2.0 ** -24)) + 2.0 ** -110
    ref = r16(o)
    return ref, round_diff(ref, delta)


def assert_unbiased(out, ref, tol, what):
    """Mean of (out - ref) sign(ref) / tol.  An error that shrinks (or grows) every probability, such as p truncated to bf16,
    moves each output towards zero (away from it) by a fixed fraction, so it shows here with the sign of the reference; an
    unsigned mean would cancel over outputs of both signs.  Rounding to nearest leaves it near zero."""
    nz = ref != 0
    bias = float(((out.double() - ref) * ref.sign() / tol)[nz].mean())
    assert abs(bias) < BIAS_MAX, f"{what}: mean signed error {bias:+.4f} of the bound (limit {BIAS_MAX})"
    return bias


# ------------------------------------------------------------------------------------------ inputs
LEVELS_4 = {0: [0.0, 5.3125, 11.125, 31.125], 1: [31.125, 11.125, 5.3125, 0.0]}      # per quarter of the keys
LEVELS_9 = [0.0, 5.3125, 11.125, 31.125, 10.0, 15.3125, 21.125, 0.0, 20.0]           # per ninth of the keys


def key_levels(seq, heads):
    """[heads, S] logit levels of the keys for the `blocks` kind, chosen by head: block maxima that rise by 5.3125 (below
    the lazy threshold 8 ln 2 = 5.545 of the tcgen05 kernel), by 5.8125 (above it), by 20, and fall.  Pattern 0 / 1 steps
    at the quarters (key blocks of 144 at S = 576), pattern 2 at the ninths (key blocks of 64), pattern 3 is flat."""
    lv = torch.zeros((heads, seq))
    pos = torch.arange(seq)
    for h in range(heads):
        pat = h % 4
        if pat < 2:
            lv[h] = torch.tensor(LEVELS_4[pat])[pos // (seq // 4)]
        elif pat == 2:
            lv[h] = torch.tensor(LEVELS_9)[pos // (seq // 9)]
    return lv.to("cuda")


def make_inputs(seq, groups, heads, kind, seed):
    """q, k, v [G, H, S, 64] (bf16 values, fp32) and the rotary table.  Where a logit is controlled it lives in a dim the
    table leaves alone: dim 40 (unrotated at S = 576, rotary pair FLAT set to angle 0 at S = 144).  Kinds:
      random / random-model: N(0, 1), random angles in [-10, 10] / the model's table;
      far:     logits spread +-30, so the softmax is nearly one-hot;
      uniform: every key is zero, so p~ = 1 exactly and the output is the mean of v;
      blocks:  small noise plus q[40] k[40] / 8 = a key_levels(head)[key], a = 1, -1 or 1/2 by query row, so that the
               block maxima of some rows rise by the amounts of key_levels and of others fall (the ragged query tiles
               512..575 and 128..143 included);
      pairs:   q and k non-zero in the first and the last rotary pair only (and, S = 576, in tail pair 16, which must not
               rotate), the same for every position, with k the swapped (pair 0, 16) or sign-flipped (last pair) copy of q.
               A score is then q . R(angle_k - angle_q) k, and a rotation of the wrong pair, by the wrong sign or at the
               wrong position changes it."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    shape = (groups, heads, seq, HD)
    q, k, v = (torch.randn(shape, device="cuda", generator=g) for _ in range(3))
    tab = model_table(seq) if kind in ("random-model", "uniform", "blocks") else random_table(seq, g)
    if kind == "far":
        q, k = q * math.sqrt(30), k * math.sqrt(30)
    elif kind == "uniform":
        k.zero_()
    elif kind == "blocks":
        q, k = q * 0.25, k * 0.25
        a = torch.tensor([8.0, -8.0, 4.0], device="cuda")[torch.arange(seq, device="cuda") % 3]
        q[..., 40] = a
        k[..., 40] = key_levels(seq, heads)[None]
    elif kind == "pairs":
        last = pairs_of(seq) - 1
        u = 4 * torch.randn((groups, heads, 1, 6), device="cuda", generator=g).expand(groups, heads, seq, 6)
        q.zero_()
        k.zero_()
        q[..., 0:2], q[..., 2 * last:2 * last + 2] = u[..., 0:2], u[..., 2:4]
        k[..., 0], k[..., 1] = u[..., 1], u[..., 0]
        k[..., 2 * last], k[..., 2 * last + 1] = u[..., 2], -u[..., 3]
        if seq == 576:
            q[..., 32:34] = u[..., 4:6]
            k[..., 32], k[..., 33] = u[..., 5], u[..., 4]
    elif kind not in ("random", "random-model"):
        raise ValueError(kind)
    if seq == 144 and kind in ("blocks", "uniform"):
        tab = tab.clone()
        tab[:, FLAT, 0], tab[:, FLAT, 1] = 1.0, 0.0
    return (*(z.to(torch.bfloat16).float() for z in (q, k, v)), tab)


def pack_qkv(q, k, v):
    """[G, H, S, 64] x 3 -> qkv rows [G * S, 3 * H * 64] (q | k | v, head-major inside each)."""
    G, H, S, _ = q.shape
    return torch.cat([z.permute(0, 2, 1, 3).reshape(G * S, H * HD) for z in (q, k, v)], dim=1).to(torch.bfloat16).contiguous()


def unpack_out(out, G, H, S):
    return out.float().view(G, S, H, HD).permute(0, 2, 1, 3)


# ------------------------------------------------------------------------------------------ launch
def attention(lib, qkv, groups, seq, heads, tab):
    """gtav_attention_seq into a NaN-filled view with GUARD rows before and after it, launched twice: the two results must
    be the same bits, the guards untouched and every output finite."""
    N = _N()
    rows, width = groups * seq, heads * HD
    outs = []
    for _ in range(2):
        buf = torch.full((rows + 2 * GUARD, width), float("nan"), dtype=torch.bfloat16, device="cuda")
        nan_bits = buf[:GUARD].view(torch.int16).clone()
        out = buf[GUARD:GUARD + rows]
        N.check(lib.gtav_attention_seq(qkv.data_ptr(), out.data_ptr(), groups, seq, heads, tab.data_ptr(), tab.shape[1],
                                       N.current_stream()), "attention_seq")
        torch.cuda.synchronize()
        assert torch.equal(buf[:GUARD].view(torch.int16), nan_bits), "rows before the output were written"
        assert torch.equal(buf[GUARD + rows:].view(torch.int16), nan_bits), "rows after the output were written"
        assert bool(torch.isfinite(out.float()).all()), f"{int((~torch.isfinite(out.float())).sum())} outputs not written or not finite"
        outs.append(out)
    assert torch.equal(outs[0], outs[1]), "two launches on the same input differ"
    return outs[0]


def set_impl(monkeypatch, impl):
    if impl is None:
        monkeypatch.delenv("GTAV_ATTN", raising=False)
    else:
        monkeypatch.setenv("GTAV_ATTN", impl)


def uses_tc(seq, groups, impl):
    """The dispatch of attn_mma.cu (attn_use_tc)."""
    if impl is not None:
        return impl == "tc"
    return groups >= (4 if seq == 576 else 96)


# ------------------------------------------------------------------------------------------ cases
PATHS = [
    # (seq, GTAV_ATTN or None for the default dispatch, groups, heads)
    (144, None, 1, 16), (144, None, 6, 16),          # attn_seq144_kernel
    (144, None, 7, 16), (144, None, 40, 16),         # attn_seq_kernel<144>
    (144, None, 96, 16), (144, None, 160, 16),       # tcgen05, several waves
    (144, "tc", 1, 16), (144, "tc", 7, 16), (144, "mma", 160, 16),
    (576, None, 1, 16), (576, None, 3, 16),          # attn_seq_kernel<576>
    (576, None, 4, 16), (576, None, 16, 16),         # tcgen05
    (576, "tc", 1, 16), (576, "mma", 16, 16),
    # three heads on every kernel
    (144, None, 2, 3), (144, None, 40, 3), (144, None, 96, 3), (576, None, 2, 3), (576, None, 4, 3),
]
KINDS = ["random", "random-model", "far", "uniform", "blocks", "pairs"]


def path_id(seq, impl, groups, heads):
    return f"S{seq}-{impl or 'default'}-g{groups}-h{heads}"


@gpu
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("seq,impl,groups,heads", PATHS, ids=[path_id(*p) for p in PATHS])
def test_attention_seq_parity(lib, monkeypatch, seq, impl, groups, heads, kind):
    set_impl(monkeypatch, impl)
    seed = 1000 * seq + 10 * groups + heads + 7 * KINDS.index(kind) + (0 if impl is None else 3)
    q, k, v, tab = make_inputs(seq, groups, heads, kind, seed)
    out = attention(lib, pack_qkv(q, k, v), groups, seq, heads, tab)
    ref, tol = spatial_ref(q, k, v, tab, key_blocks(seq, uses_tc(seq, groups, impl)))
    what = f"{path_id(seq, impl, groups, heads)} {kind}"
    out = unpack_out(out, groups, heads, seq)
    assert_within(out, ref, tol, what)
    if kind.startswith("random"):
        assert_unbiased(out, ref, tol, what)


# ------------------------------------------------------------------------------------------ rotation-rounding probe
def _f32(t):
    return t.float().double()


def _two_sum_exact(a, b):
    """a + b is exact in float64 (the TwoSum error term is zero)."""
    s = a + b
    bp = s - a
    return ((a - (s - bp)) + (b - bp)) == 0


@functools.lru_cache(maxsize=None)
def rotation_probe(comp):
    """A bf16 pair (x, y) and an fp32 table entry (c, s) whose rotated component `comp` (0: x c - y s, 1: y c + x s) rounds
    to a different bf16 value when the reference's two rounded products and rounded sum are replaced by either FMA
    contraction, fma(a, b, fp32(c d)) or fma(c, d, fp32(a b)).  Emulated in float64, where the products of a bf16 and an
    fp32 value are exact; candidates whose float64 sums are not exact are rejected.  (x, y) are then scaled by a power of
    two so that the rotated value r lies in [1, 2).  Returns (x, y, c, s, r) as Python floats."""
    g = torch.Generator().manual_seed(20261 + comp)
    n = 1 << 20
    x, y = (torch.randn(n, generator=g).to(torch.bfloat16).double() for _ in range(2))
    ang = torch.rand(n, generator=g, dtype=torch.float64) * 20 - 10
    c, s = _f32(ang.cos()), _f32(ang.sin())
    t1, t2 = (x * c, -(y * s)) if comp == 0 else (y * c, x * s)
    exact = _two_sum_exact(_f32(t1), _f32(t2)) & _two_sum_exact(t1, _f32(t2)) & _two_sum_exact(_f32(t1), t2)
    ref = r16(_f32(_f32(t1) + _f32(t2)))
    fma_a, fma_b = r16(_f32(t1 + _f32(t2))), r16(_f32(_f32(t1) + t2))
    hit = torch.nonzero(exact & (ref != fma_a) & (ref != fma_b) & (ref != 0))
    assert hit.numel() > 0, "no probe candidate found"
    i = int(hit[0])
    scale = 2.0 ** -math.floor(math.log2(abs(float(ref[i]))))
    return float(x[i]) * scale, float(y[i]) * scale, float(c[i]), float(s[i]), float(ref[i]) * scale


def _bf16_of_f32(v):
    return float(torch.tensor(np.float32(v)).to(torch.bfloat16).double())


def test_rotation_probe_property():
    """The search result, checked in exact rational arithmetic: (x, y) are bf16 and (c, s) fp32 values, every sum the
    rotation forms is exact in float64 (so the float64 emulation rounds once, like the fp32 hardware), r is the reference's
    rotation and lies in [1, 2), and both FMA contractions give another bf16 value.  The probe cases rely on this."""
    for comp in (0, 1):
        x, y, c, s, r = rotation_probe(comp)
        assert _bf16_of_f32(x) == x and _bf16_of_f32(y) == y
        assert float(np.float32(c)) == c and float(np.float32(s)) == s
        X, Y, Cc, Ss = (Fraction(z) for z in (x, y, c, s))
        t1, t2 = (X * Cc, -(Y * Ss)) if comp == 0 else (Y * Cc, X * Ss)

        def f32(q):
            assert Fraction(float(q)) == q, "sum not exact in float64"
            return Fraction(float(np.float32(float(q))))
        ref = _bf16_of_f32(float(f32(f32(t1) + f32(t2))))
        fma_a = _bf16_of_f32(float(f32(t1 + f32(t2))))
        fma_b = _bf16_of_f32(float(f32(f32(t1) + t2)))
        assert ref == r and 1.0 <= abs(r) < 2.0
        assert fma_a != ref and fma_b != ref, (comp, ref, fma_a, fma_b)


PROBE_PAIR = 3               # the rotary pair that carries the probe


def probe_inputs(seq, groups, heads, side, comp):
    """Two keys that tie exactly when the probed element is rotated as the reference rotates it; every other key is zero.
    The table is (1, 0) (an exact identity) everywhere except at position a = 5 for PROBE_PAIR, where it is the probe's
    (c, s).  The probed dim d = 2 PROBE_PAIR + comp carries a large query component Q = +-256, so that the two logits are
    32 |r| (32 to 64) and one bf16 ulp of the rotated value (2^-7) moves a logit by 0.25; v = +1 for one key and -1 for the
    other, so the reference output is 0 and an ulp moves it by about 0.12.
      side k: key A at position a holds (x, y) in PROBE_PAIR, key B at position S - 1 holds r in dim d; every query row but a
              holds Q in dim d.
      side q: query row a holds (x, y) in PROBE_PAIR and r in dim d + 2 (the same component of the next pair, rotated by
              the identity); key A at position 1 holds Q in dim d, key B at position S - 1 holds Q in dim d + 2."""
    x, y, c, s, r = rotation_probe(comp)
    a, b, d = 5, seq - 1, 2 * PROBE_PAIR + comp
    Q = math.copysign(256.0, r)
    tab = torch.zeros((seq, pairs_of(seq), 2), device="cuda")
    tab[..., 0] = 1.0
    tab[a, PROBE_PAIR] = torch.tensor([c, s], device="cuda")
    shape = (groups, heads, seq, HD)
    q, k, v = (torch.zeros(shape, device="cuda") for _ in range(3))
    xy = torch.tensor([x, y], device="cuda")
    if side == "k":
        k[..., a, 2 * PROBE_PAIR:2 * PROBE_PAIR + 2] = xy
        k[..., b, d] = r
        q[..., d] = Q
        q[..., a, :] = 0
        ka = a
    else:
        q[..., a, 2 * PROBE_PAIR:2 * PROBE_PAIR + 2] = xy
        q[..., a, d + 2] = r
        ka = 1
        k[..., ka, d] = Q
        k[..., b, d + 2] = Q
    v[..., ka, :], v[..., b, :] = 1.0, -1.0
    return q, k, v, tab


PROBE_PATHS = [(144, None, 1), (144, None, 7), (144, "tc", 1), (576, None, 1), (576, None, 4)]


@gpu
@pytest.mark.parametrize("side,comp", [("k", 0), ("k", 1), ("q", 0), ("q", 1)])
@pytest.mark.parametrize("seq,impl,groups", PROBE_PATHS, ids=[path_id(*p, 16) for p in PROBE_PATHS])
def test_attention_seq_rotation_rounding(lib, monkeypatch, seq, impl, groups, side, comp):
    """The rotation-rounding probe on every kernel: an FMA-contracted rotation moves the probed element by one ulp, which
    breaks the tie of the two keys and puts the output far outside the bound."""
    set_impl(monkeypatch, impl)
    heads = 16
    q, k, v, tab = probe_inputs(seq, groups, heads, side, comp)
    out = attention(lib, pack_qkv(q, k, v), groups, seq, heads, tab)
    ref, tol = spatial_ref(q, k, v, tab, key_blocks(seq, uses_tc(seq, groups, impl)))
    assert_within(unpack_out(out, groups, heads, seq), ref, tol, f"probe {side}[{comp}] {path_id(seq, impl, groups, heads)}")


@gpu
@pytest.mark.parametrize("side,comp", [("k", 0), ("k", 1), ("q", 0), ("q", 1)])
def test_attention_temporal_rotation_rounding(lib, side, comp):
    """The same probe through gtav_attention_temporal (window of T = 3 frames, rows (frame, position), 16 heads), whose
    rotation already rounds like the reference's.  The probe sits at frame 0 (side k) or frame 2 (side q), key A at frame 0
    and key B at frame 1.  Every score is a single exact product, so with a correct rotation the output is exact: v_A = 1
    for frame 0 (its only key), and 0 for frames 1 and 2 (two tied keys, or all scores 0, with v = +1, -1, 0)."""
    N = _N()
    x, y, c, s, r = rotation_probe(comp)
    P, H, T, d = 144, 16, 3, 2 * PROBE_PAIR + comp
    Q = math.copysign(256.0, r)
    fa = 0 if side == "k" else 2                                     # frame whose table entry is the probe's (c, s)
    rot = torch.zeros((8, 32, 2), device="cuda")
    rot[..., 0] = 1.0
    rot[fa, PROBE_PAIR] = torch.tensor([c, s], device="cuda")
    q, k, v = (torch.zeros((T, P, H, HD), device="cuda") for _ in range(3))
    xy = torch.tensor([x, y], device="cuda")
    if side == "k":
        k[0, ..., 2 * PROBE_PAIR:2 * PROBE_PAIR + 2] = xy
        k[1, ..., d] = r
        q[1:, ..., d] = Q
    else:
        q[2, ..., 2 * PROBE_PAIR:2 * PROBE_PAIR + 2] = xy
        q[2, ..., d + 2] = r
        k[0, ..., d] = Q
        k[1, ..., d + 2] = Q
    v[0], v[1] = 1.0, -1.0
    qkv = torch.cat([z.reshape(T * P, H * HD) for z in (q, k, v)], dim=1).to(torch.bfloat16).contiguous()
    out = torch.full((T * P, H * HD), float("nan"), dtype=torch.bfloat16, device="cuda")
    N.check(lib.gtav_attention_temporal(qkv.data_ptr(), out.data_ptr(), 1, T, P, H, rot.data_ptr(), N.current_stream()),
            "attention_temporal")
    expect = torch.zeros((T, P * H * HD), dtype=torch.bfloat16, device="cuda")
    expect[0] = 1.0
    got = out.view(T, P * H * HD)
    assert torch.equal(got, expect), (f"temporal probe {side}[{comp}]: frames 1, 2 max |out| "
                                      f"{float(got[1:].float().abs().max())}, frame 0 off by {float((got[0].float() - 1).abs().max())}")
