"""float64 model of bf16 rounding, shared by the kernel parity tests: a kernel's bf16 result is compared with a float64
reference that rounds where the kernel rounds, within a per-element bound derived from the fp32 error between two
rounding points."""
import torch


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
