"""In-graph per-kernel timing of the last-frame step's kernels at B=1 (144 rows): each kernel family is captured
N times back to back into a CUDA graph (programmatic dependent launch between them, as in the sampler) and the
graph replayed, so the number is GPU time per launch with no host launch cost in it.  GEMM weights rotate over
32 distinct matrices (> L2) so they stream from HBM as in the real step.  Also prints the skinny GEMM's phase
time stamps (GTAV_SKINNY_TRACE) for a few CTAs.

    python scripts/bench_graph.py
"""
import json
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gtav_b200._native as N

lib = N.load()
dev = torch.device("cuda")
D, P, H = 1024, 144, 16
NW = 32


def graph_time(calls, reps=5):
    """calls: list of zero-arg launchers, captured in order into one graph.  Returns us per launch."""
    s = torch.cuda.Stream()
    torch.cuda.synchronize()                     # a plan's workspace must not be used from two streams at once
    with torch.cuda.stream(s):
        for c in calls[: min(len(calls), 8)]:
            c()                                  # first-use configuration outside capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for c in calls:
                c()
        g.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / (reps * len(calls))


def rnd(*shape, scale=1.0):
    return (torch.randn(shape, device=dev) * scale).to(torch.bfloat16)


class Bufs:
    def __init__(self):
        self.h = rnd(P, D)
        self.hn = rnd(P, D)
        self.qkv = rnd(P, 3 * D)
        self.att = rnd(P, D)
        self.mlp = rnd(P, 4 * D)
        self.mod = rnd(4, 6 * D, scale=0.1)
        self.bias = torch.zeros(4 * D, device=dev, dtype=torch.bfloat16)
        self.rot = torch.randn((P, 32, 2), device=dev)
        self.rott = torch.randn((5, 32, 2), device=dev)
        self.cache = rnd(4 * P, 2 * D)
        self.w_qkv = [rnd(3 * D, D, scale=1 / 32) for _ in range(NW)]
        self.w_out = [rnd(D, D, scale=1 / 32) for _ in range(NW)]
        self.w_fc1 = [rnd(4 * D, D, scale=1 / 32) for _ in range(NW)]
        self.w_fc2 = [rnd(D, 4 * D, scale=1 / 64) for _ in range(NW)]
        self.ws = torch.empty(lib.gtav_gemm_skinny_workspace_bytes(P), dtype=torch.uint8, device=dev)
        self.counters = torch.zeros(512, dtype=torch.int32, device=dev)
        self.one = torch.zeros(1, dtype=torch.int32, device=dev)


b = Bufs()


def st():
    return N.current_stream()


def skinny(A, W, out, n, k, epi, splits=0, gate=False):
    def f():
        N.check(lib.gtav_gemm_skinny_bf16(A.data_ptr(), k, W.data_ptr(), k, out.data_ptr(), n, P, n, k, epi, b.bias.data_ptr(),
                                          out.data_ptr() if gate else None, n, b.mod.data_ptr() if gate else None, 6 * D, None, P,
                                          splits, b.ws.data_ptr(), b.counters.data_ptr(), st()), "skinny")
    return f


def tiled(A, W, out, m, n, k, epi):
    def f():
        N.check(lib.gtav_gemm_bf16(A.data_ptr(), k, W.data_ptr(), k, out.data_ptr(), n, m, n, k, epi, b.bias.data_ptr(), None, 0,
                                   None, 0, None, 1, 0, st()), "gemm")
    return f


def ln():
    N.check(lib.gtav_ln_modulate(b.h.data_ptr(), b.hn.data_ptr(), P, D, b.mod.data_ptr(), 6 * D, 0, D, None, P, st()), "ln")


def attn_s():
    N.check(lib.gtav_attention_seq(b.qkv.data_ptr(), b.att.data_ptr(), 1, P, H, b.rot.data_ptr(), 32, st()), "attn")


def attn_t():
    N.check(lib.gtav_attention_temporal_last(b.qkv.data_ptr(), b.att.data_ptr(), 1, 4, P, H, b.rott.data_ptr(), b.cache.data_ptr(), st()),
            "attn_t")


def ddim_like():
    N.check(lib.gtav_noise_clamp(b.ws.data_ptr(), b.ws.data_ptr() + 65536, 9216, 1, 9216, 20.0, st()), "clamp")


def report(name, us, **kw):
    print(json.dumps(dict(kernel=name, us_per_launch=round(us, 2), **kw)), flush=True)


def engine_steps():
    """The real last-frame step (gtav_dit_last_frame of a 16-block DiT, B=1, T=5) replayed from a graph, under the
    engine's environment switches."""
    import ctypes as C
    from gtav_b200.model.dit import DiT_models
    torch.manual_seed(0)
    x = torch.randn((1, 5, 16, 18, 32), device=dev)
    t = torch.tensor([[15, 15, 15, 15, 500]], device=dev)
    rows = torch.arange(5, dtype=torch.int32, device=dev)
    out = torch.empty((1, 1, 16, 18, 32), dtype=torch.bfloat16, device=dev)
    for label, env in (("default (weight-streaming GEMM, LN + temporal attention in the reduce)", {}),
                       ("separate LN / temporal-attention kernels", {"GTAV_FUSE": "0"}),
                       ("tiled GEMM everywhere", {"GTAV_SKINNY": "0"})):
        if env and "--default-only" in sys.argv:
            continue
        for k, v in env.items():
            os.environ[k] = v
        dit = DiT_models["DiT-S/2"]().to(dev).eval()
        with torch.no_grad():
            for b_ in dit.blocks:
                for h_ in ("s", "t"):
                    lin = getattr(b_, f"{h_}_adaLN_modulation")[-1]
                    lin.weight.normal_(std=0.02)
                    lin.bias.normal_(std=0.02)
        dit.forward_last_frame(x, t)                      # packs, plans, fills conditioning + K/V cache
        plan = dit._plan(1, 5)

        def step():
            N.check(lib.gtav_dit_last_frame(plan, x.data_ptr(), 0, rows[4:].data_ptr(), out.data_ptr(), st()), "last_frame")

        def ctx():
            N.check(lib.gtav_dit_context(plan, x.data_ptr(), 0, rows[:4].data_ptr(), st()), "context")

        def dense():
            N.check(lib.gtav_dit_backbone(plan, x.data_ptr(), 0, None, out.data_ptr() if False else dense_out.data_ptr(), st()), "backbone")
        dense_out = torch.empty((1, 5, 16, 18, 32), dtype=torch.bfloat16, device=dev)
        us = graph_time([step] * 8)
        usc = graph_time([ctx] * 3)
        usd = graph_time([dense] * 3)
        report(f"engine: {label}", us, ms_last_frame_step=round(us / 1e3, 4), ms_context_pass=round(usc / 1e3, 4),
               ms_dense_step=round(usd / 1e3, 4))
        for k in env:
            del os.environ[k]
        del dit


def main():
    if "--engine" in sys.argv:
        engine_steps()
        return
    n = 64
    report("noise_clamp 9216 elems (near-empty kernel: PDL chain floor)", graph_time([ddim_like] * n))
    report("ln_modulate 144 rows", graph_time([ln] * n))
    report("attention_seq 1 frame x 16 heads", graph_time([attn_s] * n))
    report("attention_temporal_last ctx=4", graph_time([attn_t] * n))
    shapes = dict(qkv=(b.hn, b.w_qkv, b.qkv, 3 * D, D, N.EPI_STORE, False), out=(b.att, b.w_out, b.h, D, D, N.EPI_BIAS_GATE_RES, True),
                  fc1=(b.hn, b.w_fc1, b.mlp, 4 * D, D, N.EPI_BIAS_GELU_TANH, False), fc2=(b.mlp, b.w_fc2, b.h, D, 4 * D, N.EPI_BIAS_GATE_RES, True))
    for name, (A, Ws, out, nn, k, epi, gate) in shapes.items():
        mb = 2.0 * (nn * k + P * k + P * nn) / 1e6
        for splits in (0, 1, 2, 4, 8, 16):
            try:
                us = graph_time([skinny(A, Ws[i % NW], out, nn, k, epi, splits, gate) for i in range(n)])
            except RuntimeError:
                continue
            report(f"gemm_skinny {name}", us, N=nn, K=k, splits=splits, gbs=round(mb / us * 1e3, 1))
        us = graph_time([tiled(A, Ws[i % NW], out, P, nn, k, N.EPI_STORE) for i in range(n)])
        report(f"gemm_tiled {name} M=144", us, N=nn, K=k, gbs=round(mb / us * 1e3, 1))
    # one half-block of the last-frame step, spatial and temporal flavour, as the engine enqueues it
    def half(i, temporal):
        return [ln, skinny(b.hn, b.w_qkv[i % NW], b.qkv, 3 * D, D, N.EPI_STORE), attn_t if temporal else attn_s,
                skinny(b.att, b.w_out[i % NW], b.h, D, D, N.EPI_BIAS_GATE_RES, 0, True), ln,
                skinny(b.hn, b.w_fc1[i % NW], b.mlp, 4 * D, D, N.EPI_BIAS_GELU_TANH),
                skinny(b.mlp, b.w_fc2[i % NW], b.h, D, 4 * D, N.EPI_BIAS_GATE_RES, 0, True)]
    calls = []
    for i in range(32):
        calls += half(i, i & 1)
    us = graph_time(calls)
    report("last-frame step body: 32 half-blocks x 7 kernels", us, us_per_half=round(us * 7, 2), ms_per_step=round(us * 7 * 32 / 1e3, 4))
    # dense-window GEMMs (M=720) in-graph
    A1, A4 = rnd(720, D), rnd(720, 4 * D)
    O1, O3, O4 = rnd(720, D), rnd(720, 3 * D), rnd(720, 4 * D)
    for name, (A, Ws, out, nn, k) in dict(qkv=(A1, b.w_qkv, O3, 3 * D, D), out=(A1, b.w_out, O1, D, D), fc1=(A1, b.w_fc1, O4, 4 * D, D),
                                          fc2=(A4, b.w_fc2, O1, D, 4 * D)).items():
        us = graph_time([tiled(A, Ws[i % NW], out, 720, nn, k, N.EPI_STORE) for i in range(n)])
        report(f"gemm_tiled {name} M=720", us, N=nn, K=k, tflops=round(2.0 * 720 * nn * k / us / 1e6, 1))

    # phase trace of the skinny GEMM (ns since the earliest CTA's entry), a few CTAs
    for name in ("qkv", "fc2"):
        A, Ws, out, nn, k, epi, gate = shapes[name]
        ctas = 160
        trace = torch.zeros((ctas, 8), dtype=torch.int64, device=dev)
        os.environ["GTAV_SKINNY_TRACE"] = str(trace.data_ptr())
        for i in range(4):
            skinny(A, Ws[i], out, nn, k, epi, 0, gate)()
        torch.cuda.synchronize()
        del os.environ["GTAV_SKINNY_TRACE"]
        t = trace.cpu()
        used = t[:, 0] > 0
        t0 = int(t[used, 0].min())
        rel = (t[used] - t0).clamp(min=0)
        names = ["entry", "setup", "W_landed", "A_landed", "acc_done", "partials", "rendezvous", "reduced"]
        print(f"# skinny {name}: phase stamps in ns relative to the first CTA's entry ({int(used.sum())} CTAs)")
        print("#   " + " ".join(f"{x:>10}" for x in names))
        for stat, fn in (("min", lambda x: x.min(0).values), ("median", lambda x: x.median(0).values), ("max", lambda x: x.max(0).values)):
            print(f"# {stat:>6} " + " ".join(f"{int(v):>10}" for v in fn(rel)))


if __name__ == "__main__":
    main()
