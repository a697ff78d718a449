"""Long sliding windows on the 16-block DiT-S/2: step times and temporal attention kernel bandwidth at max_frames 5, 8, 16
and 32 for B = 1 and 8.  One JSON line per measurement; the first line names the card and its power limit.

    python scripts/bench_long_window.py [--frames 5,8,16,32] [--batches 1,8] [--noise-steps 100]

Per (max_frames, B), with the window full (T = max_frames):
  * the last-frame step (gtav_dit_last_frame) and the context pass (gtav_dit_context), each captured N times back to back
    into a CUDA graph and timed with CUDA events over the replays, as scripts/bench_graph.py --engine does;
  * one generated frame through Sampler (context pass + noise_steps + 1 last-frame steps, one graph replay), CUDA events;
  * the temporal attention kernels alone: the dense kernel over T frames (gtav_attention_temporal) and the last-frame
    kernel against T - 1 cached frames (gtav_attention_temporal_last), in-graph.  Their inputs rotate over enough
    buffers to exceed the 126 MB L2, so every launch reads from HBM; bytes are computed from the shapes (dense: q|k|v rows
    read, output rows written; last frame: q|k|v row and the cache read, output row written), giving achieved GB/s.
The same DiT module serves every window: max_frames is changed on it between measurements (which re-packs it).
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gtav_b200._native as N
from gtav_b200.model.dit import DiT_models
from gtav_b200.sampler import Sampler

D, P, H = 1024, 144, 16
L2_BYTES = 126 * 2 ** 20


def report(**kw):
    print(json.dumps(kw), flush=True)


def graph_time(calls, reps=5):
    """calls: zero-arg launchers captured in order into one graph; GPU microseconds per launch over `reps` replays."""
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        for c in calls[: min(len(calls), 4)]:
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = ([x.strip() for x in q[0].split(",")] + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    report(card=torch.cuda.get_device_name(), nvidia_smi_name=name, power_limit=power, max_sm_clock=clock)


def kernels(lib, T, B):
    """The two temporal attention kernels alone at window T (dense) / T - 1 cached frames (last frame)."""
    dev = torch.device("cuda")
    tab = torch.stack([torch.cos(torch.arange(32.0)[:, None] * torch.ones(32)),
                       torch.sin(torch.arange(32.0)[:, None] * torch.ones(32))], dim=-1).contiguous().to(dev)
    res = {}
    # dense: reads B*T*P rows of 3D, writes B*T*P rows of D (no cache)
    rows = B * T * P
    dense_bytes = rows * (3 * D + D) * 2
    nb = max(2, math.ceil(2 * L2_BYTES / (rows * 3 * D * 2)))
    qkv = [torch.randn((rows, 3 * D), device=dev).to(torch.bfloat16) for _ in range(nb)]
    out = torch.empty((rows, D), device=dev, dtype=torch.bfloat16)

    def dense(i):
        return lambda: N.check(lib.gtav_attention_temporal(qkv[i % nb].data_ptr(), out.data_ptr(), B, T, P, H, tab.data_ptr(),
                                                           N.current_stream()), "dense")
    us = graph_time([dense(i) for i in range(4 * nb)])
    res["dense"] = dict(us=round(us, 2), bytes=dense_bytes, gbs=round(dense_bytes / us / 1e3, 1), buffers=nb)
    del qkv
    # last frame: reads B*P rows of 3D and B*(T-1)*P cache rows of 2D, writes B*P rows of D
    ctx = T - 1
    if ctx > 0:
        cache_bytes = B * ctx * P * 2 * D * 2
        last_bytes = B * P * (3 * D + D) * 2 + cache_bytes
        nb = max(2, math.ceil(2 * L2_BYTES / cache_bytes))
        caches = [torch.randn((B * ctx * P, 2 * D), device=dev).to(torch.bfloat16) for _ in range(nb)]
        q1 = torch.randn((B * P, 3 * D), device=dev).to(torch.bfloat16)
        o1 = torch.empty((B * P, D), device=dev, dtype=torch.bfloat16)

        def last(i):
            return lambda: N.check(lib.gtav_attention_temporal_last(q1.data_ptr(), o1.data_ptr(), B, ctx, P, H, tab.data_ptr(),
                                                                    caches[i % nb].data_ptr(), N.current_stream()), "last")
        us = graph_time([last(i) for i in range(4 * nb)])
        res["last"] = dict(us=round(us, 2), bytes=last_bytes, gbs=round(last_bytes / us / 1e3, 1), buffers=nb)
        del caches
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", default="5,8,16,32")
    ap.add_argument("--batches", default="1,8")
    ap.add_argument("--noise-steps", type=int, default=100)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long_window.py needs a CUDA device (gtav_b200 has no CPU path)")
    dev = torch.device("cuda")
    lib = N.load()
    card()
    torch.manual_seed(0)
    dit = DiT_models["DiT-S/2"]().to(dev).eval()
    with torch.no_grad():                                  # non-identity blocks, as scripts/bench_graph.py --engine
        for b_ in dit.blocks:
            for h_ in ("s", "t"):
                lin = getattr(b_, f"{h_}_adaLN_modulation")[-1]
                lin.weight.normal_(std=0.02)
                lin.bias.normal_(std=0.02)
    for T in [int(v) for v in args.frames.split(",")]:
        dit.max_frames = T                                 # re-packs on the next call
        for B in [int(v) for v in args.batches.split(",")]:
            x = torch.randn((B, T, 16, 18, 32), device=dev)
            t = torch.full((B, T), 15, device=dev, dtype=torch.long)
            t[:, -1] = 500
            rows = torch.arange(B * T, dtype=torch.int32, device=dev).reshape(B, T)
            ctx_rows, last_rows = rows[:, :-1].contiguous(), rows[:, -1].contiguous()
            out = torch.empty((B, 1, 16, 18, 32), dtype=torch.bfloat16, device=dev)
            dit.forward_last_frame(x, t)                   # packs, plans, fills conditioning and K/V cache
            plan = dit._plan(B, T)

            def step():
                N.check(lib.gtav_dit_last_frame(plan, x.data_ptr(), 0, last_rows.data_ptr(), out.data_ptr(), N.current_stream()),
                        "last_frame")

            def context():
                N.check(lib.gtav_dit_context(plan, x.data_ptr(), 0, ctx_rows.data_ptr(), N.current_stream()), "context")
            ms_step = graph_time([step] * 8) / 1e3
            ms_ctx = graph_time([context] * 3) / 1e3 if T > 1 else 0.0
            # one generated frame with a full window: T - 1 prompt latents, one new frame
            s = Sampler(dit, None, noise_steps=args.noise_steps)
            prompt = torch.randn((B, T - 1, 16, 18, 32), device=dev)
            noise = torch.randn((B, 1, 16, 18, 32), device=dev)
            s.sample_latents(prompt, None, T, noise=noise)          # graph capture
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            e0.record()
            for _ in range(reps):
                s.sample_latents(prompt, None, T, noise=noise)
            e1.record()
            torch.cuda.synchronize()
            ms_frame = e0.elapsed_time(e1) / reps
            s.close()
            k = kernels(lib, T, B)
            report(max_frames=T, B=B, ms_last_frame_step=round(ms_step, 4), ms_context_pass=round(ms_ctx, 4),
                   ms_sampler_frame=round(ms_frame, 2), sampler_frames_per_s=round(B * 1e3 / ms_frame, 2),
                   noise_steps=args.noise_steps, attn_temporal_dense=k["dense"], attn_temporal_last=k.get("last"))
            del s, x, out
            dit._release()                                 # free this shape's plans before the next one
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
