"""Interactive sessions batched by StreamPool against the same sessions served as B = 1 FrameStreams, on the 16-block
DiT-S/2 (non-zero adaLN) and the ViT-L/20 VAE, 100 noise steps.  One JSON line per measurement; the first line names the
card and its power limit.

    python scripts/bench_stream_pool.py [--frames 5,16] [--capacities 1,2,4,8] [--noise-steps 100] [--steps 5]

Per (max_frames, capacity), CUDA events around StreamPool.step (one generated frame for every open session, decode
included), warm-up steps excluded:
  * full: every slot open with a full window (max_frames - 1 prompt frames);
  * staggered: one session joins per step with 1 prompt frame, so short and full windows mix; timed once every slot is
    open, while the newest windows are still short;
  * the aggregate frames/s of each, capacity / step time.
Per max_frames, the same through one B = 1 FrameStream with a full window (frame time, decode included): sessions served one
after another get 1 / that time frames/s whatever their number.  Pool capacity 1 against it is the cost of running the
temporal attention as its own kernel (a plan with window lengths does not fuse it into the to_qkv GEMM).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gtav_b200.model.dit import DiT_models
from gtav_b200.model.vae import VAE_models
from gtav_b200.sampler import Sampler


def report(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = ([x.strip() for x in q[0].split(",")] + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    report(card=torch.cuda.get_device_name(), nvidia_smi_name=name, power_limit=power, max_sm_clock=clock)


def timed(fn, n):
    """GPU milliseconds per call of fn over n calls (CUDA events; fn's own host work overlaps the queued GPU work)."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def action(i):
    a = torch.zeros(25, device="cuda")
    a[3 + i % 4] = 1.0
    return a


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", default="5,16")
    ap.add_argument("--capacities", default="1,2,4,8")
    ap.add_argument("--noise-steps", type=int, default=100)
    ap.add_argument("--steps", type=int, default=5, help="timed steps per measurement")
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stream_pool.py needs a CUDA device (gtav_b200 has no CPU path)")
    dev = torch.device("cuda")
    card()
    torch.manual_seed(0)
    dit = DiT_models["DiT-S/2"]().to(dev).eval()
    with torch.no_grad():                                  # non-identity blocks, as scripts/bench_graph.py --engine
        for b_ in dit.blocks:
            for h_ in ("s", "t"):
                lin = getattr(b_, f"{h_}_adaLN_modulation")[-1]
                lin.weight.normal_(std=0.02)
                lin.bias.normal_(std=0.02)
    vae = VAE_models["vit-l-20-shallow-encoder"]().to(dev).eval()
    video = torch.rand((32, 3, 360, 640), device=dev)
    acts = torch.stack([action(i) for i in range(32)])
    for T in [int(v) for v in args.frames.split(",")]:
        dit.max_frames = T                                 # re-packs on the next call
        s = Sampler(dit, vae, noise_steps=args.noise_steps)
        n_full = max(T - 1, 1)
        # one B = 1 FrameStream, full window
        st = s.stream(video[None, :n_full], acts[None, :n_full], generator=torch.Generator(device=dev).manual_seed(0))
        k = [0]

        def solo():
            st.next(action(k[0])[None])
            k[0] += 1
        for _ in range(args.warmup):
            solo()
        solo_ms = timed(solo, args.steps)
        report(max_frames=T, what="framestream_b1", ms_per_frame=round(solo_ms, 3), fps=round(1e3 / solo_ms, 2))
        for cap in [int(v) for v in args.capacities.split(",")]:
            pool = s.pool(cap, use_actions=True)
            ids = [pool.open(video[:n_full], acts[:n_full], generator=torch.Generator(device=dev).manual_seed(i))
                   for i in range(cap)]
            step = lambda: pool.step(actions={sid: action(k[0]) for sid in ids})
            for _ in range(args.warmup):
                step()
            full_ms = timed(step, args.steps)
            for sid in ids:
                pool.close(sid)
            # staggered joins: one session per step with one prompt frame
            ids = []
            for i in range(cap):
                ids.append(pool.open(video[i:i + 1], acts[i:i + 1], generator=torch.Generator(device=dev).manual_seed(i)))
                step()
            lens = [min(1 + cap - i, T - 1) + 1 for i in range(cap)]
            stag_ms = timed(step, args.steps)
            rec = dict(max_frames=T, capacity=cap, noise_steps=args.noise_steps,
                       full=dict(ms_per_step=round(full_ms, 3), fps=round(cap * 1e3 / full_ms, 2)),
                       staggered=dict(ms_per_step=round(stag_ms, 3), fps=round(cap * 1e3 / stag_ms, 2),
                                      window_lengths_at_start=lens),
                       framestream_b1_one_after_another_fps=round(1e3 / solo_ms, 2))
            if cap == 1:
                rec["pool1_over_framestream_b1"] = round(full_ms / solo_ms, 4)
            report(**rec)
            del pool
        s.close()


if __name__ == "__main__":
    main()
