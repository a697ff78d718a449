#!/usr/bin/env python
"""Headline benchmark: generated frames/sec end-to-end (100-step DiT + VAE decode), BASELINE.json.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c1|c5] [--dump-outputs DIR]

A *step* is one complete rollout batch of the README inference shape (BASELINE config 2: B=1 rollout,
32 frames, 4 prompt frames, 100 noise steps => 28 generated frames x 101 DiT evaluations, plus VAE
encode of the prompt and decode of all 32 frames), run through gtav_b200's Sampler (C ABI -> sm_100a
kernels).  One JSON line is printed by rank 0:
  value  : generated frames/s with the prompt already resident in HBM (device-timed, max over ranks)
  e2e    : same metric through the public API with HOST buffers: pinned prompt video H2D and uint8 frames
           D2H inside the timed region
  roofline: the dominant kernel of the default (frame-cache) algorithm at B = 1, the weight-streaming tcgen05 GEMM,
           against the measured HBM bandwidth: algorithmic bytes of its 128 launches per step / their CUDA-event time
           (weights HBM-cold, as in the real step); at B > 1 and in the `dense` leg the tiled / CTA-pair GEMM against
           the measured sustained bf16 tensor throughput
  c5     : BASELINE config 5 on every N - 64 rollouts sharded r % world, one timed batch (strong scaling)
  c3, dense, c1, cpu_baseline, gpu_eager_baseline (N = 1 only): config 3 and the dense B = 8 window step; the
           reference's schedule at B = 1; config 1 through the product beside the CPU run of the same config; the CPU
           port of the reference (oracle/) timed on this box's host cores on config 1 in full; the reference's graph in
           torch eager on this GPU (informational)
With --impl reference only the CPU arm runs (the Python reference cannot travel to the GPU box; the
oracle port is its restatement) and prints the same line with "impl": "reference".
--dump-outputs DIR writes what the last timed step returned (dump_outputs); the inputs depend only on the arguments, so
two builds run with the same arguments can be compared file by file.
N > 1 (torchrun): every rank runs its own rollouts (weak scaling, no collective on the data path); every collective
of this file is in barrier() / timed(), called the same number of times by every rank.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "generated frames/sec end-to-end (100-step DiT + VAE decode)"
UNIT = "frames/s"
WORKLOADS = {
    # name: (B rollouts per GPU, total frames, prompt frames, noise steps, actions)
    "c2": dict(B=1, total=32, n_prompt=4, steps=100, actions=False,
               desc="README shape: unconditioned DiT-S/2, B=1, 32 frames (4 prompt), 100 noise steps, 360x640"),
    "c3": dict(B=8, total=32, n_prompt=4, steps=100, actions=True,
               desc="action-conditioned (W key), B=8 rollouts, 32 frames (4 prompt), 100 noise steps"),
    "c1": dict(B=1, total=8, n_prompt=4, steps=10, actions=False,
               desc="generate.py CPU case: B=1, 8 frames (4 prompt), 10 noise steps"),
    # 64 rollouts in total, sharded over the ranks (strong scaling): B = 64 / world per GPU
    "c5": dict(B=64, total=32, n_prompt=4, steps=100, actions=True, shard=True,
               desc="64 independent action-conditioned rollouts batch-sharded over the GPUs, 32 frames (4 prompt), 100 noise steps"),
}
DIT_STEP_GFLOP = 589.09          # per sample, 5-frame window (SURVEY.md section 8(d))
DIT_GEMM_GFLOP = 579.8           # the four per-half GEMMs only
VAE_ENC_GFLOP, VAE_DEC_GFLOP = 96.58, 191.69
DUMP_MAX_ELEMS = 15_000_000      # float32 values over all --dump-outputs files: 60 MB, under 64 MB with the .npy headers


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tf=d["bf16_tflops_sustained"], tf_burst=d["bf16_tflops"], hbm=d["hbm_gbs"], src="measured")
    return dict(tf=1400.0, tf_burst=1590.0, hbm=6650.0, src="fallback")


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, reasons, smax = [], set(), None
        for r in self.rows:
            try:
                sm.append(float(r[0])); smax = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        # "under load": upper half of the samples (the loop is busy the whole time; idle tails drop out)
        med = sm[len(sm) * 3 // 4] if sm else None
        return dict(sm_mhz=med, sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm))


def dump_outputs(out_dir, arrays):
    """Writes each array as out_dir/<name>.npy in float32 (uint8 frames convert exactly).  An array larger than its share
    of DUMP_MAX_ELEMS is written as a fixed sample instead: a flat vector of its elements at sorted indices drawn from a
    CPU generator seeded with 0, so the same shape always gives the same indices."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_MAX_ELEMS // len(arrays)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > share:
            idx = torch.randint(t.numel(), (share,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


# ------------------------------------------------------------------------------------------ product arm
def build_models(device):
    from gtav_b200.model.dit import DiT_models
    from gtav_b200.model.vae import VAE_models
    torch.manual_seed(0)
    dit = DiT_models["DiT-S/2"]()
    vae = VAE_models["vit-l-20-shallow-encoder"]()
    with torch.no_grad():      # random-init of the architecture, adaLN made non-zero so no block is an identity
        g = torch.Generator().manual_seed(1)
        for b in dit.blocks:
            for h in ("s", "t"):
                lin = getattr(b, f"{h}_adaLN_modulation")[-1]
                lin.weight.normal_(std=0.02, generator=g)
                lin.bias.normal_(std=0.02, generator=g)
        dit.final_layer.linear.weight.normal_(std=0.02, generator=g)
    return dit.to(device).eval(), vae.to(device).eval()


def synthetic_prompt(B, n):
    """Blue->red solid-colour ramp like the reference's dummy dataset, [B, n, 3, 360, 640] fp32 in [0,1]."""
    w = torch.linspace(0, 1, 5)[:n].view(n, 1)
    col = (1 - w) * torch.tensor([0.0, 0.0, 1.0]) + w * torch.tensor([1.0, 0.0, 0.0])
    return col.view(1, n, 3, 1, 1).expand(B, n, 3, 360, 640).contiguous()


def launches_per_rollout(wl, algorithm, depth=16, enc=6, dec=12):
    """Kernels of OURS launched per rollout batch (mirrors dit_engine.cu / vae_engine.cu / sampler.cu)."""
    backbone = 2 + 2 * depth * 7 + 3                           # patchify, patch GEMM, 7 per half, final LN/GEMM/unpatchify
    last = backbone
    if algorithm == "cached" and wl["B"] == 1 and os.environ.get("GTAV_FUSE", "1") != "0" and os.environ.get("GTAV_SKINNY", "1") != "0":
        # one rollout: LayerNorm + modulate and the temporal attention run inside the weight-streaming GEMMs' reduce
        # (dit_engine.cu: fuse_ln / fuse_tattn) - first LN, then 5 kernels per spatial half and 4 per temporal half
        last = 2 + 1 + depth * (5 + 4) + 2
    step = 1 + (last if algorithm == "cached" else backbone) + 1   # step_prep, backbone (window or last frame), ddim
    gen = wl["total"] - wl["n_prompt"]
    context = (2 + 2 * depth * 7) if algorithm == "cached" else 0
    per_frame = 1 + 1 + 4 + context + (wl["steps"] + 1) * step  # clamp, set_int, conditioning(4), context pass, steps
    vae_enc = 2 + enc * 7 + 3
    vae_dec = 2 + dec * 7 + 3
    return gen * per_frame + vae_enc + vae_dec * ((wl["B"] * wl["total"] + 31) // 32)


def measured_traffic(kernel):
    """DRAM bytes per launch of `kernel` from the committed ncu --set full capture (profiles/r*/roofline_traffic.json)."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*", "roofline_traffic.json")), reverse=True):
        try:
            d = json.load(open(path)).get(kernel)
        except Exception:
            d = None
        if d:
            return d["traffic_bytes_per_launch"]
    return None


def _hot_weights(dit):
    """Packed bf16 weights in _pack order: per half qkv_w, out_w, out_b, fc1_w, fc1_b, fc2_w, fc2_b."""
    dit._pack()
    keep = dit._engine[1]
    return [keep[i * 7:(i + 1) * 7] for i in range(2 * dit.depth)]


def _time_passes(one_pass, reps=10):
    """GPU time of one_pass: captured into a CUDA graph (the launches keep their programmatic-dependent-launch
    edges, as in the sampler) and replayed, so host launch cost is not in the number; CUDA events on the
    replay stream."""
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        one_pass()                                   # first-use configuration outside capture
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            one_pass()
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def gemm_roofline(dit, B, pk):
    """Tensor roofline of the tiled tcgen05 GEMM (the dense-window step's dominant kernel): the four hot GEMM
    shapes of a DiT step with CUDA events through the C ABI, cycling through the 16 blocks' own weight matrices so
    weights come from HBM (1.2 GB >> 126 MB L2) as in the real step."""
    import gtav_b200._native as N
    lib = N.load()
    M = B * 5 * 144
    dev = torch.device("cuda")
    D = 1024
    bufs = dict(a1=torch.randn((M, D), device=dev).to(torch.bfloat16), a4=torch.randn((M, 4 * D), device=dev).to(torch.bfloat16),
                o1=torch.empty((M, D), device=dev, dtype=torch.bfloat16), o3=torch.empty((M, 3 * D), device=dev, dtype=torch.bfloat16),
                o4=torch.empty((M, 4 * D), device=dev, dtype=torch.bfloat16))
    bias = torch.zeros(4 * D, device=dev, dtype=torch.bfloat16)
    halves = _hot_weights(dit)

    def run(a, w, out, n, k, epi):
        N.check(lib.gtav_gemm_bf16(a.data_ptr(), k, w.data_ptr(), k, out.data_ptr(), n, M, n, k, epi, bias.data_ptr(), None, 0,
                                   None, 0, None, 1, 0, N.current_stream()), "gemm")

    def one_pass():
        for h in halves:
            run(bufs["a1"], h[0], bufs["o3"], 3 * D, D, N.EPI_STORE)
            run(bufs["a1"], h[1], bufs["o1"], D, D, N.EPI_BIAS)
            run(bufs["a1"], h[3], bufs["o4"], 4 * D, D, N.EPI_BIAS_GELU_TANH)
            run(bufs["a4"], h[5], bufs["o1"], D, 4 * D, N.EPI_BIAS)
    ms = _time_passes(one_pass)                         # GEMM time of one DiT step (128 launches)
    tf = DIT_GEMM_GFLOP * B / ms                        # GFLOP / ms = TFLOP/s
    return dict(bound="tensor", achieved=round(tf, 1), peak=pk["tf"], unit="TFLOP/s", frac=round(tf / pk["tf"], 4),
                traffic=measured_traffic("gemm_bf16_kernel"), kernel="gemm_bf16_kernel (tcgen05, 128 launches per dense DiT step)",
                gemm_ms_per_dit_step=round(ms, 4), peak_source=f"{pk['src']} sustained bf16")


def skinny_roofline(dit, B, pk):
    """HBM roofline of the weight-streaming GEMM (the last-frame step's dominant kernel): algorithmic bytes per
    launch = the weight matrix (read once) + the token operand and result, / the average launch time, over the 128
    launches of one step on the blocks' own weights (805 MB per pass >> L2, so every launch streams from HBM)."""
    import gtav_b200._native as N
    lib = N.load()
    M = B * 144
    if B != 1:
        return None
    dev = torch.device("cuda")
    D = 1024
    a1 = torch.randn((M, D), device=dev).to(torch.bfloat16)
    a4 = torch.randn((M, 4 * D), device=dev).to(torch.bfloat16)
    o1 = torch.empty((M, D), device=dev, dtype=torch.bfloat16)
    o3 = torch.empty((M, 3 * D), device=dev, dtype=torch.bfloat16)
    o4 = torch.empty((M, 4 * D), device=dev, dtype=torch.bfloat16)
    bias = torch.zeros(4 * D, device=dev, dtype=torch.bfloat16)
    # the exchange the engine's last-frame pass uses: partial sums tagged with the launch's parity, one zeroed workspace per
    # GEMM shape, parity alternating along the (even number of) launches that share it (include/gtav_b200.h)
    halves = _hot_weights(dit)
    assert len(halves) % 2 == 0
    shapes = [(0, a1, o3, 3 * D, D, N.EPI_STORE), (1, a1, o1, D, D, N.EPI_BIAS), (3, a1, o4, 4 * D, D, N.EPI_BIAS_GELU_TANH),
              (5, a4, o1, D, 4 * D, N.EPI_BIAS)]
    wss = [torch.zeros(lib.gtav_gemm_skinny_workspace_bytes(M), dtype=torch.uint8, device=dev) for _ in shapes]
    def one_pass():
        for i, h in enumerate(halves):
            for (wi, a, out, n, k, epi), ws in zip(shapes, wss):
                N.check(lib.gtav_gemm_skinny_tagged_bf16(a.data_ptr(), k, h[wi].data_ptr(), k, out.data_ptr(), n, M, n, k, epi, bias.data_ptr(),
                                                         None, 0, None, 0, None, 144, 0, ws.data_ptr(), (i & 1) ^ 1, N.current_stream()),
                        "gemm_skinny_tagged")
    ms = _time_passes(one_pass)
    per_half = sum(2 * (n * k + M * k + M * n) for _, _, _, n, k, _ in shapes)          # bf16 bytes: W + A + out
    gb = len(halves) * per_half / 1e9
    gbs = gb / (ms / 1e3)
    return dict(bound="hbm", achieved=round(gbs, 1), peak=pk["hbm"], unit="GB/s", frac=round(gbs / pk["hbm"], 4),
                traffic=measured_traffic("gemm_skinny_kernel"),
                kernel="gemm_skinny_kernel (tcgen05 weight-streaming GEMM, 128 launches per last-frame DiT step)",
                algorithmic_mb_per_launch=round(gb * 1e3 / (4 * len(halves)), 3), us_per_launch=round(ms * 1e3 / (4 * len(halves)), 3),
                gemm_ms_per_last_frame_step=round(ms, 4), peak_source=f"{pk['src']} HBM copy bandwidth",
                note="bound by L2 traffic and latency, not by HBM: per launch the L2 fabric moves the weights (8 MB), the token slabs of "
                     "every row block (10.6 MB) and the split-K partial sums out and back (2 x 10.9 MB) - ~41 MB in ~6.5 us - in a "
                     "chain of phases (CTA entry + set-up 0.2 us, operand slabs 1.5, MMA 0.8, tagged partials out 1.2, reduce + fused "
                     "LayerNorm / temporal attention 2.0-3.5, next kernel's CTAs 0.6-1.0 later; "
                     "profiles/r02/skinny_in_step_trace_tagged.txt); its DRAM traffic equals the algorithmic bytes "
                     "(profiles/r02/roofline_traffic.json)")


def cpu_c1_run(init="initB", dit_steps_budget=None):
    """BASELINE config 1 EXACTLY on this box's host cores with the oracle port of the reference (fp32): B=1, dummy
    blue->red prompt, VAE-encode 4 frames, 4 generated frames x 11 DiT window evaluations (10 DDIM steps,
    generate.py:206), VAE-decode 8 frames to uint8.  Returns per-phase wall times and the final latents / frames."""
    from oracle import reference_port as rp
    from oracle.cases import C1
    from oracle.weights import DiTConfig, VAEConfig, dummy_prompt, make_dit_state, make_vae_state
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    c = C1
    dcfg, vcfg = DiTConfig(depth=c["depth"]), VAEConfig(enc_depth=c["enc_depth"], dec_depth=c["dec_depth"])
    dsd, vsd = make_dit_state(dcfg, seed=0, degenerate=(init == "initA")), make_vae_state(vcfg, seed=0)
    g = torch.Generator().manual_seed(c["seed"])
    noise = [torch.randn((1, 1, 16, 18, 32), generator=g) for _ in range(c["total_frames"] - c["n_prompt"])]
    video = dummy_prompt(5)[None, : c["n_prompt"]]
    with torch.inference_mode():
        rp.dit_forward(dsd, dcfg, torch.zeros(1, 1, 16, 18, 32), torch.zeros(1, 1, dtype=torch.long), None)      # warm-up
        t0 = time.perf_counter()
        lat = rp.encode_prompt(vsd, vcfg, video)
        t_enc = time.perf_counter() - t0
        it = iter(noise)
        t0 = time.perf_counter()
        x = rp.rollout(dsd, dcfg, lat, None, c["total_frames"], c["noise_steps"], lambda i: next(it))
        t_dit = time.perf_counter() - t0
        t0 = time.perf_counter()
        u8 = rp.decode_to_uint8(vsd, vcfg, x)
        t_dec = time.perf_counter() - t0
    n_steps = (c["total_frames"] - c["n_prompt"]) * (c["noise_steps"] + 1)
    return dict(cores=torch.get_num_threads(), encode_s=t_enc, dit_s=t_dit, decode_s=t_dec, total_s=t_enc + t_dit + t_dec,
                dit_steps=n_steps, s_per_dit_step=t_dit / n_steps, s_per_encode=t_enc / c["n_prompt"],
                s_per_decode=t_dec / c["total_frames"], latents=x, frames=u8)


def cpu_baseline(wl, c1=None):
    """The reference's CPU fp32 path (oracle port of it) on this box's host cores.  The bounded sample is BASELINE
    config 1 run in full (44 DiT window steps + 4 encodes + 8 decodes, measured, not extrapolated); `value` scales its
    measured per-step / per-encode / per-decode times to the workload's step count (the README rollout would take hours)."""
    c1 = c1 or cpu_c1_run()
    gen = wl["total"] - wl["n_prompt"]
    scale_b = 1.0 if not wl["actions"] else 1.0          # the action embedding is one 25x1024 GEMV per row: not measurable
    per_rollout = scale_b * (gen * (wl["steps"] + 1) * c1["s_per_dit_step"] + wl["n_prompt"] * c1["s_per_encode"] + wl["total"] * c1["s_per_decode"])
    return dict(value=round(gen / per_rollout, 6), unit=UNIT, cores=c1["cores"], kind="port",
                sample=(f"BASELINE config 1 in full on oracle/reference_port.py fp32: {c1['dit_steps']} DiT window steps (B=1,T=5) "
                        f"{c1['dit_s']:.2f} s + 4 VAE encodes {c1['encode_s']:.2f} s + 8 decodes {c1['decode_s']:.2f} s = {c1['total_s']:.2f} s "
                        f"wall ({4 / c1['total_s']:.4f} generated frames/s at C1); value = those per-step times scaled to the "
                        f"{gen}x{wl['steps'] + 1}-step rollout"),
                s_per_dit_step=round(c1["s_per_dit_step"], 4), c1_wall_s=round(c1["total_s"], 2),
                c1_generated_frames_per_s=round(4 / c1["total_s"], 5))


def bench_config(wl, B):
    """The `config` object of the JSON line - identical for the product arm and the reference arm."""
    gen = wl["total"] - wl["n_prompt"]
    return dict(workload=wl["desc"], rollouts_per_gpu=B, frames=wl["total"], prompt_frames=wl["n_prompt"],
                noise_steps=wl["steps"], dit_evals_per_rollout=gen * (wl["steps"] + 1),
                weights="random-init DiT-S/2 (607.9M) + ViT-L-20 VAE (229.2M), adaLN non-zero",
                l2="inputs larger than L2: 0.8-1.2 GB of bf16 weights streamed per DiT step (L2 126 MB)")


def run_reference_arm(args, wl, rank, world):
    """The reference's own CPU implementation of the path (oracle port: the Python reference cannot travel to the GPU
    box) on all host cores.  One step = one bounded sample = BASELINE config 1 in full (the same code path with 44
    instead of 2,828 DiT steps); --warmup untimed samples, then --steps timed ones."""
    if rank != 0:
        return
    t_all = time.perf_counter()
    for _ in range(args.warmup):                                    # pages in torch / MKL
        cpu_c1_run()
    vals = []
    for _ in range(args.steps):
        c1 = cpu_c1_run()
        vals.append(cpu_baseline(wl, c1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(latents=c1["latents"], frames=c1["frames"]))
    v = sum(c["value"] for c in vals) / len(vals)
    cb = dict(vals[-1], value=round(v, 6))
    gen = wl["total"] - wl["n_prompt"]
    line = dict(impl="reference", metric=METRIC, value=cb["value"], unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=round(1000.0 * sum(c["c1_wall_s"] for c in vals) / len(vals), 1),
                higher_is_better=True, scaling="strong" if wl.get("shard") else "weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=bench_config(wl, wl["B"]),
                algorithm="dense (every step recomputes the whole 5-frame window): the reference's own schedule, CPU fp32",
                cpu_baseline=cb, e2e=dict(value=cb["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0, samples_run=dict(warmup=args.warmup, timed=args.steps),
                extrapolated_ms_per_rollout=round(1000.0 * gen / v, 1),
                note="ms_per_step is the wall time of one bounded sample (config 1 in full: 44 DiT steps + 4 encodes + 8 decodes); "
                     "value scales its measured per-step times to the workload's step count",
                wall_s=round(time.perf_counter() - t_all, 1))
    print(json.dumps(line), flush=True)


def product_c1(dit_unused, vae_unused, dev, c1_cpu):
    """BASELINE config 1 through the product on the GPU, beside the CPU run of the identical config: same weights
    (oracle/weights.py, depth 16 + VAE 6/12), same dummy prompt, same noise; wall time of Sampler.generate with HOST
    prompt and HOST frames (copies inside), and - when the CPU run of this process is at hand - the parity metrics
    between the two (latent max-abs per generated frame, PSNR of the decoded uint8 frames)."""
    import math
    from gtav_b200.model.dit import DiT_models
    from gtav_b200.model.vae import VAE_models
    from gtav_b200.sampler import Sampler
    from oracle.cases import C1
    from oracle.weights import DiTConfig, VAEConfig, dummy_prompt, make_dit_state, make_vae_state
    c = C1
    dit = DiT_models["DiT-S/2"]()
    dit.load_state_dict(make_dit_state(DiTConfig(depth=c["depth"]), seed=0), strict=True)
    vae = VAE_models["vit-l-20-shallow-encoder"]()
    vae.load_state_dict(make_vae_state(VAEConfig(enc_depth=c["enc_depth"], dec_depth=c["dec_depth"]), seed=0), strict=True)
    dit, vae = dit.to(dev).eval(), vae.to(dev).eval()
    s = Sampler(dit, vae, noise_steps=c["noise_steps"])
    g = torch.Generator().manual_seed(c["seed"])
    noise = torch.stack([torch.randn((1, 1, 16, 18, 32), generator=g)[:, 0] for _ in range(c["total_frames"] - c["n_prompt"])], dim=1)
    video_host = dummy_prompt(5)[None, : c["n_prompt"]].contiguous().pin_memory()
    noise_dev = noise.to(dev)
    out_host = torch.empty((1, c["total_frames"], 360, 640, 3), dtype=torch.uint8).pin_memory()

    def run():
        frames, lat = s.generate(video_host.to(dev, non_blocking=True), None, c["total_frames"], noise=noise_dev)
        out_host.copy_(frames, non_blocking=True)
        return lat
    run()                                                        # plans + graph capture
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lat = run()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    res = dict(workload=WORKLOADS["c1"]["desc"], product_wall_s=round(wall, 4),
               product_generated_frames_per_s=round((c["total_frames"] - c["n_prompt"]) / wall, 2))
    if c1_cpu is not None:
        err = (lat.float().cpu() - c1_cpu["latents"]).abs()
        a, b = out_host.float(), c1_cpu["frames"].float()
        mse = float(((a - b) ** 2).mean())
        res.update(cpu_wall_s=round(c1_cpu["total_s"], 2), cpu_cores=c1_cpu["cores"],
                   speedup=round(c1_cpu["total_s"] / wall, 1),
                   latent_max_abs_per_frame=[round(float(err[:, f].max()), 5) for f in range(c["total_frames"])],
                   latent_mean_abs=round(float(err[:, c["n_prompt"]:].mean()), 6),
                   psnr_db_vs_cpu_fp32=round(99.0 if mse == 0 else 10 * math.log10(255.0 ** 2 / mse), 2),
                   tolerance="tests/test_full_config_gpu.py: latent max-abs <= 0.08 per generated frame, PSNR >= 41.9 dB "
                             "(= the bf16 model of the reference's autocast graph, 44.9 dB, minus 3 dB)")
    s.close()
    del dit, vae
    torch.cuda.empty_cache()
    return res


def gpu_eager_baseline(dev, batches=(1, 8), reps=3):
    """Informational: the reference's own eager graph on THIS GPU - oracle/reference_port.py (a restatement of the
    reference modules op by op) with its tensors on the device, under torch.autocast(cuda, bf16) as generate.py /
    denoise_step run it (train_dit.py:102-107): cuBLAS GEMMs + PyTorch SDPA + eager elementwise kernels.  One dense
    5-frame window step at B = 1 and B = 8.  This - not the CPU arm - is what a user of the reference gets on a B200
    today.  The port issues fewer, larger torch ops than the reference (no einops round trips, no per-call rotary
    table rebuild, no .item() syncs), so it is an optimistic stand-in for it."""
    from oracle import reference_port as rp
    from oracle.weights import DiTConfig, make_dit_state, w_key_actions
    cfg = DiTConfig()
    sd = {k: v.to(dev) for k, v in make_dit_state(cfg, seed=0).items()}
    out = {}
    with torch.inference_mode(), torch.autocast("cuda", dtype=torch.bfloat16):
        for B in batches:
            x = torch.randn(B, 5, 16, 18, 32, device=dev)
            t = torch.tensor([[15, 15, 15, 15, 499]], device=dev).expand(B, 5).contiguous()
            a = w_key_actions(B, 5).to(dev)
            for _ in range(2):
                rp.dit_forward(sd, cfg, x, t, a, rp.EAGER)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                rp.dit_forward(sd, cfg, x, t, a, rp.EAGER)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / reps
            out[f"B{B}"] = dict(ms_per_dense_dit_step=round(ms, 3), tflops=round(DIT_STEP_GFLOP * B / ms, 1))
    del sd
    torch.cuda.empty_cache()
    out["what"] = ("oracle/reference_port.py on cuda under torch.autocast(bf16): torch eager + cuBLAS + SDPA, dense 5-frame window "
                   "step, device-timed (host launch overhead included, as for a user of the reference)")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--algorithm", default="cached", choices=["cached", "dense"],
                    help="cached: context pass per frame + last-frame-only steps (default, same results); "
                         "dense: every step recomputes the whole window like the reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense-algorithm comparison leg")
    ap.add_argument("--no-c5", action="store_true", help="skip the 64-rollout strong-scaling leg (BASELINE config 5)")
    ap.add_argument("--no-c3", action="store_true", help="skip the B=8 legs (BASELINE config 3 and the dense window step at B=8)")
    ap.add_argument("--no-c1", action="store_true", help="skip the product run of BASELINE config 1")
    ap.add_argument("--no-eager", action="store_true", help="skip the torch-eager-on-GPU informational baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (fp32 latents, uint8 frames; rank 0's "
                         "rollouts) as DIR/<name>.npy in float32, at most 60 MB: a larger array becomes a fixed seeded sample of "
                         "its elements")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    wl = dict(WORKLOADS[args.workload])
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    strong = bool(wl.get("shard"))
    from gtav_b200.shard import rollout_generators, shard_rollouts
    if strong:                                   # fixed total work: this rank's share of the rollouts (shard.py: r % world)
        my_ids = shard_rollouts(wl["B"], rank, world)
        wl["B"] = len(my_ids)
    else:                                        # fixed work per GPU: world * B rollouts in total, r -> rank r % world
        my_ids = shard_rollouts(world * wl["B"], rank, world)

    if args.impl == "reference":
        run_reference_arm(args, wl, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; gtav_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    from gtav_b200.sampler import Sampler
    pk = peaks()
    dit, vae = build_models(dev)
    cached = args.algorithm == "cached"
    sampler = Sampler(dit, vae, noise_steps=wl["steps"], frame_cache=cached)
    B, total, n_prompt = wl["B"], wl["total"], wl["n_prompt"]
    gen = total - n_prompt

    def w_actions(b, frames):
        a = torch.zeros(b, frames, 25, device=dev)
        a[:, :, 3] = 1.0
        return a

    prompt_host = synthetic_prompt(B, n_prompt).pin_memory()
    prompt_dev = prompt_host.to(dev)
    actions = w_actions(B, total) if wl["actions"] else None
    # one generator per rollout, seeded by the GLOBAL rollout id (shard.py): a rollout's noise does not depend on the
    # world size or on the rank that owns it
    gens = rollout_generators(my_ids, dev)
    out_host = torch.empty((B, total, 360, 640, 3), dtype=torch.uint8).pin_memory()

    last = {}                                    # what the latest resident step returned, for --dump-outputs

    def rollout_resident():
        frames, lat = sampler.generate(prompt_dev, actions, total, generator=gens)
        last.update(latents=lat, frames=frames)
        return frames

    def rollout_e2e():
        p = prompt_host.to(dev, non_blocking=True)
        frames, _ = sampler.generate(p, actions, total, generator=gens)
        out_host.copy_(frames, non_blocking=True)
        return frames

    # Every collective of this file is in barrier() / timed(), and every rank calls timed() the same number of times, in
    # the same order; everything rank 0 does alone (dense leg, rooflines, CPU baseline) is collective-free.
    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(args.warmup):
        rollout_resident()
    with ClockSampler(local) as cs:
        ms_total = timed(rollout_resident, args.steps)
    clocks = cs.summary()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    last.clear()
    rollout_e2e()
    ms_e2e = timed(rollout_e2e, args.steps)

    # ---- BASELINE config 5 on every N: 64 action-conditioned rollouts sharded r % world (strong scaling), one timed
    # batch after a short warm-up that captures the graphs of this batch size; all ranks take part.
    c5 = None
    if not args.no_c5 and args.workload != "c5":
        w5 = WORKLOADS["c5"]
        ids5 = shard_rollouts(w5["B"], rank, world)
        B5 = len(ids5)
        s5 = Sampler(dit, vae, noise_steps=w5["steps"], frame_cache=True)
        p5 = synthetic_prompt(B5, w5["n_prompt"]).to(dev)
        a5 = w_actions(B5, w5["total"])
        g5 = rollout_generators(ids5, dev)
        s5.generate(p5, a5, w5["n_prompt"] + 2, generator=g5)            # warm-up: plans, graphs, decode of >= 32 frames
        ms5 = timed(lambda: s5.generate(p5, a5, w5["total"], generator=g5), 1)
        s5.close()
        del s5, p5, a5
        torch.cuda.empty_cache()
        gen5 = w5["total"] - w5["n_prompt"]
        c5 = dict(workload=w5["desc"], rollouts=w5["B"], rollouts_per_gpu=B5, n_gpus=world, scaling="strong",
                  value=round(w5["B"] * gen5 / (ms5 / 1000.0), 3), unit=UNIT,
                  per_gpu_frames_per_s=round(w5["B"] * gen5 / (ms5 / 1000.0) / world, 3), ms_per_batch=round(ms5, 1),
                  ms_per_dit_step=round(ms5 / (gen5 * (w5["steps"] + 1)), 4), rows_per_last_frame_step=144 * B5,
                  note="one timed batch (max over ranks) incl. VAE encode/decode; noise seeded by global rollout id; no collective on the data path")

    # ms per DiT step: two generated frames (context pass, if cached, + steps+1 steps each), device-timed; no collective
    def time_frames(smp, n_frames=2):
        lat = smp.encode_prompt(prompt_dev)
        smp.sample_latents(lat, actions, n_prompt + 1, generator=gens)          # capture / warm
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        smp.sample_latents(lat, actions, n_prompt + n_frames, generator=gens)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (n_frames * (wl["steps"] + 1))

    if rank == 0:
        ms_dit_step = time_frames(sampler)
        frames_total = world * B * gen * args.steps if not strong else WORKLOADS[args.workload]["B"] * gen * args.steps
        value = frames_total / (ms_total / 1000.0)
        e2e_v = frames_total / (ms_e2e / 1000.0)
        T = 5
        step_dense_gf = DIT_STEP_GFLOP * B
        if cached:
            # executed FLOPs per generated frame: one (T-1)-frame context pass + (steps+1) last-frame steps (SURVEY 8(d))
            last_gf = (116.411 + 1.359 + 0.009437 * T) * B
            ctx_gf = (116.411 + 1.359) * (T - 1) * B + 0.009437 * (T - 1) ** 2 * B
            exec_gf_per_step = (ctx_gf + (wl["steps"] + 1) * last_gf) / (wl["steps"] + 1)
            roof = skinny_roofline(dit, B, pk) or gemm_roofline(dit, B, pk)
            algo = ("frame cache: per generated frame one context pass over the T-1 context frames stores every temporal "
                    "layer's K/V, then each of the steps+1 DDIM steps recomputes only the frame being denoised (144*B rows) "
                    "against it - same arithmetic per row as the dense window (bit-identical with the tiled GEMM, "
                    "tests/test_model_gpu.py), 4.8x fewer executed FLOPs")
        else:
            exec_gf_per_step = step_dense_gf
            roof = gemm_roofline(dit, B, pk)
            algo = "dense (every step recomputes the whole 5-frame window, like the reference)"
        line = dict(metric=METRIC, value=round(value, 3), unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=round(ms_total / args.steps, 2), higher_is_better=True, scaling="strong" if strong else "weak",
                    vs_baseline=None, dtype="bf16", data="synthetic", config=bench_config(wl, B), algorithm=algo,
                    ms_per_dit_step=round(ms_dit_step, 4),
                    step_roofline=dict(bound="tensor", executed_tflops=round(exec_gf_per_step / ms_dit_step, 1),
                                       reference_equivalent_tflops=round(step_dense_gf / ms_dit_step, 1), peak=pk["tf"],
                                       unit="TFLOP/s", frac_executed=round(exec_gf_per_step / ms_dit_step / pk["tf"], 4),
                                       note="executed = FLOPs this algorithm runs per DDIM step / measured ms per step; "
                                            "reference-equivalent = the dense window's 589.09 GFLOP x B / the same time"),
                    roofline=roof,
                    e2e=dict(value=round(e2e_v, 3), unit=UNIT, h2d_bytes_per_step=prompt_host.numel() * 4,
                             d2h_bytes_per_step=out_host.numel()),
                    gpu_launches=launches_per_rollout(wl, args.algorithm) * args.steps, clocks=clocks)
        if c5 is not None:
            line["c5"] = c5
        if cached and not args.no_dense:
            # the dense algorithm on the same box, for the record: ms per dense step and the tiled GEMM's tensor roofline
            dense = Sampler(dit, vae, noise_steps=wl["steps"], frame_cache=False)
            ms_dense = time_frames(dense, n_frames=1)
            dense.close()
            line["dense"] = dict(ms_per_dit_step=round(ms_dense, 4), frames_per_s=round(B * 1000.0 / (ms_dense * (wl["steps"] + 1)), 3),
                                 step_tflops=round(step_dense_gf / ms_dense, 1), frac=round(step_dense_gf / ms_dense / pk["tf"], 4),
                                 gemm_roofline=gemm_roofline(dit, B, pk),
                                 note="every step recomputes the whole window; DiT steps only (no VAE), 1 generated frame timed")
        sampler.close()
        if not args.no_c3 and world == 1 and args.workload == "c2":
            # BASELINE config 3 (8 action-conditioned rollouts on one GPU): one timed batch of the shipped path, and the
            # reference's own schedule (dense 5-frame window, M = 5760 rows) for one generated frame - the regime the
            # north star's ">= 50 % of bf16 tensor peak sustained in DiT attention / MLP" is demonstrated in
            w3 = WORKLOADS["c3"]
            B3, gen3 = w3["B"], w3["total"] - w3["n_prompt"]
            p3, a3 = synthetic_prompt(B3, w3["n_prompt"]).to(dev), w_actions(B3, w3["total"])
            g3 = rollout_generators(list(range(B3)), dev)
            s3 = Sampler(dit, vae, noise_steps=w3["steps"], frame_cache=True)
            s3.generate(p3, a3, w3["n_prompt"] + 2, generator=g3)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            s3.generate(p3, a3, w3["total"], generator=g3)
            e1.record()
            torch.cuda.synchronize()
            ms3 = e0.elapsed_time(e1)
            lat3 = s3.encode_prompt(p3)
            s3.close()
            d3 = Sampler(dit, vae, noise_steps=w3["steps"], frame_cache=False)
            d3.sample_latents(lat3, a3, w3["n_prompt"] + 1, generator=g3)                      # plans, eager frame, graph capture
            torch.cuda.synchronize()
            e0.record()
            d3.sample_latents(lat3, a3, w3["n_prompt"] + 1, generator=g3)
            e1.record()
            torch.cuda.synchronize()
            ms3d = e0.elapsed_time(e1) / (w3["steps"] + 1)
            d3.close()
            line["c3"] = dict(workload=w3["desc"], value=round(B3 * gen3 / (ms3 / 1000.0), 3), unit=UNIT, ms_per_batch=round(ms3, 1),
                              ms_per_dit_step=round(ms3 / (gen3 * (w3["steps"] + 1)), 4), rows_per_last_frame_step=144 * B3,
                              dense=dict(ms_per_dit_step=round(ms3d, 4), step_tflops=round(DIT_STEP_GFLOP * B3 / ms3d, 1),
                                         frac=round(DIT_STEP_GFLOP * B3 / ms3d / pk["tf"], 4), rows=720 * B3,
                                         note="dense 5-frame window step at B=8 (the reference's schedule): whole DiT step incl. attention, "
                                              "LayerNorm, conditioning-free backbone; 589.09 GFLOP x 8 / measured time, against the measured sustained bf16 peak"),
                              note="one timed batch of 8 rollouts incl. VAE encode / decode (device-timed)")
            del s3, d3, p3, a3
            torch.cuda.empty_cache()
        c1_cpu = None
        if not args.no_cpu_baseline and world == 1:             # rank 0 at N = 1 only
            c1_cpu = cpu_c1_run()
            line["cpu_baseline"] = cpu_baseline(wl, c1_cpu)
        if not args.no_c1 and world == 1:
            line["c1"] = product_c1(dit, vae, dev, c1_cpu)
        if not args.no_eager and world == 1:
            try:
                line["gpu_eager_baseline"] = gpu_eager_baseline(dev)
            except Exception as e:                              # informational leg: never takes the line down
                line["gpu_eager_baseline"] = dict(error=f"{type(e).__name__}: {e}"[:300])
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
