"""Drop-in for the reference's generate.py CLI (reference generate.py:69-247): the same seven flags with the
same defaults and the same sampling constants, on gtav_b200's CUDA path.

    python -m gtav_b200.generate --dit_model_path dit.safetensors --vae_model_path vae.safetensors \
        --total-frames 32 --noise_steps 100 --output_path video1.mp4 [--start_frame img.jpg] [--use_actions]

What is kept (file:line of the reference):
  * flags and defaults                                  generate.py:71-118
  * B = 1, n_prompt = 4 (1 with --start_frame), noise_abs_max 20, stabilization_level 15, max_frames 5   :133-139
  * prompt from --start_frame: read_image / 255 -> Resize((360, 640))                                    :150-154
  * the all-"W" action tensor (index 3 of 25) for every frame                                            :159-160
  * VAE-encode prompt -> per frame clamp(randn) + (noise_steps + 1) DDIM steps -> VAE decode -> uint8    :186-244
  * mp4 at 10 fps                                                                                        :246
What differs, all additive or documented in DESIGN.md:
  * the loop runs inside Sampler (one CUDA-graph replay per generated frame) instead of Python;
    `--stepwise` runs the literal denoise_step loop of generate.py:200-220 through the drop-in modules instead;
  * key mismatches in a checkpoint raise (the reference prints and carries on, generate.py:32-38);
  * the inverted `--use_actions` test on the --start_frame path (generate.py:155-162: the flag raises
    AttributeError, its absence enables actions) is NOT reproduced: --use_actions means what its help says;
  * without --start_frame the reference streams its test split from the network (web_dataset.py); offline the
    prompt is the dummy dataset's 5-frame blue->red clip (dummy_dataset.py:16-28), or --prompt_video x.pt;
  * torchvision.io.write_video no longer exists: the writer is cv2.VideoWriter (mp4v), or a .npy / .pt dump
    when --output_path ends in .npy / .pt;
  * additive flags: --rollouts, --seed, --random_init, --timing_json, --stepwise, --prompt_video, --max_frames
    (sliding-window length, default 5 as generate.py:139 sets it; 1..32).
"""
from __future__ import annotations

import argparse
import json
import time

import torch

try:
    from .model.dit import DiT_models
    from .model.vae import VAE_models
    from .sampler import SCALING_FACTOR, Sampler
    from .train_dit import denoise_step
    from .utils import sigmoid_beta_schedule
except ImportError:  # package directory on sys.path, reference-style imports
    from model.dit import DiT_models
    from model.vae import VAE_models
    from sampler import SCALING_FACTOR, Sampler
    from train_dit import denoise_step
    from utils import sigmoid_beta_schedule


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description="Video generation script")
    # --- the reference's flags, verbatim (generate.py:71-118)
    p.add_argument("--total-frames", type=int, default=32, help="Total number of frames to generate (default: 32)")
    p.add_argument("--dit_model_path", type=str, default="checkpoints/oasis500m.pt",
                   help="Path to DiT model checkpoint (default: checkpoints/oasis500m.pt)")
    p.add_argument("--vae_model_path", type=str, default="checkpoints/vit-l-20.safetensors",
                   help="Path to VAE model checkpoint (default: checkpoints/vit-l-20-shallow-encoder.pt)")
    p.add_argument("--noise_steps", type=int, default=100, help="Number of noise steps (default: 100)")
    p.add_argument("--use_actions", action="store_true",
                   help="Use actions (default: False). We will use W for all the frames.")
    p.add_argument("--output_path", type=str, default="video1.mp4",
                   help="Path to save the generated video (default: video1.mp4)")
    p.add_argument("--start_frame", type=str, default=None, help="Path to save the start frame (default: None)")
    # --- additive
    p.add_argument("--rollouts", type=int, default=1, help="independent rollouts in one batch (reference: 1)")
    p.add_argument("--seed", type=int, default=None, help="seed of the CUDA noise generator (reference: unseeded)")
    p.add_argument("--random_init", action="store_true",
                   help="skip checkpoint loading: random-init weights of the architecture (benchmarks, smoke runs)")
    p.add_argument("--prompt_video", type=str, default=None,
                   help=".pt tensor [n>=4, 3, 360, 640] in [0,1] used as the prompt instead of the dummy clip")
    p.add_argument("--stepwise", action="store_true",
                   help="run the literal per-step Python loop of the reference through the drop-in modules")
    p.add_argument("--max_frames", type=int, default=5,
                   help="frames in the sliding window the DiT sees, 1..32 (reference: 5, generate.py:139)")
    p.add_argument("--timing_json", type=str, default=None, help="write a timing report to this path")
    return p


def load_models(dit_model_path, vae_model_path, device, random_init=False):
    """generate.py:28-47 (`load_models`): build both modules, load safetensors checkpoints, move to the GPU.
    The bf16 cast that `accelerator.prepare` + autocast apply happens once, when the weights are packed."""
    dit = DiT_models["DiT-S/2"]()
    vae = VAE_models["vit-l-20-shallow-encoder"]()
    if not random_init:
        from safetensors.torch import load_model
        for name, module, path in (("DiT", dit, dit_model_path), ("VAE", vae, vae_model_path)):
            missing, unexpected = load_model(module, path, strict=False)
            if missing or unexpected:
                raise RuntimeError(f"Error loading {name} model from {path}. Missing keys: {missing}. "
                                   f"Unexpected keys: {unexpected}")
    return dit.to(device).eval(), vae.to(device).eval()


def dummy_clip(n_frames=5, height=360, width=640):
    """The dummy dataset's clip: solid colour moving from blue to red (reference dummy_dataset.py:16-28)."""
    w = torch.linspace(0, 1, n_frames).view(n_frames, 1)
    col = (1 - w) * torch.tensor([0.0, 0.0, 1.0]) + w * torch.tensor([1.0, 0.0, 0.0])
    return col.view(n_frames, 3, 1, 1).expand(n_frames, 3, height, width).contiguous()


def load_prompt(args, device):
    """-> video [1, n_prompt, 3, 360, 640] fp32 in [0, 1] (generate.py:149-184)."""
    if args.start_frame is not None:
        from torchvision import transforms
        from torchvision.io import read_image
        img = read_image(args.start_frame).float() / 255.0
        img = transforms.Resize((360, 640))(img[:3])
        return img.view(1, 1, 3, 360, 640).to(device), 1
    if args.prompt_video is not None:
        clip = torch.load(args.prompt_video).float()
    else:
        clip = dummy_clip()
    if clip.dim() != 4 or clip.shape[0] < 4 or tuple(clip.shape[1:]) != (3, 360, 640):
        raise RuntimeError(f"prompt video must be [n>=4, 3, 360, 640], got {tuple(clip.shape)}")
    return clip[:4].unsqueeze(0).to(device), 4


def write_video(path, frames_u8, fps=10):
    """frames_u8 [T, H, W, 3] uint8 RGB on the host.  Stands in for torchvision.io.write_video (generate.py:246),
    which torchvision 0.26 removed."""
    if path.endswith(".npy"):
        import numpy as np
        np.save(path, frames_u8.numpy())
        return
    if path.endswith(".pt"):
        torch.save(frames_u8, path)
        return
    import cv2
    T, H, W, _ = frames_u8.shape
    writer = cv2.VideoWriter(path, cv2.VideoWriter_fourcc(*"mp4v"), float(fps), (W, H))
    if not writer.isOpened():
        raise RuntimeError(f"cannot open a video writer for {path}")
    for f in frames_u8.numpy():
        writer.write(cv2.cvtColor(f, cv2.COLOR_RGB2BGR))
    writer.release()


@torch.inference_mode()
def rollout_stepwise(model, vae, video, actions, total_frames, n_prompt, noise_steps, generator=None,
                     noise_abs_max=20, stabilization_level=15):
    """The reference's own loop, line for line in behaviour (generate.py:186-244), with the drop-in modules doing
    the arithmetic: one DiT.forward + one DDIM kernel per step, Python bookkeeping in between."""
    sampler = Sampler(model, vae, noise_steps=noise_steps)            # only for encode / decode helpers
    x = sampler.encode_prompt(video[:, :n_prompt])
    B = x.shape[0]
    noise_range = torch.linspace(0, 999, noise_steps + 1)
    betas = sigmoid_beta_schedule(1000).float().to(x.device)
    alphas_cumprod = torch.cumprod(1.0 - betas, dim=0).view(-1, 1, 1, 1)
    for i in range(n_prompt, total_frames):
        chunk = torch.randn((B, 1, *x.shape[-3:]), device=x.device, generator=generator)
        chunk = torch.clamp(chunk, -noise_abs_max, +noise_abs_max)
        x = torch.cat([x, chunk], dim=1)
        start = max(0, i + 1 - model.max_frames)
        for noise_idx in reversed(range(0, noise_steps + 1)):
            x_pred, _ = denoise_step(dit_model=model, x_noisy=x, noise_idx=noise_idx,
                                     stabilization_level=stabilization_level, noise_range=noise_range,
                                     alphas_cumprod=alphas_cumprod, start_frame=start, dtype=torch.bfloat16,
                                     actions=actions)
            x[:, -1:] = x_pred[:, -1:]
    return sampler.decode_frames(x), x


def main(argv=None):
    args = build_parser().parse_args(argv)
    assert torch.cuda.is_available(), "gtav_b200 runs only on sm_100a GPUs (no CPU fallback)"
    device = torch.device("cuda", torch.cuda.current_device())
    print("Using bf16 precision.")
    t_load = time.perf_counter()
    model, vae = load_models(args.dit_model_path, args.vae_model_path, device, random_init=args.random_init)
    t_load = time.perf_counter() - t_load

    B = max(1, args.rollouts)
    total_frames = args.total_frames
    noise_abs_max, stabilization_level = 20, 15
    model.max_frames = args.max_frames
    video, n_prompt = load_prompt(args, device)
    video = video.expand(B, *video.shape[1:]).contiguous()
    print(f"We will generate {total_frames} frames, starting with {n_prompt} frames.")
    print(f"Model max frames: {model.max_frames}")
    print(f"Noise steps: {args.noise_steps}")
    print(f"Stabilization level: {stabilization_level}")
    print(f"Noise absolute max: {noise_abs_max}")
    print(f"Actions is set to {args.use_actions}.")
    actions = None
    if args.use_actions:
        actions = torch.zeros((B, total_frames, 25), device=device)
        actions[:, :, 3] = 1  # W for all frames (generate.py:159-160, 180)
    gen = None
    if args.seed is not None:
        gen = torch.Generator(device=device).manual_seed(args.seed)

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if args.stepwise:
        frames, latents = rollout_stepwise(model, vae, video, actions, total_frames, n_prompt, args.noise_steps, gen,
                                           noise_abs_max, stabilization_level)
    else:
        sampler = Sampler(model, vae, noise_steps=args.noise_steps, stabilization_level=stabilization_level,
                          noise_abs_max=noise_abs_max)
        frames, latents = sampler.generate(video, actions, total_frames, generator=gen)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0

    host = frames.cpu()
    write_video(args.output_path, host[0])
    for r in range(1, B):
        stem, dot, ext = args.output_path.rpartition(".")
        write_video(f"{stem}_{r}{dot}{ext}" if dot else f"{args.output_path}_{r}", host[r])
    print(f"generation saved to {args.output_path}.")
    gen_frames = B * (total_frames - n_prompt)
    report = dict(rollouts=B, total_frames=total_frames, prompt_frames=n_prompt, noise_steps=args.noise_steps,
                  seconds=round(dt, 4), generated_frames_per_s=round(gen_frames / dt, 3), load_seconds=round(t_load, 2),
                  mode="stepwise" if args.stepwise else "sampler", scaling_factor=SCALING_FACTOR,
                  note="first call includes CUDA-graph capture and lazy module load")
    print(json.dumps(report))
    if args.timing_json:
        with open(args.timing_json, "w") as f:
            json.dump(report, f)
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
