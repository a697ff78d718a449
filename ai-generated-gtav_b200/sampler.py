"""Whole-rollout sampler: the autoregressive loop of reference generate.py:186-244 driven through the
C ABI with one CUDA-graph replay per DDIM step.

    s = Sampler(dit, vae, noise_steps=100)
    frames_u8, latents = s.generate(prompt_video, actions, total_frames=32)

Semantics are the reference's: context frames at t = stabilization_level, last frame walks
linspace(0, 999, steps+1) truncated to integers from the top, steps+1 DiT evaluations per frame, only
the last frame of the window is updated, new frames start from clamp(randn, +-noise_abs_max), frames are
decoded with the pixel epilogue of generate.py:241-244.  What differs is scheduling only:
  * B independent rollouts per call (the reference hard-codes B = 1, generate.py:133);
  * the adaLN conditioning table of a frame is computed once per frame instead of once per step
    (it depends on (t, action) only - an exact hoist);
  * frame_cache (default on): the context frames of the window do not change during the steps of a
    frame and cannot see the frame being denoised (per-frame spatial attention, causal temporal
    attention), so one context pass per frame stores their K/V and every step recomputes only the last
    frame against that cache - the same arithmetic on 1/5 of the rows;
  * no host work per step: timestep rows and DDIM coefficients are derived on the device.
Noise comes from torch (`torch.randn` on the rollout's device, as generate.py:201) unless the caller
supplies it, so a seeded torch generator reproduces a run.
"""
from __future__ import annotations

import ctypes as C

import torch

try:
    from . import _native as N
    from .utils import sigmoid_beta_schedule
except ImportError:
    import _native as N
    from utils import sigmoid_beta_schedule

SCALING_FACTOR = 0.07843137255   # generate.py:51,241


class Sampler:
    def __init__(self, dit, vae=None, noise_steps: int = 100, stabilization_level: int = 15, noise_abs_max: float = 20.0,
                 max_noise_level: int = 1000, use_graph: bool = True, frame_cache: bool = True, alphas_cumprod=None):
        self.dit, self.vae = dit, vae
        self.steps = int(noise_steps)
        self.stab = int(stabilization_level)
        self.noise_abs_max = float(noise_abs_max)
        self.use_graph = bool(use_graph)
        self.frame_cache = bool(frame_cache)
        self.levels = [int(v) for v in torch.linspace(0, max_noise_level - 1, self.steps + 1).tolist()]
        if alphas_cumprod is None:              # generate.py:195-197 (clamp_min 1e-4, the schedule's default)
            betas = sigmoid_beta_schedule(max_noise_level).float()
            self.abar_host = torch.cumprod(1.0 - betas, dim=0)
        else:                                   # a caller's own table, e.g. the trainer's clamp_min 1e-6 one (train_dit.py:297-307)
            self.abar_host = alphas_cumprod.detach().reshape(-1).to(device="cpu", dtype=torch.float32).clone()
            if self.abar_host.numel() != max_noise_level:
                raise RuntimeError(f"alphas_cumprod must hold {max_noise_level} levels, got {self.abar_host.numel()}")
        self._ctx = {}          # (B, T) -> dict(sampler handle, buffers)
        self._stream = None
        dit._dependants.add(self)   # the DiT drops our handles / graphs before it releases the plans they were built on
        self.frame_elems = dit.in_channels * dit.input_h * dit.input_w

    # ------------------------------------------------------------------ per-(B,T) context
    def _context(self, B, T, dev):
        key = (B, T)
        # first: a load_state_dict / in-place weight change / .to() since the last call re-packs the weights, which
        # releases every plan and (through DiT._release -> _invalidate) every cached context of this sampler
        self.dit._pack()
        if key not in self._ctx:
            self._ctx[key] = self._new_context(B, T, dev)
        return self._ctx[key]

    def _new_context(self, B, T, dev, lengths=None, owner=None):
        """Sampler handle and buffers over a (B, T) DiT plan.  lengths: device int32 [B] window lengths attached to the
        plan of `owner`'s own (StreamPool), before the sampler handle captures anything."""
        lib = N.load()
        rows = lib.gtav_sampler_cond_rows(B, T, self.steps)
        plan = self.dit._plan(B, T, rows, owner=owner)
        if lengths is not None:
            N.check(lib.gtav_dit_plan_set_window_lengths(plan, lengths.data_ptr()), "gtav_dit_plan_set_window_lengths")
        n = self.frame_elems
        x_win = torch.zeros((B, T, n), dtype=torch.float32, device=dev)
        v_out = torch.zeros((B, T, n), dtype=torch.bfloat16, device=dev)
        scratch = torch.zeros(lib.gtav_sampler_scratch_bytes(B, T, self.steps) + 256, dtype=torch.uint8, device=dev)
        sbase = (scratch.data_ptr() + 255) & ~255
        abar = self.abar_host.to(dev)
        levels = (C.c_int * (self.steps + 1))(*self.levels)
        h = N.vp()
        flags = (N.SAMPLER_GRAPH if self.use_graph else 0) | (N.SAMPLER_FRAME_CACHE if self.frame_cache else 0)
        N.check(lib.gtav_sampler_create(plan, B, T, self.steps, n, x_win.data_ptr(), v_out.data_ptr(), abar.data_ptr(), levels,
                                        sbase, scratch.numel() - 256, flags, N.current_stream(), C.byref(h)),
                "gtav_sampler_create")
        return dict(h=h, plan=plan, x_win=x_win, v_out=v_out, scratch=scratch, abar=abar, rows=rows, lengths=lengths)

    def close(self):
        lib = N.load()
        for ctx in self._ctx.values():
            lib.gtav_sampler_destroy(ctx["h"])
        self._ctx = {}

    def _invalidate(self):
        """Called by the DiT before it releases its plans (weights re-packed): captured graphs and sampler handles refer
        to the old plans' workspaces and weight copies, so they are destroyed once pending work has drained."""
        if self._ctx:
            torch.cuda.synchronize()
            self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ conditioning rows of one frame
    def _cond_inputs(self, B, T, act_win, dev):
        """t [rows] int64 and actions [rows, A] for the table layout of gtav_sampler_cond_rows; act_win: the window's
        actions [B, T, A] (context frames then the frame being generated) or None."""
        S1 = self.steps + 1
        t_ctx = torch.full((B * (T - 1),), self.stab, dtype=torch.long, device=dev)
        t_last = torch.tensor(self.levels, dtype=torch.long, device=dev).repeat(B)
        t = torch.cat([t_ctx, t_last])
        if act_win is None:
            return t, None
        a_ctx = act_win[:, : T - 1].reshape(B * (T - 1), -1)
        a_last = act_win[:, T - 1].unsqueeze(1).expand(B, S1, -1).reshape(B * S1, -1)
        return t, torch.cat([a_ctx, a_last]).to(torch.float32).contiguous()

    # ------------------------------------------------------------------ one generated frame
    def _denoise_frame(self, ctx_latents, chunk, act_win, stream, steps_limit=None, ctx=None):
        """ctx_latents [B, T-1, n] fp32 (the window's context frames), chunk [B, n] N(0,1) draws for the new frame,
        act_win [B, T, A] or None -> the new frame's latent [B, n] (a view of the window buffer: copy it before the
        next call).  Enqueued on `stream`: clamp, conditioning table, context pass + (steps+1) DDIM steps.
        ctx: a context of the caller's own (_new_context) instead of this sampler's (B, T) one."""
        lib = N.load()
        dev = chunk.device
        B, n = chunk.shape
        T = ctx_latents.shape[1] + 1
        if ctx is None:
            ctx = self._context(B, T, dev)
        xw = ctx["x_win"]
        xw[:, : T - 1] = ctx_latents
        N.check(lib.gtav_noise_clamp(chunk.data_ptr(), xw.data_ptr() + (T - 1) * n * 4, T * n, B, n,
                                     self.noise_abs_max, stream.cuda_stream), "gtav_noise_clamp")
        t_rows, a_rows = self._cond_inputs(B, T, act_win, dev)
        N.check(lib.gtav_dit_conditioning(ctx["plan"], t_rows.data_ptr(), N.ptr(a_rows), stream.cuda_stream),
                "gtav_dit_conditioning")
        N.check(lib.gtav_sampler_run_frame(ctx["h"], -1 if steps_limit is None else int(steps_limit),
                                           stream.cuda_stream), "gtav_sampler_run_frame")
        return xw[:, T - 1]

    # ------------------------------------------------------------------ latents -> latents
    @torch.no_grad()
    def sample_latents(self, prompt_latents, actions, total_frames, noise=None, generator=None, steps_limit=None,
                       on_frame=None):
        """prompt_latents [B, n_prompt, C, h, w] -> fp32 latents [B, total_frames, C, h, w].
        noise: optional [B, total_frames - n_prompt, C, h, w] (unclamped N(0,1) draws)."""
        N.require_cuda(prompt_latents, "prompt_latents")
        lib = N.load()
        dev = prompt_latents.device
        B, n_prompt = prompt_latents.shape[:2]
        shape = tuple(prompt_latents.shape[2:])
        n = self.frame_elems
        if actions is not None:
            actions = actions.to(dev)
        x = torch.zeros((B, total_frames, n), dtype=torch.float32, device=dev)
        x[:, :n_prompt] = prompt_latents.reshape(B, n_prompt, n).float()
        if self.use_graph and self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)     # graph capture needs a non-default stream
        stream = self._stream if self.use_graph else torch.cuda.current_stream(dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev), torch.cuda.stream(stream):
            for i in range(n_prompt, total_frames):
                start = max(0, i + 1 - self.dit.max_frames)
                T = i + 1 - start
                if noise is not None:
                    chunk = noise[:, i - n_prompt].to(device=dev, dtype=torch.float32).reshape(B, n).contiguous()
                elif isinstance(generator, (list, tuple)):
                    # one generator per rollout (shard.rollout_generators: seeded by the GLOBAL rollout id, so a
                    # rollout's noise does not depend on which rank owns it or on how many rollouts share the batch)
                    if len(generator) != B:
                        raise RuntimeError(f"sample_latents: {len(generator)} generators for {B} rollouts")
                    chunk = torch.stack([torch.randn((n,), device=dev, generator=g) for g in generator])
                else:
                    chunk = torch.randn((B, n), device=dev, generator=generator)
                act_win = None if actions is None else actions[:, start:start + T]
                x[:, i] = self._denoise_frame(x[:, start:i], chunk, act_win, stream, steps_limit)
                if on_frame is not None:
                    on_frame(i, x)
        torch.cuda.current_stream(dev).wait_stream(stream)
        return x.reshape(B, total_frames, *shape)

    # ------------------------------------------------------------------ pixels -> pixels
    @torch.no_grad()
    def encode_prompt(self, video):
        """video [B, n, 3, H, W] in [0,1] -> latents [B, n, C, h, w] (generate.py:50-66 `vae_encode`)."""
        B, n = video.shape[:2]
        vae = self.vae
        frames = video.reshape(B * n, *video.shape[2:])
        mean = vae.encode_mean(frames * 2 - 1, scale=SCALING_FACTOR, round_bf16=True)
        return mean.reshape(B, n, vae.seq_h, vae.seq_w, vae.latent_dim).permute(0, 1, 4, 2, 3).contiguous()

    @torch.no_grad()
    def decode_frames(self, latents, chunk: int = 32):
        """latents [B, F, C, h, w] -> uint8 [B, F, H, W, 3] (generate.py:238-244)."""
        B, F = latents.shape[:2]
        vae = self.vae
        z = latents.permute(0, 1, 3, 4, 2).reshape(B * F, vae.seq_len, vae.latent_dim).float().contiguous()
        outs = [vae.decode(z[s:s + chunk], divisor=SCALING_FACTOR, to_uint8=True) for s in range(0, B * F, chunk)]
        return torch.cat(outs).reshape(B, F, vae.input_height, vae.input_width, 3)

    @torch.no_grad()
    def generate(self, prompt_video, actions, total_frames, noise=None, generator=None):
        lat = self.encode_prompt(prompt_video)
        lat = self.sample_latents(lat, actions, total_frames, noise=noise, generator=generator)
        return self.decode_frames(lat), lat


    # ------------------------------------------------------------------ interactive / streaming
    def stream(self, prompt_video, prompt_actions=None, generator=None):
        """Frame-at-a-time generation with a per-frame action (SURVEY 8(f).3: the "playable" use of the model): returns a
        FrameStream whose next(action) denoises ONE new frame against the sliding window and decodes only that frame."""
        return FrameStream(self, prompt_video, prompt_actions, generator)

    def pool(self, capacity, use_actions=False):
        """Interactive sessions that join and leave one batch: a StreamPool of `capacity` slots, each session a FrameStream
        of B = 1 that runs batched with the others."""
        return StreamPool(self, capacity, use_actions)


class FrameStream:
    """Interactive rollout over a Sampler: the window of the last max_frames - 1 latents (and their actions) is kept on
    the device; every next() runs clamp -> conditioning -> context pass -> (steps+1) DDIM steps for one frame (one CUDA
    graph replay) and one single-frame VAE decode.  Same arithmetic as Sampler.generate: with the same noise draws the
    frames are identical (tests/test_sampler_gpu.py)."""

    def __init__(self, sampler: Sampler, prompt_video, prompt_actions=None, generator=None):
        N.require_cuda(prompt_video, "prompt_video")
        self.s = sampler
        self.dev = prompt_video.device
        self.generator = generator
        lat = sampler.encode_prompt(prompt_video)                                  # [B, n, C, h, w]
        self.B, n_prompt = lat.shape[:2]
        self.shape = tuple(lat.shape[2:])
        keep = sampler.dit.max_frames - 1
        self.window = lat.reshape(self.B, n_prompt, -1).float()[:, -keep:].contiguous() if keep > 0 else lat.new_zeros((self.B, 0, sampler.frame_elems))
        self.actions = None
        if prompt_actions is not None:
            a = prompt_actions.to(self.dev, torch.float32)
            if a.shape[:2] != (self.B, n_prompt):
                raise RuntimeError(f"prompt_actions must be [B={self.B}, n_prompt={n_prompt}, A], got {tuple(a.shape)}")
            self.actions = a[:, -keep:].contiguous() if keep > 0 else a[:, :0]
        self.frames_generated = 0
        if sampler.use_graph and sampler._stream is None:
            sampler._stream = torch.cuda.Stream(device=self.dev)

    @torch.no_grad()
    def next(self, action=None, noise=None, decode=True):
        """action: [B, A] (or [A]) for the frame to generate - required iff the stream was opened with prompt_actions;
        noise: optional [B, C, h, w] N(0,1) draws.  Returns (uint8 frame [B, H, W, 3] or None, latent [B, C, h, w])."""
        s, dev, B = self.s, self.dev, self.B
        n = s.frame_elems
        if (action is None) != (self.actions is None):
            raise RuntimeError("FrameStream.next: pass an action iff the stream was opened with prompt_actions")
        act_win = None
        if action is not None:
            a = action.to(dev, torch.float32).reshape(-1, action.shape[-1])
            if a.shape[0] == 1 and B > 1:
                a = a.expand(B, -1)
            act_win = torch.cat([self.actions, a.unsqueeze(1)], dim=1)
        if noise is not None:
            chunk = noise.to(device=dev, dtype=torch.float32).reshape(B, n).contiguous()
        else:
            chunk = torch.randn((B, n), device=dev, generator=self.generator)
        stream = s._stream if s.use_graph else torch.cuda.current_stream(dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev), torch.cuda.stream(stream):
            new = s._denoise_frame(self.window, chunk, act_win, stream).clone()
        torch.cuda.current_stream(dev).wait_stream(stream)
        keep = s.dit.max_frames - 1
        if keep > 0:
            self.window = torch.cat([self.window, new.unsqueeze(1)], dim=1)[:, -keep:].contiguous()
            if act_win is not None:
                self.actions = act_win[:, -keep:].contiguous()
        self.frames_generated += 1
        latent = new.reshape(B, *self.shape)
        frame = s.decode_frames(latent.unsqueeze(1))[:, 0] if decode else None
        return frame, latent


class StreamPool:
    """A fixed set of `capacity` slots, each holding one interactive session (a B = 1 FrameStream's state: the last
    max_frames - 1 latents and actions on the device).  step() generates one frame for every open session in one batched
    call: the pool's own (capacity, max_frames) DiT plan with per-slot window lengths attached
    (gtav_dit_plan_set_window_lengths), so a session that joined recently runs its short, left-padded window next to full
    ones.  Free slots run as length-1 windows and their results are dropped; the batch never changes shape, so one captured
    frame graph serves every step.  Each session gets what a B = 1 FrameStream with the same prompt, actions and noise gives
    (tests/test_stream_pool_gpu.py): bit for bit with the tiled GEMMs, and within the frame cache's bounds on the default
    path, whose GEMM kernels depend on the row count."""

    def __init__(self, sampler: Sampler, capacity: int, use_actions: bool = False):
        capacity = int(capacity)
        if capacity < 1:
            raise RuntimeError(f"StreamPool: capacity must be at least 1, got {capacity}")
        self.s = sampler
        self.capacity = capacity
        self.use_actions = bool(use_actions)
        self.dev = sampler.dit.final_layer.linear.weight.device
        self._slots = [None] * capacity         # session id per slot
        self._sessions = {}                     # id -> dict(slot, window [k, n], actions [k, A] or None, generator, shape)
        self._next_id = 0
        self._ctx = None
        sampler.dit._dependants.add(self)       # dropped with the DiT's plans when the weights are re-packed

    # ------------------------------------------------------------------ sessions
    @torch.no_grad()
    def open(self, prompt_video, prompt_actions=None, generator=None):
        """prompt_video [n, 3, H, W] in [0, 1] (n >= 1); prompt_actions [n, A], required iff the pool uses actions.
        Returns the new session's id."""
        N.require_cuda(prompt_video, "prompt_video")
        s, vae = self.s, self.s.vae
        want = (3, vae.input_height, vae.input_width)
        if prompt_video.dim() != 4 or prompt_video.shape[0] < 1 or tuple(prompt_video.shape[1:]) != want:
            raise RuntimeError(f"StreamPool.open: prompt_video must be [n >= 1, {want[0]}, {want[1]}, {want[2]}], "
                               f"got {tuple(prompt_video.shape)}")
        if (prompt_actions is None) == self.use_actions:
            raise RuntimeError("StreamPool.open: pass prompt_actions iff the pool was created with use_actions=True")
        if None not in self._slots:
            raise RuntimeError(f"StreamPool.open: all {self.capacity} slots are taken")
        n_prompt = prompt_video.shape[0]
        keep = s.dit.max_frames - 1
        actions = None
        if prompt_actions is not None:
            actions = prompt_actions.to(self.dev, torch.float32)
            if tuple(actions.shape) != (n_prompt, s.dit.external_cond_dim):
                raise RuntimeError(f"StreamPool.open: prompt_actions must be [n_prompt={n_prompt}, "
                                   f"{s.dit.external_cond_dim}], got {tuple(prompt_actions.shape)}")
            actions = actions[n_prompt - keep:] if keep > 0 else actions[:0]
        lat = s.encode_prompt(prompt_video.to(self.dev)[None])[0]                 # [n, C, h, w]
        window = lat.reshape(n_prompt, -1).float()
        window = window[n_prompt - keep:] if keep > 0 else window[:0]
        sid = self._next_id
        self._next_id += 1
        slot = self._slots.index(None)
        self._slots[slot] = sid
        self._sessions[sid] = dict(slot=slot, window=window.contiguous(), generator=generator, shape=tuple(lat.shape[1:]),
                                   actions=None if actions is None else actions.contiguous())
        return sid

    def close(self, sid):
        """Frees the session's slot for the next open()."""
        self._session(sid, "close")
        self._slots[self._sessions.pop(sid)["slot"]] = None

    def _session(self, sid, what):
        if sid not in self._sessions:
            raise RuntimeError(f"StreamPool.{what}: no open session {sid!r}")
        return self._sessions[sid]

    @property
    def sessions(self):
        """Ids of the open sessions, in slot order."""
        return [sid for sid in self._slots if sid is not None]

    # ------------------------------------------------------------------ plan / sampler handle of the pool
    def _context(self):
        s = self.s
        s.dit._pack()                           # a weight change releases the plans and (_invalidate) our handle
        if self._ctx is None:
            lengths = torch.ones(self.capacity, dtype=torch.int32, device=self.dev)
            with torch.cuda.device(self.dev):
                self._ctx = s._new_context(self.capacity, s.dit.max_frames, self.dev, lengths=lengths, owner=("pool", id(self)))
        return self._ctx

    def _release_context(self):
        if self._ctx is not None:
            torch.cuda.synchronize()
            N.load().gtav_sampler_destroy(self._ctx["h"])
            self._ctx = None

    def _invalidate(self):
        """Called by the DiT before it releases its plans: the sampler handle and its graph refer to the pool's plan."""
        self._release_context()

    def __del__(self):
        try:
            self._release_context()
            self.s.dit._drop_plans(("pool", id(self)))
        except Exception:
            pass

    # ------------------------------------------------------------------ one frame for every session
    @torch.no_grad()
    def step(self, actions=None, noise=None, decode=True):
        """actions: {session id: [A]} for every open session iff the pool uses actions; noise: optional {session id:
        [C, h, w]} N(0, 1) draws (a session without an entry draws from its own generator, as a B = 1 FrameStream).
        Returns {session id: (uint8 frame [H, W, 3] or None, latent [C, h, w])}."""
        s, dev, cap = self.s, self.dev, self.capacity
        n = s.frame_elems
        actions = {} if actions is None else dict(actions)
        noise = {} if noise is None else dict(noise)
        for sid in list(actions) + list(noise):
            self._session(sid, "step")
        open_ids = self.sessions
        if not self.use_actions and actions:
            raise RuntimeError("StreamPool.step: the pool was created without actions; pass none")
        if self.use_actions and set(actions) != set(open_ids):
            raise RuntimeError(f"StreamPool.step: an action is needed for every open session; missing "
                               f"{sorted(set(open_ids) - set(actions))}")
        if not open_ids:
            return {}
        ctx = self._context()
        T = s.dit.max_frames
        keep = T - 1
        lens = [1] * cap
        ctx_lat = torch.zeros((cap, T - 1, n), dtype=torch.float32, device=dev)      # left-padded windows
        act_win = torch.zeros((cap, T, s.dit.external_cond_dim), dtype=torch.float32, device=dev) if self.use_actions else None
        chunk = torch.zeros((cap, n), dtype=torch.float32, device=dev)
        for sid in open_ids:
            ses = self._sessions[sid]
            b, k = ses["slot"], ses["window"].shape[0]
            lens[b] = k + 1
            if k:
                ctx_lat[b, T - 1 - k:] = ses["window"]
            if act_win is not None:
                a = actions[sid].to(dev, torch.float32).reshape(-1)
                if k:
                    act_win[b, T - 1 - k: T - 1] = ses["actions"]
                act_win[b, T - 1] = a
            if sid in noise:
                chunk[b] = noise[sid].to(device=dev, dtype=torch.float32).reshape(n)
            else:
                chunk[b] = torch.randn((1, n), device=dev, generator=ses["generator"])[0]
        if s.use_graph and s._stream is None:
            s._stream = torch.cuda.Stream(device=dev)
        stream = s._stream if s.use_graph else torch.cuda.current_stream(dev)
        stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.device(dev), torch.cuda.stream(stream):
            # on the stream that replays the frame graph, so the graph reads this step's lengths
            ctx["lengths"].copy_(torch.tensor(lens, dtype=torch.int32))
            new = s._denoise_frame(ctx_lat, chunk, act_win, stream, ctx=ctx).clone()
        torch.cuda.current_stream(dev).wait_stream(stream)
        out = {}
        for sid in open_ids:
            ses = self._sessions[sid]
            b = ses["slot"]
            if keep > 0:
                ses["window"] = torch.cat([ses["window"], new[b][None]])[-keep:].contiguous()
                if act_win is not None:
                    ses["actions"] = act_win[b, T - 1 - (lens[b] - 1):].clone()[-keep:].contiguous()
            out[sid] = (None, new[b].reshape(ses["shape"]))
        if decode:
            lat = torch.stack([out[sid][1] for sid in open_ids])
            frames = s.decode_frames(lat.unsqueeze(1))[:, 0]
            out = {sid: (frames[i], out[sid][1]) for i, sid in enumerate(open_ids)}
        return out
