"""Drop-in for the reference's model/dit.py: same constructor, attributes, state_dict keys and
`DiT.forward(x, t, external_cond)` contract (reference model/dit.py:228-392), but the module only
HOLDS parameters - the arithmetic runs in libgtav_b200.so (tcgen05 GEMMs with fused epilogues,
fused-rotary attention, LayerNorm+modulate kernels) through the C ABI of include/gtav_b200.h.

Differences a caller can observe, all documented in DESIGN.md:
  * CUDA (sm_100a) tensors only - a CPU tensor raises instead of falling back;
  * the result is always bf16, i.e. what the reference returns under torch.autocast("cuda", bf16),
    which is how generate.py and denoise_step call it (train_dit.py:102-107);
  * inference only (no autograd graph is recorded).
"""
from __future__ import annotations

import ctypes as C
import math
import weakref

import torch
from torch import nn

try:  # imported as gtav_b200.model.dit
    from .. import _native as N
except ImportError:  # imported as top-level `model.dit` with the package directory on sys.path
    import _native as N


MAX_FRAMES = 32      # longest sliding window the temporal attention kernels run (csrc/attn_temporal_long.cu)


def _check_max_frames(max_frames):
    if not 1 <= max_frames <= MAX_FRAMES:
        raise RuntimeError(f"gtav_b200.DiT: max_frames={max_frames} is unsupported: the temporal attention kernels run "
                           f"sliding windows of 1 to {MAX_FRAMES} frames")


class _Rotary(nn.Module):
    """Holds the `freqs` parameter of the reference's RotaryEmbedding so checkpoints load unchanged
    (model/rotary_embedding_torch.py:118-136); the angle tables are built in DiT._pack."""

    def __init__(self, freqs: torch.Tensor):
        super().__init__()
        self.freqs = nn.Parameter(freqs, requires_grad=False)


class _Holder(nn.Module):
    """Attribute container whose children carry the reference's parameter names."""


def _linear(i, o, bias=True):
    return nn.utils.skip_init(nn.Linear, i, o, bias=bias)


class DiT(nn.Module):
    def __init__(self, input_h=18, input_w=32, patch_size=2, in_channels=16, hidden_size=1024, depth=12, num_heads=16,
                 mlp_ratio=4.0, external_cond_dim=25, max_frames=5):
        super().__init__()
        _check_max_frames(max_frames)
        self.in_channels = in_channels
        self.out_channels = in_channels
        self.patch_size = patch_size
        self.num_heads = num_heads
        self.max_frames = max_frames
        self.input_h, self.input_w = input_h, input_w
        self.hidden_size, self.depth = hidden_size, depth
        self.external_cond_dim = external_cond_dim
        D, Hm = hidden_size, int(hidden_size * mlp_ratio)
        head_dim = D // num_heads

        self.x_embedder = _Holder()
        self.x_embedder.proj = nn.utils.skip_init(nn.Conv2d, in_channels, D, kernel_size=patch_size, stride=patch_size)
        self.x_embedder.grid_size = (input_h // patch_size, input_w // patch_size)
        self.x_embedder.patch_size = (patch_size, patch_size)
        self.t_embedder = _Holder()
        self.t_embedder.mlp = nn.Sequential(_linear(256, D), nn.SiLU(), _linear(D, D))
        sdim = head_dim // 2
        self.spatial_rotary_emb = _Rotary(torch.linspace(1.0, 256 / 2, sdim // 2) * math.pi)
        self.temporal_rotary_emb = _Rotary(1.0 / (10000 ** (torch.arange(0, head_dim, 2)[: head_dim // 2].float() / head_dim)))
        self.external_cond = _linear(external_cond_dim, D) if external_cond_dim > 0 else nn.Identity()

        blocks = []
        for _ in range(depth):
            b = _Holder()
            for h, rot in (("s", self.spatial_rotary_emb), ("t", self.temporal_rotary_emb)):
                attn = _Holder()
                attn.to_qkv = _linear(D, 3 * D, bias=False)
                attn.to_out = _linear(D, D)
                attn.rotary_emb = rot
                mlp = _Holder()
                mlp.fc1 = _linear(D, Hm)
                mlp.fc2 = _linear(Hm, D)
                setattr(b, f"{h}_attn", attn)
                setattr(b, f"{h}_mlp", mlp)
                setattr(b, f"{h}_adaLN_modulation", nn.Sequential(nn.SiLU(), _linear(D, 6 * D)))
            blocks.append(b)
        self.blocks = nn.ModuleList(blocks)
        self.final_layer = _Holder()
        self.final_layer.linear = _linear(D, patch_size * patch_size * in_channels)
        self.final_layer.adaLN_modulation = nn.Sequential(nn.SiLU(), _linear(D, 2 * D))
        self.initialize_weights()

        self._engine = None      # (handle, keep-alive tensors)
        self._packed_sig = None
        self._packed_max_frames = None
        self._plans = {}
        self._dirty = False
        self._pack_generation = 0
        self._dependants = weakref.WeakSet()     # Samplers holding handles / CUDA graphs built on this module's plans
        self.register_load_state_dict_post_hook(lambda module, _keys: module._mark_dirty())

    # ------------------------------------------------------------------ init (same distributions as dit.py:304-326)
    @torch.no_grad()
    def initialize_weights(self):
        for m in self.modules():
            if isinstance(m, nn.Linear):
                m.weight.normal_(std=0.02)
                if m.bias is not None:
                    m.bias.zero_()
        self.x_embedder.proj.weight.normal_(std=0.02)
        self.x_embedder.proj.bias.zero_()
        self.t_embedder.mlp[0].weight.normal_(std=0.01)
        self.t_embedder.mlp[2].weight.normal_(std=0.01)
        for b in self.blocks:
            for h in ("s", "t"):
                lin = getattr(b, f"{h}_adaLN_modulation")[-1]
                lin.weight.zero_()
                lin.bias.zero_()
        self.final_layer.adaLN_modulation[-1].weight.normal_(std=0.01)
        self.final_layer.adaLN_modulation[-1].bias.zero_()
        self.final_layer.linear.weight.normal_(std=0.001)
        self.final_layer.linear.bias.zero_()

    # ------------------------------------------------------------------ weight packing
    def _signature(self):
        return N.param_signature(self)

    def _mark_dirty(self, *_):
        self._dirty = True

    def _apply(self, fn, *a, **k):          # .to() / .cuda() / .half(): new storage -> repack on the next call
        self._dirty = True
        return super()._apply(fn, *a, **k)

    def repack(self):
        """Force a re-pack of the bf16 weights on the next call (after editing parameters in place in a way the version
        counters cannot show, e.g. on inference tensors)."""
        self._dirty = True

    def _release(self):
        lib = N.load()
        # sampler handles and their captured graphs point into the plans' workspaces and at the packed weights: they
        # go first (the Sampler rebuilds them on its next call)
        for dep in list(self._dependants):
            dep._invalidate()
        for plan, _ws in self._plans.values():
            lib.gtav_dit_plan_destroy(plan)
        self._plans = {}
        if self._engine is not None:
            lib.gtav_dit_destroy(self._engine[0])
            self._engine = None

    def __del__(self):
        try:
            self._release()
        except Exception:
            pass

    @torch.no_grad()
    def _pack(self):
        """fp32 parameters -> bf16 (RNE, the cast autocast applies) laid out for the kernels; the 33
        adaLN linears are concatenated into one [depth*2*6D + 2D, D] matrix so that all modulation
        vectors come out of a single GEMM."""
        sig = self._signature()
        # max_frames is a plain attribute the reference's generate.py sets after construction; the engine and its
        # temporal rotary table are built for the value at packing time, so a new value re-packs like a weight change
        if self._engine is not None and sig == self._packed_sig and self.max_frames == self._packed_max_frames \
                and not self._dirty:
            return
        _check_max_frames(self.max_frames)
        self._release()
        self._dirty = False
        self._pack_generation += 1
        lib = N.load()
        dev = self.final_layer.linear.weight.device
        if dev.type != "cuda":
            raise RuntimeError("gtav_b200.DiT: parameters must live on a CUDA device (call .to('cuda')); no CPU fallback")
        bf = lambda p: p.detach().to(device=dev, dtype=torch.bfloat16).contiguous()
        keep = []

        def k(t):
            keep.append(t)
            return t.data_ptr()

        D = self.hidden_size
        gh, gw = self.x_embedder.grid_size
        halves = (N.DitHalf * (2 * self.depth))()
        ada_w, ada_b = [], []
        for n, b in enumerate(self.blocks):
            for j, h in enumerate(("s", "t")):
                attn, mlp = getattr(b, f"{h}_attn"), getattr(b, f"{h}_mlp")
                hh = halves[2 * n + j]
                hh.qkv_w = k(bf(attn.to_qkv.weight))
                hh.out_w, hh.out_b = k(bf(attn.to_out.weight)), k(bf(attn.to_out.bias))
                hh.fc1_w, hh.fc1_b = k(bf(mlp.fc1.weight)), k(bf(mlp.fc1.bias))
                hh.fc2_w, hh.fc2_b = k(bf(mlp.fc2.weight)), k(bf(mlp.fc2.bias))
                lin = getattr(b, f"{h}_adaLN_modulation")[-1]
                ada_w.append(lin.weight)
                ada_b.append(lin.bias)
        ada_w.append(self.final_layer.adaLN_modulation[-1].weight)
        ada_b.append(self.final_layer.adaLN_modulation[-1].bias)
        w = N.DitWeights()
        w.patch_w = k(bf(self.x_embedder.proj.weight.reshape(D, -1)))
        w.patch_b = k(bf(self.x_embedder.proj.bias))
        w.t0_w, w.t0_b = k(bf(self.t_embedder.mlp[0].weight)), k(bf(self.t_embedder.mlp[0].bias))
        w.t2_w, w.t2_b = k(bf(self.t_embedder.mlp[2].weight)), k(bf(self.t_embedder.mlp[2].bias))
        if self.external_cond_dim > 0:
            w.act_w, w.act_b = k(bf(self.external_cond.weight)), k(bf(self.external_cond.bias))
        w.ada_w = k(torch.cat([bf(x) for x in ada_w], dim=0))
        w.ada_b = k(torch.cat([bf(x) for x in ada_b], dim=0))
        w.final_w, w.final_b = k(bf(self.final_layer.linear.weight)), k(bf(self.final_layer.linear.bias))
        # tables, built with the same torch expressions the reference evaluates
        f32 = dict(device=dev, dtype=torch.float32)
        w.temb_freqs = k(torch.exp(-math.log(10000) * torch.arange(0, 128, dtype=torch.float32) / 128).to(dev))
        sf = self.spatial_rotary_emb.freqs.detach().to(**f32)
        # 32 rotary pairs per head: pairs 0..15 turn by row_pos * f[p], pairs 16..31 by col_pos * f[p-16]
        # (get_axial_freqs concatenates the row table and the column table, each angle shared by the two
        # elements of a pair - rotary_embedding_torch.py:290-317, 340)
        ah = torch.linspace(-1, 1, steps=gh, device=dev)[:, None] * sf[None]          # [gh, 16]
        aw = torch.linspace(-1, 1, steps=gw, device=dev)[:, None] * sf[None]          # [gw, 16]
        ang = torch.cat([ah[:, None].expand(gh, gw, -1), aw[None].expand(gh, gw, -1)], dim=-1).reshape(gh * gw, -1)
        assert ang.shape[1] == 32
        w.rot_spatial = k(torch.stack([ang.cos(), ang.sin()], dim=-1).contiguous())   # (cos, sin) [144, 32]
        tf = self.temporal_rotary_emb.freqs.detach().to(**f32)
        pos = torch.arange(self.max_frames, device=dev, dtype=torch.bfloat16).to(torch.float32)
        tang = pos[:, None] * tf[None]                                                 # [T, 32]
        w.rot_temporal = k(torch.stack([tang.cos(), tang.sin()], dim=-1).contiguous())
        w.halves = C.cast(halves, C.POINTER(N.DitHalf))
        keep.append(halves)
        cfg = N.DitConfig(self.depth, D, self.num_heads, gh, gw, self.patch_size, self.in_channels,
                          max(self.external_cond_dim, 0), self.max_frames)
        handle = N.vp()
        N.check(lib.gtav_dit_create(C.byref(cfg), C.byref(w), C.byref(handle)), "gtav_dit_create")
        self._engine = (handle, keep)
        self._packed_sig = sig
        self._packed_max_frames = self.max_frames

    def _plan(self, B, T, cond_rows=None, owner=None):
        """The (B, T, cond_rows) plan, shared by every caller; owner: a key of the caller's own for a plan nobody else uses
        (a StreamPool attaches window lengths to its plan)."""
        cond_rows = B * T if cond_rows is None else cond_rows
        key = (B, T, cond_rows) if owner is None else (B, T, cond_rows, owner)
        if key not in self._plans:
            lib = N.load()
            handle = self._engine[0]
            nbytes = lib.gtav_dit_workspace_bytes(handle, B, T, cond_rows)
            dev = self.final_layer.linear.weight.device
            ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
            base = (ws.data_ptr() + 1023) & ~1023
            plan = N.vp()
            with torch.cuda.device(dev):
                # the caller's current stream: the one the workspace was just allocated on and the passes will run on
                N.check(lib.gtav_dit_plan_create(handle, B, T, cond_rows, base, nbytes, N.current_stream(), C.byref(plan)),
                        "gtav_dit_plan_create")
            self._plans[key] = (plan, ws)
        return self._plans[key][0]

    def _drop_plans(self, owner):
        """Release the plans created with this owner key (pending work on them drains first)."""
        keys = [k for k in self._plans if len(k) == 4 and k[3] == owner]
        if not keys:
            return
        torch.cuda.synchronize()
        lib = N.load()
        for k in keys:
            lib.gtav_dit_plan_destroy(self._plans.pop(k)[0])

    # ------------------------------------------------------------------ forward
    @torch.no_grad()
    def forward(self, x, t, external_cond=None):
        """x: (B, T, C, H, W) latents, t: (B, T) long timesteps, external_cond: (B, T, 25) or None
        -> (B, T, C, H, W) bf16 v-prediction."""
        N.require_cuda(x, "x")
        B, T, Cc, H, W = x.shape
        if (Cc, H, W) != (self.in_channels, self.input_h, self.input_w):
            raise AssertionError(f"Input latent size ({Cc}x{H}x{W}) doesn't match model "
                                 f"({self.in_channels}x{self.input_h}x{self.input_w}).")
        if T > self.max_frames:
            raise RuntimeError(f"window of {T} frames exceeds max_frames={self.max_frames}")
        self._pack()
        lib = N.load()
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        t = t.to(device=x.device, dtype=torch.long).reshape(B * T).contiguous()
        act = None
        if torch.is_tensor(external_cond):
            if self.external_cond_dim <= 0:
                raise RuntimeError("model was built with external_cond_dim=0")
            act = external_cond.to(device=x.device, dtype=torch.float32).reshape(B * T, self.external_cond_dim).contiguous()
        out = torch.empty((B, T, Cc, H, W), dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            plan = self._plan(B, T)
            N.check(lib.gtav_dit_forward(plan, x.data_ptr(), int(x.dtype == torch.bfloat16), t.data_ptr(), N.ptr(act),
                                         out.data_ptr(), N.current_stream()), "gtav_dit_forward")
        return out


    @torch.no_grad()
    def forward_last_frame(self, x, t, external_cond=None):
        """v-prediction of the LAST frame of the window only, computed the way the sampler's frame cache does it:
        context pass over frames 0..T-2 (stores every temporal layer's K/V), then the last frame alone against that
        cache.  Equals forward(x, t, external_cond)[:, -1:] (frames before the last cannot see it: per-frame
        spatial attention, causal temporal attention - reference model/attention.py:62,127)."""
        N.require_cuda(x, "x")
        B, T, Cc, H, W = x.shape
        if T > self.max_frames:
            raise RuntimeError(f"window of {T} frames exceeds max_frames={self.max_frames}")
        self._pack()
        lib = N.load()
        if x.dtype not in (torch.float32, torch.bfloat16):
            x = x.float()
        x = x.contiguous()
        dev = x.device
        t = t.to(device=dev, dtype=torch.long).reshape(B * T).contiguous()
        act = None
        if torch.is_tensor(external_cond):
            act = external_cond.to(device=dev, dtype=torch.float32).reshape(B * T, self.external_cond_dim).contiguous()
        rows = torch.arange(B * T, dtype=torch.int32, device=dev).reshape(B, T)
        ctx_rows, last_rows = rows[:, :-1].contiguous(), rows[:, -1].contiguous()
        out = torch.empty((B, 1, Cc, H, W), dtype=torch.bfloat16, device=dev)
        is_bf16 = int(x.dtype == torch.bfloat16)
        with torch.cuda.device(dev):
            plan = self._plan(B, T)
            s = N.current_stream()
            N.check(lib.gtav_dit_conditioning(plan, t.data_ptr(), N.ptr(act), s), "gtav_dit_conditioning")
            N.check(lib.gtav_dit_context(plan, x.data_ptr(), is_bf16, ctx_rows.data_ptr(), s), "gtav_dit_context")
            N.check(lib.gtav_dit_last_frame(plan, x.data_ptr(), is_bf16, last_rows.data_ptr(), out.data_ptr(), s),
                    "gtav_dit_last_frame")
        return out


def DiT_S_2():
    return DiT(input_h=18, input_w=32, patch_size=2, hidden_size=1024, depth=16, num_heads=16, max_frames=5)


DiT_models = {"DiT-S/2": DiT_S_2}
