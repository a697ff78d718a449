"""ctypes binding of libgtav_b200.so (include/gtav_b200.h).  There is no fallback: if the library is
missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libgtav_b200.so")

(EPI_STORE, EPI_BIAS, EPI_BIAS_GELU_TANH, EPI_BIAS_GELU_ERF, EPI_BIAS_SILU, EPI_BIAS_GATE_RES, EPI_BIAS_RES,
 EPI_BIAS_RES_SILU) = range(8)

# every symbol include/gtav_b200.h declares (tests check the .so exports exactly these)
EXPORTS = [
    "gtav_last_error", "gtav_abi_version", "gtav_gemm_bf16", "gtav_gemm_skinny_bf16", "gtav_gemm_skinny_tagged_bf16", "gtav_gemm_skinny_fused_bf16",
    "gtav_gemm_skinny_workspace_bytes",
    "gtav_dit_context", "gtav_dit_last_frame", "gtav_attention_temporal_last", "gtav_ln_modulate", "gtav_ln_affine",
    "gtav_attention_seq", "gtav_attention_temporal", "gtav_ddim_update", "gtav_dit_create", "gtav_dit_destroy",
    "gtav_dit_mod_width", "gtav_dit_workspace_bytes", "gtav_dit_plan_create", "gtav_dit_plan_destroy",
    "gtav_dit_conditioning", "gtav_dit_backbone", "gtav_dit_forward", "gtav_vae_create", "gtav_vae_destroy",
    "gtav_vae_workspace_bytes", "gtav_vae_plan_create", "gtav_vae_plan_destroy", "gtav_vae_encode", "gtav_vae_encode_moments", "gtav_vae_decode",
    "gtav_sampler_cond_rows", "gtav_sampler_scratch_bytes", "gtav_sampler_create", "gtav_sampler_destroy",
    "gtav_sampler_run_frame", "gtav_noise_clamp", "gtav_attention_temporal_ragged", "gtav_attention_temporal_last_ragged",
    "gtav_dit_plan_set_window_lengths",
]

SAMPLER_GRAPH, SAMPLER_FRAME_CACHE = 1, 2      # gtav_sampler_flags

vp = C.c_void_p


class DitConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("depth", "hidden", "heads", "grid_h", "grid_w", "patch", "in_channels",
                                       "act_dim", "max_frames")]


class DitHalf(C.Structure):
    _fields_ = [(n, vp) for n in ("qkv_w", "out_w", "out_b", "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class DitWeights(C.Structure):
    _fields_ = [(n, vp) for n in ("patch_w", "patch_b", "t0_w", "t0_b", "t2_w", "t2_b", "act_w", "act_b", "ada_w",
                                  "ada_b", "final_w", "final_b", "temb_freqs", "rot_spatial", "rot_temporal")] + \
               [("halves", C.POINTER(DitHalf))]


class VaeConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("dim", "heads", "enc_depth", "dec_depth", "latent_dim", "patch", "seq_h",
                                       "seq_w")]


class VaeBlock(C.Structure):
    _fields_ = [(n, vp) for n in ("norm1_w", "norm1_b", "norm2_w", "norm2_b", "qkv_w", "qkv_b", "proj_w", "proj_b",
                                  "fc1_w", "fc1_b", "fc2_w", "fc2_b")]


class VaeWeights(C.Structure):
    _fields_ = [(n, vp) for n in ("patch_w", "patch_b", "enc_norm_w", "enc_norm_b", "dec_norm_w", "dec_norm_b",
                                  "quant_w", "quant_b", "post_w", "post_b", "pred_w", "pred_b", "rot")] + \
               [("enc", C.POINTER(VaeBlock)), ("dec", C.POINTER(VaeBlock))]


_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library (after torch, so libcudart resolves to the copy torch loaded)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python ai-generated-gtav_b200/build.py` "
            "(gtav_b200 has no CPU or PyTorch fallback)")
    import torch  # noqa: F401  (loads libcudart.so.12 into the process first)
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    i, sz, i64p, fp, ip = C.c_int, C.c_size_t, vp, vp, vp
    lib.gtav_last_error.restype = C.c_char_p
    lib.gtav_last_error.argtypes = []
    lib.gtav_abi_version.restype = i
    sig = {
        "gtav_gemm_bf16": [vp, i, vp, i, vp, i, i, i, i, i, vp, vp, i, vp, i, ip, i, i, vp],
        "gtav_gemm_skinny_bf16": [vp, i, vp, i, vp, i, i, i, i, i, vp, vp, i, vp, i, ip, i, i, vp, vp, vp],
        "gtav_gemm_skinny_tagged_bf16": [vp, i, vp, i, vp, i, i, i, i, i, vp, vp, i, vp, i, ip, i, i, vp, i, vp],
        "gtav_gemm_skinny_fused_bf16": [vp, i, vp, i, vp, i, i, i, i, vp, vp, i, vp, i, ip, i, vp, ip, i, vp, vp, i, i, i, vp, fp,
                                        i, i, i, vp],
        "gtav_dit_context": [vp, vp, i, ip, vp],
        "gtav_dit_last_frame": [vp, vp, i, ip, vp, vp],
        "gtav_ln_modulate": [vp, vp, i, i, vp, i, i, i, ip, i, vp],
        "gtav_ln_affine": [vp, vp, i, i, fp, fp, vp],
        "gtav_attention_seq": [vp, vp, i, i, i, fp, i, vp],
        "gtav_attention_temporal": [vp, vp, i, i, i, i, fp, vp],
        "gtav_attention_temporal_last": [vp, vp, i, i, i, i, fp, vp, vp],
        "gtav_attention_temporal_ragged": [vp, vp, i, i, i, i, fp, ip, vp, vp],
        "gtav_attention_temporal_last_ragged": [vp, vp, i, i, i, i, fp, ip, vp, vp],
        "gtav_dit_plan_set_window_lengths": [vp, ip],
        "gtav_ddim_update": [fp, vp, fp, i, i, fp, fp, ip, vp],
        "gtav_dit_create": [C.POINTER(DitConfig), C.POINTER(DitWeights), C.POINTER(vp)],
        "gtav_dit_destroy": [vp],
        "gtav_dit_mod_width": [vp],
        "gtav_dit_plan_create": [vp, i, i, i, vp, sz, vp, C.POINTER(vp)],
        "gtav_dit_plan_destroy": [vp],
        "gtav_dit_conditioning": [vp, i64p, fp, vp],
        "gtav_dit_backbone": [vp, vp, i, ip, vp, vp],
        "gtav_dit_forward": [vp, vp, i, i64p, fp, vp, vp],
        "gtav_vae_create": [C.POINTER(VaeConfig), C.POINTER(VaeWeights), C.POINTER(vp)],
        "gtav_vae_destroy": [vp],
        "gtav_vae_plan_create": [vp, i, vp, sz, C.POINTER(vp)],
        "gtav_vae_plan_destroy": [vp],
        "gtav_vae_encode": [vp, vp, i, fp, C.c_float, i, vp],
        "gtav_vae_encode_moments": [vp, vp, i, fp, fp, vp],
        "gtav_vae_decode": [vp, fp, C.c_float, vp, i, vp],
        "gtav_sampler_cond_rows": [i, i, i],
        "gtav_sampler_create": [vp, i, i, i, i, fp, vp, fp, ip, vp, sz, i, vp, C.POINTER(vp)],
        "gtav_sampler_destroy": [vp],
        "gtav_sampler_run_frame": [vp, i, vp],
        "gtav_noise_clamp": [fp, fp, C.c_long, i, i, C.c_float, vp],
    }
    for name, args in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = None if name.endswith("_destroy") else i
    lib.gtav_dit_workspace_bytes.argtypes = [vp, i, i, i]
    lib.gtav_dit_workspace_bytes.restype = sz
    lib.gtav_vae_workspace_bytes.argtypes = [vp, i]
    lib.gtav_vae_workspace_bytes.restype = sz
    lib.gtav_gemm_skinny_workspace_bytes.argtypes = [i]
    lib.gtav_gemm_skinny_workspace_bytes.restype = sz
    lib.gtav_sampler_scratch_bytes.argtypes = [i, i, i]
    lib.gtav_sampler_scratch_bytes.restype = sz
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().gtav_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def ptr(t) -> int | None:
    """Raw device address of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda(t, name: str):
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: gtav_b200 runs only on sm_100a GPUs (no CPU fallback)")


def param_signature(module):
    """(data_ptr, version) of every parameter: a change of either means the packed bf16 copies are stale.
    Inference tensors (modules built or moved under torch.inference_mode, as the reference's generate.py does for
    load_models / main) have no version counter: they get version -1 and in-place edits of them are only seen through
    load_state_dict / .to() (which mark the module dirty) or an explicit repack()."""
    sig = []
    for p in module.parameters():
        sig.append((p.data_ptr(), -1 if p.is_inference() else p._version))
    return tuple(sig)
