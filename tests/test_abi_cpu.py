"""CPU-side checks: the C-ABI library loads and exports every symbol include/gtav_b200.h declares, the
drop-in modules keep the reference's state_dict contract, and the product refuses to run without CUDA."""
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as ge
    ge.build()
    import gtav_b200._native as N
    return N


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "gtav_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(gtav_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_exactly_the_header(native):
    lib = native.load()
    decl = declared_symbols()
    assert decl == sorted(native.EXPORTS)
    for s in decl:
        assert hasattr(lib, s), s
    out = subprocess.run(["nm", "-D", "--defined-only", native.LIB_PATH], capture_output=True, text=True).stdout
    exported = sorted(l.split()[-1] for l in out.splitlines() if " T " in l)
    assert exported == decl, set(exported) ^ set(decl)          # nothing else leaks out of the .so
    assert lib.gtav_abi_version() == 5


def test_library_is_sm100a_tcgen05(native):
    sass = subprocess.run(["cuobjdump", "-sass", native.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in sass
    for mnemonic in ("UTCHMMA", "UTMALDG", "LDTM"):             # tcgen05.mma, TMA load, tcgen05.ld
        assert mnemonic in sass, mnemonic


def test_host_side_argument_checks_need_no_gpu(native):
    lib = native.load()
    assert lib.gtav_sampler_cond_rows(2, 5, 100) == 2 * 4 + 2 * 101
    assert lib.gtav_sampler_scratch_bytes(2, 5, 100) > 0
    cfg = native.DitConfig(16, 768, 12, 9, 16, 2, 16, 25, 5)
    import ctypes as C
    h = native.vp()
    rc = lib.gtav_dit_create(C.byref(cfg), C.byref(native.DitWeights()), C.byref(h))
    assert rc != 0 and b"unsupported geometry" in lib.gtav_last_error()
    # the tagged weight-streaming GEMM refuses a missing workspace and a parity outside {0, 1} before touching the device
    args = [None, 1024, None, 1024, None, 1024, 144, 1024, 1024, native.EPI_STORE, None, None, 0, None, 0, None, 144, 0]
    assert lib.gtav_gemm_skinny_tagged_bf16(*args, None, 1, None) != 0 and b"workspace" in lib.gtav_last_error()
    assert lib.gtav_gemm_skinny_tagged_bf16(*args, 4096, 2, None) != 0 and b"parity" in lib.gtav_last_error()
    assert lib.gtav_gemm_skinny_workspace_bytes(144) == 160 * 144 * 128 * 4
    # the fused-reduce entry point: the same host checks, then skinny_prepare's refusals of a shape the fused mode cannot
    # run, all before any descriptor or launch (the non-null device addresses below are never dereferenced)
    fake = 4096

    def fused(mode, N, ws=fake, counters=None, ctx_frames=0, parity=0):
        return lib.gtav_gemm_skinny_fused_bf16(fake, 1024, fake, 1024, fake, N, 144, N, 1024, fake, fake, N, fake, N, None, 4, ws,
                                               counters, mode, fake, fake, 6 * 1024, 0, 1024, fake, fake, ctx_frames, 144, parity,
                                               None)
    assert fused(1, 1024, ws=None) != 0 and b"workspace" in lib.gtav_last_error()
    assert fused(1, 1024, parity=2) != 0 and b"parity" in lib.gtav_last_error()
    assert fused(1, 1024, parity=-1) != 0 and b"counters" in lib.gtav_last_error()
    assert fused(0, 1024) != 0 and b"mode" in lib.gtav_last_error()
    assert fused(1, 2048) != 0 and b"fused reduce mode 1 does not fit" in lib.gtav_last_error()      # LayerNorm: N = 1024 only
    assert fused(2, 3072, ctx_frames=8) != 0 and b"fused reduce mode 2 does not fit" in lib.gtav_last_error()   # <= 7 cached frames


def test_dit_state_dict_contract():
    from gtav_b200.model.dit import DiT_models
    from oracle.weights import DiTConfig, make_dit_state
    m = DiT_models["DiT-S/2"]()
    sd = m.state_dict()
    ref = make_dit_state(DiTConfig(), seed=0)
    assert len(sd) == 334 and set(sd) == set(ref)
    for k, v in ref.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    assert sum(p.numel() for p in m.parameters()) == 607_943_792
    assert m.max_frames == 5 and m.patch_size == 2
    # default init: adaLN of every block is zero (blocks are identities), like the reference
    assert float(sd["blocks.3.t_adaLN_modulation.1.weight"].abs().max()) == 0.0
    assert torch.equal(sd["blocks.0.s_attn.rotary_emb.freqs"], sd["spatial_rotary_emb.freqs"])
    assert torch.allclose(sd["spatial_rotary_emb.freqs"], ref["spatial_rotary_emb.freqs"])
    assert torch.allclose(sd["temporal_rotary_emb.freqs"], ref["temporal_rotary_emb.freqs"])


def test_vae_state_dict_contract():
    from gtav_b200.model.vae import VAE_models
    from oracle.weights import VAEConfig, make_vae_state
    m = VAE_models["vit-l-20-shallow-encoder"]()
    sd = m.state_dict()
    ref = make_vae_state(VAEConfig(), seed=0)
    assert len(sd) == 228 and set(sd) == set(ref)
    for k, v in ref.items():
        assert tuple(sd[k].shape) == tuple(v.shape), k
    assert sum(p.numel() for p in m.parameters()) == 229_246_160
    assert m.patch_size == 20 and m.seq_len == 576


def test_safetensors_roundtrip_like_load_model(tmp_path):
    """generate.py loads checkpoints with safetensors.torch.load_model; shared rotary tensors must not trip it."""
    from safetensors.torch import load_model, save_model
    from gtav_b200.model.dit import DiT
    a, b = DiT(depth=1), DiT(depth=1)
    with torch.no_grad():
        a.final_layer.linear.weight.normal_()
    path = str(tmp_path / "dit.safetensors")
    save_model(a, path)
    missing, unexpected = load_model(b, path)
    assert not missing and not unexpected
    assert torch.equal(a.final_layer.linear.weight, b.final_layer.linear.weight)


def test_product_has_no_cpu_path():
    from gtav_b200.model.dit import DiT
    from gtav_b200.model.vae import VAE_models
    from gtav_b200.train_dit import denoise_step
    m = DiT(depth=1)
    with pytest.raises(RuntimeError, match="CUDA"):
        m(torch.zeros(1, 1, 16, 18, 32), torch.zeros(1, 1, dtype=torch.long))
    with pytest.raises(RuntimeError, match="CUDA"):
        denoise_step(m, torch.zeros(1, 2, 16, 18, 32), None, 3, 15, torch.linspace(0, 999, 11), torch.ones(1000))
    v = VAE_models["vit-l-20-shallow-encoder"](enc_depth=1, dec_depth=1) if False else None
    assert v is None


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "ai-generated-gtav_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text or f == "build.py", os.path.join(dirpath, f)


def test_schedule_dropin_matches_oracle():
    from gtav_b200.utils import sigmoid_beta_schedule
    from oracle.reference_port import sigmoid_beta_schedule as ref
    assert torch.equal(sigmoid_beta_schedule(1000), ref(1000))
    assert torch.equal(sigmoid_beta_schedule(50, start=-2, end=4, tau=0.9), ref(50, start=-2.0, end=4.0, tau=0.9))


def test_trainer_inference_contract_cpu():
    """The inference-side DiffusionTrainer surface (reference train_dit.py:128-157, 288-552) exists with the reference's
    defaults; nothing here touches the GPU."""
    import dataclasses
    import inspect
    from gtav_b200.train_dit import DiffusionTrainer, TrainingConfig, denoise_step
    cfg = TrainingConfig()
    assert (cfg.ddim_noise_steps, cfg.ddim_noise_steps_inference, cfg.ctx_max_noise_idx, cfg.noise_abs_max, cfg.n_prompt_frames,
            cfg.use_action_conditioning, cfg.model_name, cfg.seed) == (16, 16, 3, 20.0, 1, True, "dit", 42)
    assert TrainingConfig.from_dict(dict(ddim_noise_steps=8, learning_rate=1e-5)).ddim_noise_steps == 8   # unknown keys ignored
    for name in ("register_buffers", "encode_frames", "decode_frames", "predict", "predict_noise", "train"):
        assert callable(getattr(DiffusionTrainer, name))
    assert list(inspect.signature(DiffusionTrainer.decode_frames).parameters)[:3] == ["self", "frames", "num_frames"]
    assert list(inspect.signature(DiffusionTrainer.predict).parameters)[:5] == ["self", "test_loader", "epoch", "global_step", "num_frames"]
    assert list(inspect.signature(denoise_step).parameters) == ["dit_model", "x_noisy", "actions", "noise_idx", "stabilization_level",
                                                                "noise_range", "alphas_cumprod", "start_frame", "dtype"]


def test_frame_stream_contract_cpu():
    from gtav_b200.sampler import FrameStream, Sampler
    import inspect
    assert list(inspect.signature(FrameStream.next).parameters) == ["self", "action", "noise", "decode"]
    assert callable(Sampler.stream)


def test_modules_built_under_inference_mode_have_a_signature():
    """The reference's generate.py builds and moves both models under @torch.inference_mode (load_models / main): their
    parameters are inference tensors, which have no version counter - the pack signature must not touch it."""
    import torch
    from gtav_b200.model.dit import DiT
    from gtav_b200.model.vae import AutoencoderKL
    with torch.inference_mode():
        dit = DiT(depth=1)
        vae = AutoencoderKL(latent_dim=16, patch_size=20, enc_dim=1024, enc_depth=1, enc_heads=16, dec_dim=1024, dec_depth=1,
                            dec_heads=16, input_height=360, input_width=640)
        assert all(p.is_inference() for p in dit.parameters())
        s1, s2 = dit._signature(), vae._signature()
        assert len(s1) == len(list(dit.parameters())) and len(s2) == len(list(vae.parameters()))
        assert all(v == -1 for _, v in s1)
        # load_state_dict and .to() mark the packed copies stale even where no version counter can show it
        assert not dit._dirty
        dit.load_state_dict(dit.state_dict())
        assert dit._dirty
    vae._dirty = False
    vae.to(torch.float32)
    assert vae._dirty
    dit._dirty = False
    dit.repack()
    assert dit._dirty
