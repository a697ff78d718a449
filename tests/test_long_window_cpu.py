"""Sliding windows of up to 32 frames, host side: the engine, the two temporal attention entry points, the DiT module and
the CLI accept 1..32 frames and refuse longer windows with a message that states the limit, before touching a device."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as ge
    ge.build()
    import gtav_b200._native as N
    return N


def dit_create(N, max_frames, depth=2):
    """gtav_dit_create with the real geometry and no weights: it only records the configuration and the pointers."""
    lib = N.load()
    halves = (N.DitHalf * (2 * depth))()
    w = N.DitWeights()
    w.halves = C.cast(halves, C.POINTER(N.DitHalf))
    cfg = N.DitConfig(depth, 1024, 16, 9, 16, 2, 16, 0, max_frames)
    h = N.vp()
    rc = lib.gtav_dit_create(C.byref(cfg), C.byref(w), C.byref(h))
    if rc == 0:
        lib.gtav_dit_destroy(h)
    return rc


def test_dit_create_accepts_windows_up_to_32_frames(native):
    lib = native.load()
    for max_frames in (1, 5, 8, 9, 16, 32):
        assert dit_create(native, max_frames) == 0, (max_frames, lib.gtav_last_error())
    for max_frames in (0, 33):
        assert dit_create(native, max_frames) != 0
        msg = lib.gtav_last_error()
        assert b"unsupported geometry" in msg and b"1..32 frames" in msg, msg


def test_temporal_attention_refuses_longer_windows_before_any_launch(native):
    """T = 33 for the dense kernel and 32 cached frames for the last-frame kernel are refused with the supported ranges in
    the message.  The device addresses are never dereferenced: the refusal comes before any launch."""
    lib = native.load()
    fake = 4096
    assert lib.gtav_attention_temporal(fake, fake, 1, 33, 144, 16, fake, None) != 0
    assert b"window of 33 frames unsupported (1..32)" in lib.gtav_last_error()
    assert lib.gtav_attention_temporal(fake, fake, 1, 0, 144, 16, fake, None) != 0
    assert b"(1..32)" in lib.gtav_last_error()
    assert lib.gtav_attention_temporal_last(fake, fake, 1, 32, 144, 16, fake, fake, None) != 0
    assert b"32 cached frames unsupported (0..31)" in lib.gtav_last_error()
    assert lib.gtav_attention_temporal_last(fake, fake, 1, -1, 144, 16, fake, fake, None) != 0
    assert b"(0..31)" in lib.gtav_last_error()
    # a long window without its cache is refused too
    assert lib.gtav_attention_temporal_last(fake, fake, 1, 20, 144, 16, fake, None, None) != 0
    assert b"missing K/V cache" in lib.gtav_last_error()


def test_dit_module_max_frames_limit(native):
    from gtav_b200.model.dit import MAX_FRAMES, DiT
    assert MAX_FRAMES == 32
    assert DiT(depth=1, max_frames=32).max_frames == 32
    with pytest.raises(RuntimeError, match="max_frames=33 .* 1 to 32 frames"):
        DiT(depth=1, max_frames=33)
    with pytest.raises(RuntimeError, match="max_frames=0"):
        DiT(depth=1, max_frames=0)
    # the attribute the reference's generate.py sets after construction is checked when the weights are packed, before
    # anything is allocated on a device
    m = DiT(depth=1)
    m.max_frames = 33
    with pytest.raises(RuntimeError, match="1 to 32 frames"):
        m._pack()


def test_cli_max_frames_flag():
    from gtav_b200.generate import build_parser
    assert build_parser().parse_args([]).max_frames == 5
    assert build_parser().parse_args(["--max_frames", "16"]).max_frames == 16
