"""Ragged windows and StreamPool, host side: the ragged temporal attention entry points and
gtav_dit_plan_set_window_lengths refuse bad arguments with a message before any launch, and the StreamPool surface has the
documented signatures.  Nothing here touches a device."""
import inspect

import pytest


@pytest.fixture(scope="module")
def native():
    import __graft_entry__ as ge
    ge.build()
    import gtav_b200._native as N
    return N


def test_ragged_temporal_attention_refusals(native):
    """A null length array, T outside 1..32 and ctx_frames outside 0..31 are refused before any launch: the fake device
    addresses are never dereferenced."""
    lib = native.load()
    fake = 4096
    assert lib.gtav_attention_temporal_ragged(fake, fake, 2, 5, 144, 16, fake, None, None, None) != 0
    assert b"missing window lengths" in lib.gtav_last_error()
    assert lib.gtav_attention_temporal_last_ragged(fake, fake, 2, 4, 144, 16, fake, None, fake, None) != 0
    assert b"missing window lengths" in lib.gtav_last_error()
    for T in (0, 33, -1):
        assert lib.gtav_attention_temporal_ragged(fake, fake, 2, T, 144, 16, fake, fake, None, None) != 0
        assert f"window of {T} frames unsupported (1..32)".encode() in lib.gtav_last_error()
    for ctx in (32, -1):
        assert lib.gtav_attention_temporal_last_ragged(fake, fake, 2, ctx, 144, 16, fake, fake, fake, None) != 0
        assert f"{ctx} cached frames unsupported (0..31)".encode() in lib.gtav_last_error()
    # a cache is needed as soon as there are cached frames, short or long
    for ctx in (3, 20):
        assert lib.gtav_attention_temporal_last_ragged(fake, fake, 2, ctx, 144, 16, fake, fake, None, None) != 0
        assert b"missing K/V cache" in lib.gtav_last_error()


def test_set_window_lengths_refuses_a_null_plan(native):
    lib = native.load()
    assert lib.gtav_dit_plan_set_window_lengths(None, 4096) != 0
    assert b"null plan" in lib.gtav_last_error()


def test_stream_pool_contract_cpu():
    from gtav_b200.sampler import Sampler, StreamPool
    assert list(inspect.signature(Sampler.pool).parameters) == ["self", "capacity", "use_actions"]
    assert inspect.signature(Sampler.pool).parameters["use_actions"].default is False
    assert list(inspect.signature(StreamPool.open).parameters) == ["self", "prompt_video", "prompt_actions", "generator"]
    assert list(inspect.signature(StreamPool.close).parameters) == ["self", "sid"]
    assert list(inspect.signature(StreamPool.step).parameters) == ["self", "actions", "noise", "decode"]
    step = inspect.signature(StreamPool.step).parameters
    assert (step["actions"].default, step["noise"].default, step["decode"].default) == (None, None, True)
