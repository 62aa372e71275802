"""
The one-hot observation in compressible device memory (ml2048_alloc_compressible): an environment whose one-hot lives there
must compute exactly what one with plain torch memory (ML2048_ONEHOT_COMPRESSIBLE=0) computes -- every array, bit for bit,
through auto-resets, fused and separate prepare(), a CUDA-graph replay and a state_dict round trip -- and the memory must
live exactly as long as a tensor view of it and then go back to the driver.
"""

from __future__ import annotations

import ctypes
import gc

import pytest
import torch

STATE = ("_board", "_valid", "_id", "_step_score", "_reward", "_terminated_padded", "_invalid", "_reset_count_dev", "_game_count_dev",
         "_stats_dev", "_merged", "_onehot", "_actions_out")


def test_alloc_arguments_and_no_device(monkeypatch):
    """Runs without a GPU: argument errors, a no-op free, and an error code (never a crash) where there is no device."""
    from ml2048_b200 import _lib, build

    build.build()
    lib = _lib.load()
    c = _lib.Compressible()
    assert lib.ml2048_alloc_compressible(0, 1 << 20, None) == -1
    assert lib.ml2048_alloc_compressible(0, 0, ctypes.byref(c)) == -3
    assert lib.ml2048_alloc_compressible(0, -5, ctypes.byref(c)) == -3
    assert lib.ml2048_free_compressible(None) == -1
    assert lib.ml2048_free_compressible(ctypes.byref(c)) == 0  # nothing mapped
    assert lib.ml2048_alloc_compressible(1 << 20, 1 << 20, ctypes.byref(c)) == _lib.E_UNSUPPORTED  # no such device
    assert c.ptr == 0 and c.granted == 0
    rc = lib.ml2048_alloc_compressible(0, 3 << 20, ctypes.byref(c))
    if rc == 0:  # a device with generic compression
        assert c.ptr and c.size >= 3 << 20 and 0 <= c.granted <= c.size and c.chunks >= 1
        assert lib.ml2048_free_compressible(ctypes.byref(c)) == 0
        assert c.ptr == 0
    else:
        assert rc == _lib.E_UNSUPPORTED
        assert c.ptr == 0


@pytest.fixture(scope="module")
def ml():
    import ml2048_b200

    assert torch.cuda.is_available()
    return ml2048_b200


def make(ml, monkeypatch, m: int, onehot: str, compressible: bool):
    monkeypatch.setenv("ML2048_ONEHOT_COMPRESSIBLE", "1" if compressible else "0")
    return ml.VecGame(m, "improved", output="torch", onehot=onehot, sync_free=True)


def assert_same(a, b, what: str) -> None:
    assert a._cur == b._cur, what
    for name in STATE:
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), f"{name} {what}"
        if x is not None:
            assert torch.equal(x, y), f"{name} {what}"
    n = int(a._reset_count_dev.item())
    assert torch.equal(a._reset_indices_dev[:n], b._reset_indices_dev[:n]), f"reset indices {what}"


def expect_compressed(m: int, onehot: str) -> bool:
    """A B200 grants generic compression; only a one-hot larger than the L2 is put in compressible memory."""
    nbytes = m * 256 * {"f32": 4, "bf16": 2, "u8": 1}[onehot]
    return torch.cuda.get_device_capability()[0] >= 10 and nbytes > torch.cuda.get_device_properties(0).L2_cache_size


def advance(env, fused: bool) -> None:
    if fused:
        env.step_random(return_actions=True, auto_reset=True)
    else:
        env.prepare()
        env.step_random(return_actions=True)


@pytest.mark.gpu
def test_compression_granted(ml, monkeypatch):
    env = make(ml, monkeypatch, 1 << 22, "f32", True)
    print(f"\n{torch.cuda.get_device_name()}: one-hot of 2^22 games in compressible memory: {env.onehot_compressed}")
    assert env.onehot_compressed == expect_compressed(1 << 22, "f32")
    assert make(ml, monkeypatch, 1 << 22, "f32", False).onehot_compressed is False
    # a one-hot that fits in the L2 stays in plain memory (2 MiB at the training shape)
    assert make(ml, monkeypatch, 2048, "f32", True).onehot_compressed is False


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True], ids=["prepare_then_step", "fused_autoreset"])
@pytest.mark.parametrize("onehot", ["f32", "bf16", "u8"])
@pytest.mark.parametrize("m", [2048, (1 << 19) + 5, 1 << 22])
def test_compressible_equals_plain(ml, monkeypatch, m, onehot, fused):
    comp = make(ml, monkeypatch, m, onehot, True)
    plain = make(ml, monkeypatch, m, onehot, False)
    assert not plain.onehot_compressed
    assert comp.onehot_compressed == expect_compressed(m, onehot)
    comp.reset(11)
    plain.reset(11)
    assert_same(comp, plain, "after reset")
    steps = 300
    for t in range(steps):
        advance(comp, fused)
        advance(plain, fused)
        if t % 50 == 0 or t == steps - 1:
            assert_same(comp, plain, f"after step {t}")
    assert int(comp._game_count_dev.item()) > m  # the rollout went through auto-resets
    # a snapshot restored into a fresh compressible environment continues exactly as the plain one
    restored = make(ml, monkeypatch, m, onehot, True)
    restored.load_state_dict(comp.state_dict())
    for t in range(20):
        advance(restored, fused)
        advance(plain, fused)
    assert_same(restored, plain, "after the state_dict round trip")


@pytest.mark.gpu
@pytest.mark.parametrize("m", [2048, (1 << 19) + 5, 1 << 22])
def test_graphed_rollout(ml, monkeypatch, m):
    from ml2048_b200.graph import GraphedRollout

    envs = [make(ml, monkeypatch, m, "f32", c) for c in (True, False)]
    for env in envs:
        env.reset(5)
        for _ in range(40):
            advance(env, True)
        GraphedRollout(env, 16, auto_reset=True).replay()
    torch.cuda.synchronize()
    assert_same(envs[0], envs[1], "after one graph replay")


@pytest.mark.gpu
def test_view_outlives_env(ml, monkeypatch):
    env = make(ml, monkeypatch, 1 << 18, "f32", True)  # 256 MiB: larger than the L2
    assert env.onehot_compressed == expect_compressed(1 << 18, "f32")
    env.reset(3)
    for _ in range(30):
        advance(env, True)
    view = env.observations_onehot()[100:200]
    want = view.clone()
    del env
    gc.collect()
    torch.cuda.synchronize()
    assert torch.equal(view, want)
    view.add_(1)  # still writable device memory
    assert torch.equal(view, want + 1)


@pytest.mark.gpu
def test_memory_is_returned(ml, monkeypatch):
    m = 1 << 22  # 4 GiB of fp32 one-hot
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    for i in range(20):
        env = make(ml, monkeypatch, m, "f32", True)
        assert env.onehot_compressed == expect_compressed(m, "f32")
        if i == 0:
            assert torch.cuda.mem_get_info()[0] < free0 - (4 << 30)  # the one-hot really is allocated
        env.step_random(auto_reset=True)
        del env
        gc.collect()
        torch.cuda.empty_cache()
    assert torch.cuda.mem_get_info()[0] > free0 - (256 << 20)


@pytest.mark.gpu
def test_release_during_capture_is_deferred(ml, monkeypatch):
    """The free synchronises the device, which a capture forbids: a one-hot released inside a capture is freed later."""
    from ml2048_b200 import vecgame

    env = make(ml, monkeypatch, 1 << 18, "f32", True)
    if not env.onehot_compressed:
        pytest.skip("no compressible memory on this device")
    onehot = env.observations_onehot()
    del env
    gc.collect()
    x = torch.zeros(16, device="cuda")
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        x.add_(1)
        del onehot  # the last reference: the range is released while the stream captures
    assert len(vecgame._PENDING_FREES) == 1
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(x, torch.ones_like(x))  # the capture stayed valid
    free0 = torch.cuda.mem_get_info()[0]
    make(ml, monkeypatch, 2048, "u8", True)  # the next one-hot allocation frees the deferred range
    assert not vecgame._PENDING_FREES
    assert torch.cuda.mem_get_info()[0] > free0 + (200 << 20)
