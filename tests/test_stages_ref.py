"""
Multi-stage n-tuple networks without a GPU: the stage function of tests/_stage_ref.py against a brute-force loop, the device
header's stage arithmetic (board_ops.cuh compiled for the host by tests/host_shim/stage_host.cpp) against the reference, the
staged references against direct per-board loops, and the Python and C argument checks that need no device.
"""

from __future__ import annotations

import ctypes
import itertools
import os
import re
import subprocess

import numpy as np
import pytest

import _lambda_ref as lref
import _ntuple_ref as nref
import _stage_ref as sref
import _tc_ref as tref

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SHIM_SRC = os.path.join(HERE, "host_shim", "stage_host.cpp")
HEADER = os.path.join(ROOT, "include", "ml2048_b200.h")


def _all_stage_sets():
    """every threshold set of S = 1..4 stages over exponents 1..6, and two of S = 8"""
    sets = [()]
    for r in (1, 2, 3):
        sets += list(itertools.combinations(range(1, 7), r))
    return sets + [(2, 3, 4, 5, 6, 7, 8), (1, 3, 5, 7, 9, 11, 15)]


def _brute_stage(board, stages) -> int:
    m = 0
    for x in board:
        m = max(m, min(int(x), 15))
    return sum(1 for t in stages if t <= m)


def _boards(rng, m: int) -> np.ndarray:
    """every max exponent 0..15 (at a random cell), plus arbitrary bytes (>= 16 among them) in every fourth board"""
    b = np.where(rng.random((m, 16)) < 0.5, 0, rng.integers(1, 16, size=(m, 16))).astype(np.uint8)
    top = rng.integers(0, 16, size=m)
    b = np.minimum(b, top[:, None]).astype(np.uint8)
    b[np.arange(m), rng.integers(0, 16, size=m)] = top
    b[::4] = rng.integers(0, 256, size=b[::4].shape, dtype=np.uint8)
    return b


def _spec_arrays(tuples):
    cells = np.zeros((len(tuples), 6), np.uint8)
    for i, t in enumerate(tuples):
        cells[i, :len(t)] = t
    return cells, np.array([len(t) for t in tuples], np.uint8)


# ---- the stage function --------------------------------------------------------------------------


def test_stage_against_brute_force():
    rng = np.random.default_rng(0)
    boards = _boards(rng, 600)
    every_m = np.zeros((16, 16), np.uint8)
    every_m[np.arange(16), np.arange(16) % 16] = np.arange(16)  # m = 0 (empty) .. 15
    high = np.repeat(np.arange(16, 256, dtype=np.uint8)[:, None], 16, axis=1)  # bytes 16..255 count as 15
    boards = np.concatenate([boards, every_m, high])
    for stages in _all_stage_sets():
        want = np.array([_brute_stage(b, stages) for b in boards])
        np.testing.assert_array_equal(sref.stage(boards, stages), want)
    assert (sref.stage(high, (15,)) == 1).all() and (sref.stage(every_m, (4,)) == (np.arange(16) >= 4)).all()


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("stage_shim") / "libstage_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, SHIM_SRC], check=True)
    lib = ctypes.CDLL(so)
    vp, i64, i32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32
    lib.st_table.argtypes = [vp, i32]
    lib.st_table.restype = ctypes.c_uint64
    lib.st_stage_batch.argtypes = [vp, i64, vp, i32, vp]
    lib.st_value_batch.argtypes = [vp, i64, vp, vp, vp, i32, vp, i32, vp]
    return lib


def _tau(stages):
    return np.array(stages if stages else [0], np.uint8)


def test_host_stage_table_and_stage(shim):
    rng = np.random.default_rng(1)
    boards = np.concatenate([_boards(rng, 3000), rng.integers(0, 256, (500, 16), dtype=np.uint8)])
    out = np.zeros(boards.shape[0], np.uint32)
    for stages in _all_stage_sets():
        tau = _tau(stages)
        table = shim.st_table(tau.ctypes.data, len(stages) + 1)
        assert [(table >> (4 * m)) & 15 for m in range(16)] == [_brute_stage([m], stages) for m in range(16)]
        shim.st_stage_batch(boards.ctypes.data, boards.shape[0], tau.ctypes.data, len(stages) + 1, out.ctypes.data)
        np.testing.assert_array_equal(out.astype(np.int64), sref.stage(boards, stages))


def test_host_staged_value_bit_exact(shim):
    rng = np.random.default_rng(2)
    for tuples, stages in ((nref.STANDARD_4X6, (4, 6)), (((0, 1, 2), (5, 9)), (2, 3, 4, 5, 6, 7, 8)), (((3, 7),), ()),
                           (((0, 5, 10, 15),), (15,))):
        cells, lens = _spec_arrays(tuples)
        w = (rng.standard_normal(sref.num_weights(tuples, stages)) * 100).astype(np.float32)
        boards = np.concatenate([_boards(rng, 2000), rng.integers(0, 256, (300, 16), dtype=np.uint8)])
        out = np.zeros(boards.shape[0], np.float32)
        tau = _tau(stages)
        shim.st_value_batch(boards.ctypes.data, boards.shape[0], w.ctypes.data, cells.ctypes.data, lens.ctypes.data, len(tuples),
                            tau.ctypes.data, len(stages) + 1, out.ctypes.data)
        np.testing.assert_array_equal(out.view(np.uint32), sref.value(boards, w, tuples, stages).view(np.uint32))


# ---- the staged references against per-board loops ----------------------------------------------------


def _loop_value(board, w, tuples, stages):
    base = _brute_stage(board, stages) * nref.num_weights(tuples)
    acc = np.float32(0)
    for e in nref.entries(board[None], tuples)[0]:
        acc = np.float32(acc + w[base + e])
    return acc


def test_staged_references_against_loops():
    rng = np.random.default_rng(3)
    tuples, stages = ((0, 1, 2), (5, 9)), (3, 5)
    n = sref.num_weights(tuples, stages)
    w = np.round(rng.standard_normal(n) * 8).astype(np.float32)
    m = 160
    boards = _boards(rng, m)
    v = sref.value(boards, w, tuples, stages)
    np.testing.assert_array_equal(v.view(np.uint32), np.array([_loop_value(b, w, tuples, stages) for b in boards]).view(np.uint32))
    # greedy: every afterstate on its own stage
    after = _boards(rng, 4 * m).reshape(m, 4, 16)
    reward = rng.integers(0, 3, size=(m, 4)).astype(np.float32)
    valid = rng.integers(0, 2, size=(m, 4)).astype(np.uint8)
    valid[:10] = 0
    g = sref.greedy(boards, after, reward, valid, w, tuples, stages)
    for i in range(m):
        qs = [(np.float32(reward[i, a] + _loop_value(after[i, a], w, tuples, stages)), a) for a in range(4) if valid[i, a]]
        if not qs:
            assert g["action"][i] == 0 and (g["state"][i] == boards[i]).all() and g["value"][i] == 0
            continue
        best = max(qs, key=lambda qa: (qa[0], -qa[1]))[1]
        assert g["action"][i] == best and g["value"][i] == _loop_value(after[i, best], w, tuples, stages)
    # TD(0): delta on x_0's stage, the adds into x_0's stage
    target = rng.standard_normal(m).astype(np.float32)
    mask = rng.integers(0, 2, m).astype(np.uint8)
    d = sref.td_delta(boards, target, w, tuples, stages, 0.25, mask)
    loop = w.astype(np.float64).copy()
    for i in range(m):
        want = np.float32(np.float32(0.25) * np.float32(target[i] - _loop_value(boards[i], w, tuples, stages))) if mask[i] else 0
        assert d[i] == want
        if mask[i]:
            for e in sref.entries(boards[i:i + 1], tuples, stages)[0]:
                loop[e] += d[i]
    w64, cnt, _ = sref.td_apply_f64(boards, d, w, tuples, stages, mask)
    np.testing.assert_allclose(w64, loop, rtol=0, atol=1e-9)
    np.testing.assert_allclose(sref.td_apply_f32(boards, d, w, tuples, stages, mask), loop, rtol=1e-5, atol=1e-4)
    assert cnt.sum() == 8 * len(tuples) * int(mask.sum())
    # TC: the accumulator holds x_0's stage's entries; the apply is entry by entry
    de, da = sref.tc_accumulate(boards, d, tuples, stages, mask)
    de64 = np.zeros(n)
    for i in range(m):
        if mask[i]:
            for e in sref.entries(boards[i:i + 1], tuples, stages)[0]:
                de64[e] += d[i]
    np.testing.assert_allclose(de, de64, rtol=1e-5, atol=1e-4)
    coh = np.zeros((n, 2), np.float32)
    w2, c2 = sref.tc_update_f32(boards, d, w, coh, tuples, stages, mask)
    w3, c3 = tref.tc_apply_f32(de, da, w, coh)
    np.testing.assert_array_equal(w2.view(np.uint32), w3.view(np.uint32))
    # TC in float64: sums per entry of x_0's stage, beta from the coherence before the call
    coh = np.abs(rng.standard_normal((n, 2))).astype(np.float32)
    w64, e64, a64, cnt, sabs = sref.tc_apply_f64(boards, d, w, coh, tuples, stages, mask)
    beta = tref.tc_beta_f32(coh).astype(np.float64)
    hit = sabs != 0
    np.testing.assert_allclose(w64, np.where(hit, w + beta * de64, w), rtol=0, atol=1e-9)
    np.testing.assert_allclose(e64, np.where(hit, coh[:, 0] + de64, coh[:, 0]), rtol=0, atol=1e-9)
    np.testing.assert_array_equal(cnt, sref.td_apply_f64(boards, d, w, tuples, stages, mask)[1])
    # TD(lambda): every window board valued on its own stage
    h = 3
    ring = _boards(rng, (h + 1) * m).reshape(h + 1, m, 16)
    rew = rng.integers(0, 5, size=(h + 1, m)).astype(np.float32)
    ended = (rng.random((h + 1, m)) < 0.2).astype(np.uint8)
    got, x0 = sref.ring_delta(ring, rew, ended, 1, w, tuples, stages, 0.3, 0.1, mask)
    win = lref.window(ring, 1)
    vals = np.array([[_loop_value(win[k, i], w, tuples, stages) for i in range(m)] for k in range(h + 1)], np.float32)
    want = lref.lambda_delta(vals, lref.window(rew, 1), lref.window(ended, 1), 0.3, 0.1, mask)
    np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))
    assert (x0 == win[0]).all()


def test_one_stage_is_the_single_stage_reference():
    rng = np.random.default_rng(4)
    tuples = nref.STANDARD_4X6
    w = (rng.standard_normal(nref.num_weights(tuples)) * 50).astype(np.float32)
    boards = _boards(rng, 500)
    np.testing.assert_array_equal(sref.value(boards, w, tuples, ()).view(np.uint32), nref.value(boards, w, tuples).view(np.uint32))
    np.testing.assert_array_equal(sref.entries(boards, tuples, ()), nref.entries(boards, tuples))


# ---- Python argument checks ---------------------------------------------------------------------------------


def test_stage_validation():
    from ml2048_b200 import ops

    assert ops.ntuple_stages(()) == () and ops.ntuple_stages([4, 6]) == (4, 6) and ops.ntuple_stages(np.array([1, 15])) == (1, 15)
    assert ops.ntuple_stages(range(2, 9)) == (2, 3, 4, 5, 6, 7, 8)
    assert ops.ntuple_num_weights(nref.STANDARD_4X6) == 4 * 16 ** 6
    assert ops.ntuple_num_weights(nref.STANDARD_4X6, (10,)) == 2 * 4 * 16 ** 6
    assert ops.ntuple_num_weights([[0]], range(1, 8)) == 8 * 16
    for bad in ([5, 4], [4, 4], [0], [16], [-1], list(range(1, 9)), [4.0], [True], [4, False], ["4"], 4, None):
        with pytest.raises(ValueError):
            ops.ntuple_stages(bad)
        with pytest.raises(ValueError):
            ops.ntuple_num_weights([[0]], bad)
    # the same thresholds are checked on every call, whatever was cached by an earlier one: (True,) == (1,), (4.0,) == (4,)
    assert ops._stage_array((1,))[1] == 2 and ops._stage_array((4,))[1] == 2
    for bad in ((True,), (4.0,)):
        with pytest.raises(ValueError):
            ops._stage_array(bad)


def test_network_stage_checks_without_gpu():
    from ml2048_b200.ntuple import NTupleNetwork

    with pytest.raises(ValueError):
        NTupleNetwork([[0]], device="cpu", stages=(4,))  # CUDA only
    with pytest.raises(ValueError):
        NTupleNetwork([[0]], device="cuda", stages=(3, 2))


def test_c_argument_errors_without_gpu():
    """the stage checks of all seven entries, each returning its code before any launch (the pointers are never
    dereferenced)"""
    from ml2048_b200 import _lib, build

    build.build()
    lib = _lib.load()
    cells, lens = _spec_arrays(((0, 1), (5,)))
    n = 16 ** 2 + 16
    c, ln = cells.ctypes.data, lens.ctypes.data
    P = [0x10000 * (i + 1) for i in range(12)]  # distinct 16-byte aligned fake pointers

    calls = {
        "value": lambda nw, tau, s: lib.ml2048_staged_value(P[0], P[1], nw, c, ln, 2, tau, s, P[2], 8, None),
        "greedy": lambda nw, tau, s: lib.ml2048_staged_greedy(P[0], P[1], nw, c, ln, 2, tau, s, 0, P[2], None, P[3], P[4], P[5], 8, None),
        "td": lambda nw, tau, s: lib.ml2048_staged_td_update(P[0], P[1], None, 0.1, P[2], nw, c, ln, 2, tau, s, P[3], 8, None),
        "tc": lambda nw, tau, s: lib.ml2048_staged_tc_update(P[0], P[1], None, 0.1, P[2], P[3], P[4], nw, c, ln, 2, tau, s, P[5], 8, None),
        "lambda_td": lambda nw, tau, s: lib.ml2048_staged_lambda_td_update(P[0], P[1], P[2], 2, 0, 0.5, None, 0.1, P[3], nw, c, ln, 2, tau, s,
                                                                           P[4], 8, None),
        "lambda_tc": lambda nw, tau, s: lib.ml2048_staged_lambda_tc_update(P[0], P[1], P[2], 2, 0, 0.5, None, 0.1, P[3], P[4], P[5], nw, c,
                                                                           ln, 2, tau, s, P[6], 8, None),
        "expectimax": lambda nw, tau, s: lib.ml2048_staged_expectimax(P[0], P[1], nw, c, ln, 2, tau, s, 0, 1, 0.9, P[2], None, P[3], P[4],
                                                                      P[5], P[6], 8, None),
    }
    ok2 = np.array([4], np.uint8)
    for name, call in calls.items():
        assert call(2 * n, None, 2) == -1, name  # E_NULL: no thresholds with S > 1
        assert call(n, None, 0) == -3 and call(9 * n, None, 9) == -3 and call(n, None, -1) == -3, name  # E_SIZE: S outside 1..8
        assert call(n, ok2.ctypes.data, 2) == -3 and call(3 * n, ok2.ctypes.data, 2) == -3, name  # E_SIZE: num_weights != S * N
        assert call(2 * n, None, 1) == -3, name  # S = 1 with S * N weights
        for bad in ([0], [16], [255], [5, 5], [6, 5], [1, 2, 3, 4, 5, 6, 6]):
            tau = np.array(bad, np.uint8)
            assert call((len(bad) + 1) * n, tau.ctypes.data, len(bad) + 1) == -4, (name, bad)  # E_ENUM


def test_header_declarations_compile(tmp_path):
    """the staged entries compile from C with their documented argument types, and _lib.SYMBOLS lists them"""
    from ml2048_b200 import _lib

    src = tmp_path / "st.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *w, uint8_t *c, uint8_t *l, const uint8_t *t, float *v, uint8_t *a8, int64_t *a64, void *s) {\n"
        "  return ml2048_staged_value(b, w, 32, c, l, 1, t, 2, v, 1, s)\n"
        "       + ml2048_staged_greedy(b, w, 32, c, l, 1, t, 2, 0, a8, a64, b, v, v, 1, s)\n"
        "       + ml2048_staged_td_update(b, v, a8, 0.5f, w, 32, c, l, 1, t, 2, v, 1, s)\n"
        "       + ml2048_staged_tc_update(b, v, a8, 0.5f, w, v, v, 32, c, l, 1, t, 2, v, 1, s)\n"
        "       + ml2048_staged_lambda_td_update(b, v, a8, 2, 0, 0.5f, a8, 0.5f, w, 32, c, l, 1, t, 2, v, 1, s)\n"
        "       + ml2048_staged_lambda_tc_update(b, v, a8, 2, 0, 0.5f, a8, 0.5f, w, v, v, 32, c, l, 1, t, 2, v, 1, s)\n"
        "       + ml2048_staged_expectimax(b, w, 32, c, l, 1, t, 2, 0, 1, 0.9, a8, a64, b, v, v, v, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "st.o")], check=True)
    declared = set(re.findall(r"ML2048_API\s+[\w\s\*]+?\b(ml2048_staged_\w+)\s*\(", open(HEADER).read()))
    assert declared == {"ml2048_staged_value", "ml2048_staged_greedy", "ml2048_staged_td_update", "ml2048_staged_tc_update",
                        "ml2048_staged_lambda_td_update", "ml2048_staged_lambda_tc_update", "ml2048_staged_expectimax"}
    assert declared <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 12
