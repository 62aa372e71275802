"""
Weight promotion of multi-stage n-tuple networks without a GPU: the reference of tests/_promotion_ref.py against per-entry
brute-force loops, the device header's source stage and promoted value (board_ops.cuh compiled for the host by
tests/host_shim/promotion_host.cpp) against it, and the Python and C argument checks that need no device.
"""

from __future__ import annotations

import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import _ntuple_ref as nref
import _promotion_ref as pref
import _stage_ref as sref

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SHIM_SRC = os.path.join(HERE, "host_shim", "promotion_host.cpp")
HEADER = os.path.join(ROOT, "include", "ml2048_b200.h")
TUPLES = ((0, 1, 2), (5, 9))


def _boards(rng, m: int) -> np.ndarray:
    """boards of every largest tile 0..15, a few with bytes >= 16"""
    top = rng.integers(0, 16, size=m)
    b = np.minimum(np.where(rng.random((m, 16)) < 0.5, 0, rng.integers(1, 16, size=(m, 16))), top[:, None]).astype(np.uint8)
    b[np.arange(m), rng.integers(0, 16, size=m)] = top
    b[::7] = rng.integers(0, 256, size=b[::7].shape, dtype=np.uint8)
    return b


def _brute_stage(board, stages) -> int:
    return sum(1 for t in stages if t <= max(min(int(x), 15) for x in board))


def _brute_w(w, marks, n, s, e):
    """W(s, e) by its recursive definition"""
    if s == 0 or (marks[e] >> (s - 1)) & 1:
        return w[s * n + e]
    return _brute_w(w, marks, n, s - 1, e)


def _brute_value(board, w, marks, tuples, stages):
    n = nref.num_weights(tuples)
    s = _brute_stage(board, stages)
    acc = np.float32(0)
    for e in nref.entries(board[None], tuples)[0]:
        acc = np.float32(acc + _brute_w(w, marks, n, s, int(e)))
    return acc


def _net(rng, stages, tuples=TUPLES):
    n = nref.num_weights(tuples)
    w = np.round(rng.standard_normal(sref.num_stages(stages) * n) * 8).astype(np.float32)
    marks = rng.integers(0, 256, n, dtype=np.uint8)
    return n, w, marks


# ---- the reference against brute force ------------------------------------------------------------------


def test_source_stage_and_effective_weights():
    for s in range(8):
        for m in range(256):
            want = max([0] + [k for k in range(1, s + 1) if (m >> (k - 1)) & 1])
            assert pref.source_stage(s, m) == want
            assert (((m << 1) | 1) & ((2 << s) - 1)).bit_length() - 1 == want  # the header's 31 - clz(...)
    rng = np.random.default_rng(0)
    for stages in ((4,), (3, 5), tuple(range(2, 9))):
        n, w, marks = _net(rng, stages)
        eff = pref.effective(w, marks, TUPLES, stages)
        for s in range(len(stages) + 1):
            for e in range(n):
                assert eff[s * n + e] == _brute_w(w, marks, n, s, e) == w[pref.source_stage(s, int(marks[e])) * n + e]


def test_reads_against_loops():
    rng = np.random.default_rng(1)
    stages = (3, 5)
    n, w, marks = _net(rng, stages)
    boards = _boards(rng, 200)
    want = np.array([_brute_value(b, w, marks, TUPLES, stages) for b in boards])
    np.testing.assert_array_equal(pref.value(boards, w, marks, TUPLES, stages).view(np.uint32), want.view(np.uint32))
    # unmarked storage never enters a value
    poisoned = w.copy().reshape(3, n)
    for s in (1, 2):
        poisoned[s][(marks >> (s - 1)) & 1 == 0] = np.nan
    np.testing.assert_array_equal(pref.value(boards, poisoned.reshape(-1), marks, TUPLES, stages).view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("rule", ["td", "tc"])
def test_update_with_promotion_against_loops(rule):
    """delta on W before the call; every masked-in x_0 in stage s0 >= 1 copies W(s0 - 1, e) into its unmarked entries (TC:
    coherence (0, 0)) and marks them; then the staged apply.  Integer data: every sum is exact."""
    rng = np.random.default_rng(2)
    stages = (3, 5)
    n, w, marks = _net(rng, stages)
    m = 120
    boards = _boards(rng, m)
    boards[100:110] = boards[90:100]  # the same boards twice in one call
    target = np.round(rng.standard_normal(m) * 16).astype(np.float32)
    mask = rng.integers(0, 2, m).astype(np.uint8)
    mask[90:110] = 1
    alpha = 0.0625
    coh = np.abs(np.round(rng.standard_normal((3 * n, 2)) * 4)).astype(np.float32)
    # brute force
    bw, bm, bc = w.astype(np.float64).copy(), marks.copy(), coh.copy()
    d = np.zeros(m, np.float32)
    for i in range(m):
        if mask[i]:
            d[i] = np.float32(np.float32(alpha) * np.float32(target[i] - _brute_value(boards[i], w, marks, TUPLES, stages)))
    for i in range(m):
        s0 = _brute_stage(boards[i], stages)
        if mask[i] and s0 >= 1:
            for e in nref.entries(boards[i:i + 1], TUPLES)[0]:
                if not (marks[e] >> (s0 - 1)) & 1:
                    bw[s0 * n + e] = _brute_w(w, marks, n, s0 - 1, int(e))
                    bc[s0 * n + e] = 0.0
                    bm[e] |= 1 << (s0 - 1)
    if rule == "td":
        got_d, got_w, got_m = pref.td_update(boards, target, w, marks, TUPLES, stages, alpha, mask)
        for i in range(m):
            if mask[i]:
                for e in sref.entries(boards[i:i + 1], TUPLES, stages)[0]:
                    bw[e] += d[i]
        np.testing.assert_array_equal(got_w, bw.astype(np.float32))
    else:
        got_d, got_w, got_c, got_m = pref.tc_update(boards, target, w, coh, marks, TUPLES, stages, alpha, mask)
        de, da = np.zeros(3 * n), np.zeros(3 * n)
        for i in range(m):
            if mask[i]:
                for e in sref.entries(boards[i:i + 1], TUPLES, stages)[0]:
                    de[e] += d[i]
                    da[e] += abs(d[i])
        for j in np.nonzero(da)[0]:
            beta = 1.0 if bc[j, 1] == 0 else np.float32(abs(bc[j, 0]) / bc[j, 1])
            bw[j] = np.float32(bw[j] + np.float32(beta * np.float32(de[j])))
            bc[j] = (bc[j, 0] + de[j], bc[j, 1] + da[j])
        np.testing.assert_array_equal(got_w, bw.astype(np.float32))
        np.testing.assert_array_equal(got_c, bc)
    np.testing.assert_array_equal(got_d, d)
    np.testing.assert_array_equal(got_m, bm)
    # promotion alone changes no effective weight; stage 0 is never written by it
    pw, pm, _ = pref.promote(boards, w, marks, TUPLES, stages, mask)
    np.testing.assert_array_equal(pref.effective(pw, pm, TUPLES, stages), pref.effective(w, marks, TUPLES, stages))
    np.testing.assert_array_equal(pw[:n], w[:n])


def test_all_marks_set_and_one_stage_are_the_staged_reference():
    rng = np.random.default_rng(3)
    stages = (3, 5)
    n, w, _ = _net(rng, stages)
    full = np.full(n, 3, np.uint8)
    boards = _boards(rng, 300)
    np.testing.assert_array_equal(pref.value(boards, w, full, TUPLES, stages), sref.value(boards, w, TUPLES, stages))
    target = np.round(rng.standard_normal(300) * 16).astype(np.float32)
    d, w2, m2 = pref.td_update(boards, target, w, full, TUPLES, stages, 0.0625)
    np.testing.assert_array_equal(m2, full)
    np.testing.assert_array_equal(w2, sref.td_apply_f32(boards, d, w, TUPLES, stages))
    w1 = w[:n]
    any_marks = rng.integers(0, 256, n, dtype=np.uint8)
    np.testing.assert_array_equal(pref.value(boards, w1, any_marks, TUPLES, ()), nref.value(boards, w1, TUPLES))
    assert (pref.promote(boards, w1, any_marks, TUPLES, ())[1] == any_marks).all()


# ---- the header compiled for the host ---------------------------------------------------------------------


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("promotion_shim") / "libpromotion_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, SHIM_SRC], check=True)
    lib = ctypes.CDLL(so)
    vp, i64, i32, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_uint32
    lib.pr_source_stage.argtypes = [u32, u32]
    lib.pr_source_stage.restype = u32
    lib.pr_value_batch.argtypes = [vp, i64, vp, vp, vp, i32, vp, i32, vp, vp]
    return lib


def test_host_source_stage(shim):
    for s in range(8):
        for m in range(256):
            assert shim.pr_source_stage(s, m) == pref.source_stage(s, m), (s, m)


def test_host_promoted_value_bit_exact(shim):
    rng = np.random.default_rng(4)
    for tuples, stages in ((nref.STANDARD_4X6, (4, 6)), (TUPLES, tuple(range(2, 9))), (((0, 5, 10, 15),), (15,))):
        n = nref.num_weights(tuples)
        w = (rng.standard_normal(sref.num_weights(tuples, stages)) * 100).astype(np.float32)
        marks = rng.integers(0, 256, n, dtype=np.uint8)
        cells = np.zeros((len(tuples), 6), np.uint8)
        for i, t in enumerate(tuples):
            cells[i, :len(t)] = t
        lens = np.array([len(t) for t in tuples], np.uint8)
        boards = _boards(rng, 2000)
        want = pref.value(boards, w, marks, tuples, stages)
        eff = pref.effective(w, marks, tuples, stages).reshape(len(stages) + 1, n)
        poisoned = w.copy().reshape(len(stages) + 1, n)
        for s in range(1, len(stages) + 1):
            poisoned[s][(marks >> (s - 1)) & 1 == 0] = np.nan
        assert not np.isnan(eff).any()
        tau = np.array(stages, np.uint8)
        for ww in (w, poisoned.reshape(-1)):
            out = np.zeros(boards.shape[0], np.float32)
            shim.pr_value_batch(boards.ctypes.data, boards.shape[0], ww.ctypes.data, cells.ctypes.data, lens.ctypes.data, len(tuples),
                                tau.ctypes.data, len(stages) + 1, marks.ctypes.data, out.ctypes.data)
            np.testing.assert_array_equal(out.view(np.uint32), want.view(np.uint32))


# ---- argument checks ---------------------------------------------------------------------------------------


def test_python_argument_errors_without_gpu():
    import torch

    from ml2048_b200 import ops
    from ml2048_b200.ntuple import NTupleNetwork

    with pytest.raises(ValueError):
        NTupleNetwork([[0]], device="cuda", promotion=True)  # promotion needs stages
    with pytest.raises(ValueError):
        NTupleNetwork([[0]], device="cpu", stages=(4,), promotion=True)  # CUDA only
    w = torch.zeros(2 * 16)
    with pytest.raises(ValueError):
        ops.ntuple_promoted_weights(w, torch.zeros(16, dtype=torch.uint8), [[0]], (4,))  # CPU tensors
    with pytest.raises(ValueError):
        ops._promoted_arg(torch.zeros(16, dtype=torch.uint8), 16, torch.device("cpu"))
    assert ops._promoted_arg(None, 16, None) == () and ops._entry("value", ()) == "ml2048_staged_value"
    assert ops._entry("td_update", (1,)) == "ml2048_promoted_td_update"


def _calls(lib, cells, lens, n):
    c, ln = cells.ctypes.data, lens.ctypes.data
    P = [0x10000 * (i + 1) for i in range(12)]  # distinct 16-byte aligned fake pointers, never dereferenced
    tau = np.array([4], np.uint8)
    t = tau.ctypes.data
    return tau, {
        "value": lambda nw, s, pm: lib.ml2048_promoted_value(P[0], P[1], nw, c, ln, 2, t, s, pm, P[2], 8, None),
        "greedy": lambda nw, s, pm: lib.ml2048_promoted_greedy(P[0], P[1], nw, c, ln, 2, t, s, pm, 0, P[2], None, P[3], P[4], P[5], 8, None),
        "td": lambda nw, s, pm: lib.ml2048_promoted_td_update(P[0], P[1], None, 0.1, P[2], nw, c, ln, 2, t, s, pm, P[3], 8, None),
        "tc": lambda nw, s, pm: lib.ml2048_promoted_tc_update(P[0], P[1], None, 0.1, P[2], P[3], P[4], nw, c, ln, 2, t, s, pm, P[5], 8,
                                                             None),
        "lambda_td": lambda nw, s, pm: lib.ml2048_promoted_lambda_td_update(P[0], P[1], P[2], 2, 0, 0.5, None, 0.1, P[3], nw, c, ln, 2, t,
                                                                            s, pm, P[4], 8, None),
        "lambda_tc": lambda nw, s, pm: lib.ml2048_promoted_lambda_tc_update(P[0], P[1], P[2], 2, 0, 0.5, None, 0.1, P[3], P[4], P[5], nw,
                                                                            c, ln, 2, t, s, pm, P[6], 8, None),
        "expectimax": lambda nw, s, pm: lib.ml2048_promoted_expectimax(P[0], P[1], nw, c, ln, 2, t, s, pm, 0, 1, 0.9, P[2], None, P[3],
                                                                       P[4], P[5], P[6], 8, None),
    }


def test_c_argument_errors_without_gpu():
    """each of the seven entries returns E_NULL / E_ALIGN for its marks, and the staged entry's codes otherwise, before any
    launch"""
    from ml2048_b200 import _lib, build

    build.build()
    lib = _lib.load()
    cells = np.zeros((2, 6), np.uint8)
    cells[0, :2] = (0, 1)
    cells[1, 0] = 5
    lens = np.array([2, 1], np.uint8)
    n = 16 ** 2 + 16
    pm = 0x200000
    _keep, calls = _calls(lib, cells, lens, n)
    for name, call in calls.items():
        assert call(2 * n, 2, None) == -1, name  # E_NULL
        for off in (1, 2, 3):
            assert call(2 * n, 2, pm + off) == -2, (name, off)  # E_ALIGN
        assert call(3 * n, 2, pm) == -3 and call(2 * n, 9, pm) == -3, name  # the staged entry's E_SIZE
        assert call(n, 1, None) == -1, name  # marks are required whatever S is


def test_header_declarations_compile(tmp_path):
    """the promoted entries compile from C with their documented argument types, and _lib.SYMBOLS lists them"""
    from ml2048_b200 import _lib

    src = tmp_path / "pr.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *w, uint8_t *c, uint8_t *l, const uint8_t *t, uint8_t *p, float *v, uint8_t *a8, int64_t *a64, void *s) {\n"
        "  const uint8_t *cp = p;\n"
        "  return ml2048_promoted_value(b, w, 32, c, l, 1, t, 2, cp, v, 1, s)\n"
        "       + ml2048_promoted_greedy(b, w, 32, c, l, 1, t, 2, cp, 0, a8, a64, b, v, v, 1, s)\n"
        "       + ml2048_promoted_td_update(b, v, a8, 0.5f, w, 32, c, l, 1, t, 2, p, v, 1, s)\n"
        "       + ml2048_promoted_tc_update(b, v, a8, 0.5f, w, v, v, 32, c, l, 1, t, 2, p, v, 1, s)\n"
        "       + ml2048_promoted_lambda_td_update(b, v, a8, 2, 0, 0.5f, a8, 0.5f, w, 32, c, l, 1, t, 2, p, v, 1, s)\n"
        "       + ml2048_promoted_lambda_tc_update(b, v, a8, 2, 0, 0.5f, a8, 0.5f, w, v, v, 32, c, l, 1, t, 2, p, v, 1, s)\n"
        "       + ml2048_promoted_expectimax(b, w, 32, c, l, 1, t, 2, cp, 0, 1, 0.9, a8, a64, b, v, v, v, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "pr.o")], check=True)
    declared = set(re.findall(r"ML2048_API\s+[\w\s\*]+?\b(ml2048_promoted_\w+)\s*\(", open(HEADER).read()))
    assert declared == {"ml2048_promoted_value", "ml2048_promoted_greedy", "ml2048_promoted_td_update", "ml2048_promoted_tc_update",
                        "ml2048_promoted_lambda_td_update", "ml2048_promoted_lambda_tc_update", "ml2048_promoted_expectimax"}
    assert declared <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 12
