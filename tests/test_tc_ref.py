"""
Temporal coherence learning without a GPU: the NumPy definition (tests/_tc_ref.py) against a scalar loop written from the
definition, and the checks of the Python and C arguments and of the header that need no device.
"""

from __future__ import annotations

import os
import re
import subprocess

import numpy as np
import pytest

import _ntuple_ref as nref
import _tc_ref as ref

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "ml2048_b200.h")


@pytest.fixture(scope="module")
def lib():
    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    return _lib.load()


def _loop(after, delta, w0, c0, tuples, mask):
    """the definition, one scalar float32 operation at a time, entries collected in a dict"""
    with np.errstate(all="ignore"):
        return _loop_body(after, delta, w0, c0, tuples, mask)


def _loop_body(after, delta, w0, c0, tuples, mask):
    f = np.float32
    acc: dict = {}
    for i in range(after.shape[0]):
        if mask is not None and not mask[i]:
            continue
        off = 0
        for cells in tuples:
            for g in range(8):
                j = off + sum(min(int(after[i][nref.SRC[g][c]]), 15) << (4 * k) for k, c in enumerate(cells))
                de, da = acc.get(j, (f(0), f(0)))
                acc[j] = (f(de + f(delta[i])), f(da + f(abs(f(delta[i])))))
            off += 16 ** len(cells)
    w, c = w0.copy(), c0.copy()
    for j, (de, da) in acc.items():
        if da == 0:
            continue
        e, a = f(c0[j, 0]), f(c0[j, 1])
        beta = f(1) if a == 0 else f(f(abs(e)) / a)
        w[j] = f(w0[j] + f(beta * de))
        c[j, 0] = f(e + de)
        c[j, 1] = f(a + da)
    return w, c


def _same(got, want):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def test_reference_against_scalar_loop():
    """NaN, +-inf, +-0 and ordinary deltas, entries with A = 0, -0 weights and E, an afterstate that hits one entry twice,
    games that share entries, a mask"""
    rng = np.random.default_rng(0)
    tuples = ((0, 1), (5,), (0, 3))  # (0, 1) on a board symmetric under the column flip reads one entry in two images
    n = nref.num_weights(tuples)
    m = 120
    after = rng.integers(0, 4, size=(m, 16)).astype(np.uint8)
    after[0] = [1, 2, 2, 1, 0, 3, 3, 0, 0, 3, 3, 0, 1, 2, 2, 1]  # symmetric: every entry of game 0 is hit more than once
    delta = (rng.standard_normal(m) * 4).astype(np.float32)
    delta[3], delta[4], delta[5], delta[6], delta[7] = np.nan, np.inf, -np.inf, 0.0, -0.0
    delta[8:12] = -0.0
    mask = (rng.random(m) < 0.8).astype(np.uint8)
    mask[:12] = 1
    w0 = (rng.standard_normal(n) * 10).astype(np.float32)
    w0[::7] = -0.0
    c0 = np.abs(rng.standard_normal((n, 2))).astype(np.float32)
    c0[:, 0] *= np.where(rng.random(n) < 0.5, -1, 1).astype(np.float32)
    c0[:, 1] += np.abs(c0[:, 0])  # A >= |E|
    c0[::3] = 0.0  # A = 0: beta = 1
    c0[1::11, 0] = -0.0
    e = nref.entries(after, tuples)
    assert len(set(e[0])) < e.shape[1]
    for msk in (None, mask):
        de, da = ref.tc_accumulate(after, delta, tuples, msk)
        w, c = ref.tc_apply_f32(de, da, w0, c0)
        lw, lc = _loop(after, delta, w0, c0, tuples, msk)
        _same(w, lw)
        _same(c, lc)
    # an entry that only the +-0 deltas reach keeps its -0 weight; one that the NaN delta reaches becomes NaN
    only_zero = set(e[6]) | set(e[7]) | set(int(x) for x in e[8:12].ravel())
    others = set(int(x) for i in range(m) if i not in range(6, 12) for x in e[i])
    for j in only_zero - others:
        assert w[j].tobytes() == w0[j].tobytes() and c[j].tobytes() == c0[j].tobytes()
    for j in set(e[3]):
        assert np.isnan(w[j]) and np.isnan(c[j]).all()


def test_reference_float64_matches_float32_on_disjoint_games():
    """where no entry is shared, the float64 sums differ from float32 only by the final roundings"""
    rng = np.random.default_rng(1)
    tuples = ((0, 1, 2), (4, 9))
    n = nref.num_weights(tuples)
    after = rng.integers(0, 16, size=(30, 16)).astype(np.uint8)
    delta = (rng.standard_normal(30) * 3).astype(np.float32)
    w0 = rng.standard_normal(n).astype(np.float32)
    c0 = np.abs(rng.standard_normal((n, 2))).astype(np.float32)
    c0[:, 1] += np.abs(c0[:, 0])
    w32, c32 = ref.tc_apply_f32(*ref.tc_accumulate(after, delta, tuples), w0, c0)
    w64, e64, a64, adds, sabs = ref.tc_apply_f64(after, delta, w0, c0, tuples)
    assert adds.sum() == 30 * 8 * len(tuples)
    touched = adds > 0
    beta = ref.tc_beta_f32(c0)
    bound = (adds + 2) * 2.0 ** -24 * (np.abs(w0) + beta * sabs)
    assert (np.abs(w32 - w64) <= bound).all()
    np.testing.assert_array_equal(w32[~touched], w0[~touched])
    assert (np.abs(c32[:, 0] - e64) <= adds * 2.0 ** -24 * (np.abs(c0[:, 0]) + sabs)).all()
    assert (np.abs(c32[:, 1] - a64) <= adds * 2.0 ** -24 * (np.abs(c0[:, 1]) + sabs)).all()


def test_python_argument_errors_without_gpu():
    import torch

    from ml2048_b200 import ops

    b = torch.zeros((4, 16), dtype=torch.uint8)
    w = torch.zeros(16, dtype=torch.float32)
    c = torch.zeros((16, 2), dtype=torch.float32)
    y = torch.zeros(4)
    with pytest.raises(ValueError):
        ops.ntuple_tc_update(b, y, w, c, c.clone(), [[0]], alpha=0.1)  # CPU tensors
    with pytest.raises(ValueError):
        ops.ntuple_tc_update(b, y, w, c, c.clone(), [[0, 0]], alpha=0.1)
    with pytest.raises(ValueError):
        ops.ntuple_tc_update(torch.zeros((4, 15), dtype=torch.uint8), y, w, c, c.clone(), [[0]], alpha=0.1)


def test_c_argument_errors_without_gpu(lib):
    """every check returns before a launch (the pointers below are never dereferenced)"""
    cells = np.zeros((2, 6), np.uint8)
    cells[0, :2] = (0, 1)
    cells[1, 0] = 5
    lens = np.array([2, 1], np.uint8)
    n = 16 ** 2 + 16
    B, W, CO, AC, D, T = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000, 0x60000

    def tc(*, after=B, target=T, w=W, coh=CO, acc=AC, nw=n, cl=cells.ctypes.data, k=2, delta=D, m=8):
        return lib.ml2048_tc_update(after, target, None, 0.1, w, coh, acc, nw, cl, lens.ctypes.data, k, delta, m, None)

    assert tc(m=0) == -3 and tc(m=-1) == -3
    for kw in ("after", "target", "w", "coh", "acc", "delta", "cl"):
        assert tc(**{kw: None}) == -1, kw
    assert tc(after=B + 8) == -2 and tc(target=T + 2) == -2 and tc(w=W + 2) == -2 and tc(delta=D + 1) == -2
    assert tc(coh=CO + 4) == -2 and tc(acc=AC + 4) == -2
    assert tc(nw=n - 1) == -3 and tc(k=0) == -3 and tc(k=17) == -3
    bad = cells.copy()
    bad[0, 1] = 0
    assert tc(cl=bad.ctypes.data) == -4


def test_header_declaration_compiles(tmp_path):
    """the new entry compiles from C with its documented argument types, and _lib.SYMBOLS lists it"""
    from ml2048_b200 import _lib

    src = tmp_path / "tc.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *y, uint8_t *m, float *w, float *c, float *a, uint8_t *cl, uint8_t *l, float *d, void *s) {\n"
        "  return ml2048_tc_update(b, y, m, 0.5f, w, c, a, 16, cl, l, 1, d, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "tc.o")], check=True)
    declared = set(re.findall(r"ML2048_API\s+[\w\s\*]+?\b(ml2048_tc_\w+)\s*\(", open(HEADER).read()))
    assert declared == {"ml2048_tc_update"}
    assert declared <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 12
