"""
Delayed TD(lambda) / TC(lambda) without a GPU: the NumPy definition (tests/_lambda_ref.py) against scalar loops written from
the definition and against the float64 weighted sum of n-step returns, h = 1 against TD(0)'s target, and the checks of the
Python and C arguments and of the header that need no device.
"""

from __future__ import annotations

import os
import re
import subprocess

import numpy as np
import pytest

import _lambda_ref as ref
import _ntuple_ref as nref

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(HERE), "include", "ml2048_b200.h")

LAMS = (0.0, 0.5, 1.0, 0.3)
HORIZONS = (1, 2, 3, 16)


@pytest.fixture(scope="module")
def lib():
    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    return _lib.load()


def _loop(v, rho, e, lam, alpha):
    """the definition for one game, one scalar float32 operation at a time, from R_{h-1} down"""
    f = np.float32
    lf = f(lam)
    c = f(f(1) - lf)
    h = len(v) - 1
    with np.errstate(all="ignore"):
        r = f(0) if e[h - 1] else f(f(rho[h]) + f(v[h]))
        for k in range(h - 2, -1, -1):
            r = f(0) if e[k] else f(f(f(rho[k + 1]) + f(c * f(v[k + 1]))) + f(lf * r))
        return f(f(alpha) * f(r - f(v[0])))


def _loop_from_first_end(v, rho, e, lam, alpha):
    """the kernel's order: find the first end, start there, never read a value after it"""
    f = np.float32
    lf = f(lam)
    c = f(f(1) - lf)
    h = len(v) - 1
    ends = [k for k in range(h) if e[k]]
    with np.errstate(all="ignore"):
        if ends:
            top, r = ends[0], f(0)
        else:
            top, r = h - 1, f(f(rho[h]) + f(v[h]))
        for k in range(top - 1, -1, -1):
            r = f(f(f(rho[k + 1]) + f(c * f(v[k + 1]))) + f(lf * r))
        return f(f(alpha) * f(r - f(v[0]))), (ends[0] if ends else h)


def _same(got, want):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    nan = np.isnan(want)
    np.testing.assert_array_equal(np.isnan(got), nan)
    np.testing.assert_array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))


def _windows(rng, h: int, m: int, special: bool):
    """window-ordered V (h+1, M), rho (h+1, M), ended (h+1, M): game i has its first end at k = i mod (h+1) (h = none),
    every third game a second end later; with `special`, NaN / +-inf values and +-0 rewards"""
    v = (rng.standard_normal((h + 1, m)) * 3000).astype(np.float32)
    rho = rng.choice(np.array([0, 4, 8, 16, 32, 64, 128, 1024], np.float32), size=(h + 1, m))
    e = np.zeros((h + 1, m), np.uint8)
    for i in range(m):
        first = i % (h + 1)
        if first < h:
            e[first, i] = 1
            if i % 3 == 0 and first + 1 < h:
                e[rng.integers(first + 1, h), i] = 1
    e[h] = rng.integers(0, 2, m)  # the newest slot's flag is not read
    if special:
        v.flat[rng.choice(v.size, v.size // 10, replace=False)] = np.nan
        v.flat[rng.choice(v.size, v.size // 10, replace=False)] = np.inf
        v.flat[rng.choice(v.size, v.size // 10, replace=False)] = -np.inf
        v.flat[rng.choice(v.size, v.size // 20, replace=False)] = -0.0
        rho.flat[rng.choice(rho.size, rho.size // 4, replace=False)] = -0.0
    return v, rho, e


@pytest.mark.parametrize("special", [False, True])
@pytest.mark.parametrize("h", HORIZONS)
def test_reference_against_scalar_loops(h, special):
    """bit for bit against both loops; values after the first end replaced by garbage change no bit"""
    rng = np.random.default_rng(100 * h + special)
    m = 6 * (h + 1)
    v, rho, e = _windows(rng, h, m, special)
    for lam in LAMS:
        for alpha in (0.01, 1.0):
            want = ref.lambda_delta(v, rho, e, lam, alpha)
            _same(want, [_loop(v[:, i], rho[:, i], e[:, i], lam, alpha) for i in range(m)])
            got, firsts = zip(*[_loop_from_first_end(v[:, i], rho[:, i], e[:, i], lam, alpha) for i in range(m)])
            _same(want, got)
            assert set(firsts) == set(range(h + 1))  # an end at every window position, and none
            vg, rg = v.copy(), rho.copy()
            for i, first in enumerate(firsts):
                vg[first + 1:, i] = np.nan  # after the first end: V_{m+1..h} and rho_{m+1..h}
                rg[first + 1:, i] = np.inf
            _same(ref.lambda_delta(vg, rg, e, lam, alpha), want)
    mask = (rng.random(m) < 0.6).astype(np.uint8)
    d = ref.lambda_delta(v, rho, e, 0.5, 0.1, mask)
    assert (d[mask == 0].view(np.uint32) == 0).all()


@pytest.mark.parametrize("h", HORIZONS)
def test_reference_against_float64_nstep_returns(h):
    """R_0 is the lambda-weighted sum of the n-step returns truncated at the first end, within float32 rounding: each of the
    h levels rounds c, the product, two adds and lf * R, on terms bounded by T = sum_k |rho_k| + |V_k|"""
    rng = np.random.default_rng(7 + h)
    m = 40 * (h + 1)
    v, rho, e = _windows(rng, h, m, False)
    t = np.abs(rho[1:].astype(np.float64)).sum(0) + np.abs(v.astype(np.float64)).sum(0)
    for lam in LAMS + (0.25, 0.75, 0.9):
        got = ref.lambda_return(v, rho, e, lam).astype(np.float64)
        want = ref.nstep_weighted_f64(v, rho, e, lam)
        bound = (5 * h + 1) * 2.0 ** -24 * t
        assert (np.abs(got - want) <= bound).all(), (lam, (np.abs(got - want) - bound).max())
    # lambda = 0 is the one-step target, 0 where x_0's game ended
    first = np.argmax(np.vstack([e[:h], np.ones((1, m), np.uint8)]), axis=0)
    with np.errstate(all="ignore"):
        one = np.where(first == 0, np.float32(0), rho[1] + v[1]).astype(np.float32)
    _same(ref.lambda_return(v, rho, e, 0.0), one)


def test_h1_is_td0_target():
    """h = 1: R_0 = reward + value with masked_fill(ended, 0), the TD(0) learner's target, and delta is TD(0)'s delta"""
    import torch

    rng = np.random.default_rng(5)
    tuples = ((0, 1, 2), (5, 6), (3,))
    n = nref.num_weights(tuples)
    m = 500
    w = (rng.standard_normal(n) * 50).astype(np.float32)
    w[::9] = np.nan
    w[1::13] = -0.0
    after = rng.integers(0, 14, size=(2, m, 16)).astype(np.uint8)
    reward = rng.choice(np.array([0, -0.0, 4, 12, 2048, np.inf], np.float32), size=(2, m))
    ended = rng.integers(0, 2, size=(2, m)).astype(np.uint8)
    mask = (rng.random(m) < 0.7).astype(np.uint8)
    for newest in (0, 1):
        for lam in LAMS:
            d, x0 = ref.ring_delta(after, reward, ended, newest, w, tuples, lam, 0.01, mask)
            old = 1 - newest
            value = torch.from_numpy(nref.value(after[newest], w, tuples))
            target = torch.add(torch.from_numpy(reward[newest]), value).masked_fill(torch.from_numpy(ended[old]).bool(), 0.0)
            v = np.stack([nref.value(after[old], w, tuples), value.numpy()])
            _same(ref.lambda_return(v, np.stack([reward[old], reward[newest]]), np.stack([ended[old], ended[newest]]), lam),
                  target.numpy())
            np.testing.assert_array_equal(x0, after[old])
            with np.errstate(all="ignore"):
                _same(d, nref.td_delta(after[old], target.numpy(), w, tuples, 0.01, mask))


def test_window_order():
    ring = np.arange(5)[:, None] * 10 + np.zeros((5, 2), np.int64)
    for newest in range(5):
        win = ref.window(ring, newest)
        assert win[4, 0] == 10 * newest  # x_h is the newest slot
        assert win[0, 0] == 10 * ((newest + 1) % 5)  # x_0 the slot after it
        assert list(win[:, 0]) == [10 * ((newest - (4 - k)) % 5) for k in range(5)]


def test_python_argument_errors_without_gpu():
    import torch

    from ml2048_b200 import ops

    m, h = 4, 3
    a = torch.zeros((h + 1, m, 16), dtype=torch.uint8)
    r = torch.zeros((h + 1, m))
    e = torch.zeros((h + 1, m), dtype=torch.uint8)
    w = torch.zeros(16)
    c = torch.zeros((16, 2))

    def both(*args, **kw):
        kw = dict(dict(alpha=0.1, lam=0.5), **kw)
        args = list(args) + [a, r, e, 0][len(args):]
        errs = []
        for fn, extra in ((ops.ntuple_td_lambda_update, (w,)), (ops.ntuple_tc_lambda_update, (w, c, c.clone()))):
            with pytest.raises(ValueError) as info:
                fn(*args, *extra, [[0]], **kw)
            errs.append(str(info.value))
        assert errs[0] == errs[1]
        return errs[0]

    assert "after_ring" in both(a[0])
    assert "after_ring" in both(a.float())
    assert "horizon" in both(a[:1], r[:1], e[:1])
    assert "horizon" in both(torch.zeros((18, m, 16), dtype=torch.uint8))
    for bad in (-1, h + 1, True, 1.0):
        assert "newest" in both(a, r, e, bad)
    for bad in (-0.1, 1.5, float("nan"), "x", None):
        assert "lam" in both(lam=bad)
    assert "contiguous CUDA tensor" in both()  # CPU tensors


def test_c_argument_errors_without_gpu(lib):
    """every check returns before a launch (the pointers below are never dereferenced)"""
    cells = np.zeros((2, 6), np.uint8)
    cells[0, :2] = (0, 1)
    cells[1, 0] = 5
    lens = np.array([2, 1], np.uint8)
    n = 16 ** 2 + 16
    B, R, E, W, CO, AC, D = 0x10000, 0x20000, 0x30000, 0x40000, 0x50000, 0x60000, 0x70000

    def td(*, after=B, rew=R, end=E, h=3, newest=0, lam=0.5, w=W, nw=n, cl=cells.ctypes.data, k=2, delta=D, m=8):
        return lib.ml2048_lambda_td_update(after, rew, end, h, newest, lam, None, 0.1, w, nw, cl, lens.ctypes.data, k, delta, m,
                                           None)

    def tc(*, after=B, rew=R, end=E, h=3, newest=0, lam=0.5, w=W, coh=CO, acc=AC, nw=n, cl=cells.ctypes.data, k=2, delta=D,
           m=8):
        return lib.ml2048_lambda_tc_update(after, rew, end, h, newest, lam, None, 0.1, w, coh, acc, nw, cl, lens.ctypes.data, k,
                                           delta, m, None)

    for fn in (td, tc):
        assert fn(m=0) == -3 and fn(m=-1) == -3
        for kw in ("after", "rew", "end", "w", "delta", "cl"):
            assert fn(**{kw: None}) == -1, kw
        assert fn(after=B + 8) == -2 and fn(rew=R + 2) == -2 and fn(w=W + 2) == -2 and fn(delta=D + 1) == -2
        for h, newest in ((0, 0), (17, 0), (-1, 0), (3, 4), (3, -1), (1, 2)):
            assert fn(h=h, newest=newest) == -3, (h, newest)
        for lam in (-0.25, 1.001, float("nan"), float("inf"), -float("inf")):
            assert fn(lam=lam) == -4, lam
        assert fn(nw=n - 1) == -3 and fn(k=0) == -3 and fn(k=17) == -3
        bad = cells.copy()
        bad[0, 1] = 0
        assert fn(cl=bad.ctypes.data) == -4
    assert tc(coh=None) == -1 and tc(acc=None) == -1
    assert tc(coh=CO + 4) == -2 and tc(acc=AC + 4) == -2


def test_header_declaration_compiles(tmp_path):
    """the new entries compile from C with their documented argument types, and _lib.SYMBOLS lists them"""
    from ml2048_b200 import _lib

    src = tmp_path / "lambda.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *r, uint8_t *e, uint8_t *m, float *w, float *c, float *a, uint8_t *cl, uint8_t *l, float *d,\n"
        "      void *s) {\n"
        "  return ml2048_lambda_td_update(b, r, e, 3, 0, 0.5f, m, 0.1f, w, 16, cl, l, 1, d, 1, s) +\n"
        "         ml2048_lambda_tc_update(b, r, e, 3, 0, 0.5f, m, 0.1f, w, c, a, 16, cl, l, 1, d, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "lambda.o")], check=True)
    declared = set(re.findall(r"ML2048_API\s+[\w\s\*]+?\b(ml2048_lambda_\w+)\s*\(", open(HEADER).read()))
    assert declared == {"ml2048_lambda_td_update", "ml2048_lambda_tc_update"}
    assert declared <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 12
