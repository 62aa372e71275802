"""
N-tuple networks without a GPU: the NumPy reference (tests/_ntuple_ref.py) against brute-force loops, the symmetry maps as the
dihedral group, the product's index / value arithmetic (board_ops.cuh compiled for the host by tests/host_shim/ntuple_host.cpp)
against the reference, and the checks of the spec and of the C arguments that need no device.
"""

from __future__ import annotations

import ctypes
import itertools
import os
import re
import subprocess

import numpy as np
import pytest

import _ntuple_ref as ref

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SHIM_SRC = os.path.join(HERE, "host_shim", "ntuple_host.cpp")
HEADER = os.path.join(ROOT, "include", "ml2048_b200.h")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("ntuple_shim") / "libntuple_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas", "-o", so, SHIM_SRC], check=True)
    lib = ctypes.CDLL(so)
    vp, i64, i32, u32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_uint32
    lib.nt_sym_src.argtypes = [u32, u32]
    lib.nt_sym_src.restype = u32
    lib.nt_expand.argtypes = [vp, vp, i32, vp, vp]
    lib.nt_expand.restype = i64
    lib.nt_index_batch.argtypes = [vp, i64, vp, vp, i32, i32, i32, vp]
    lib.nt_value_batch.argtypes = [vp, i64, vp, vp, vp, i32, vp]
    return lib


@pytest.fixture(scope="module")
def lib():
    from ml2048_b200 import _lib, build

    build.build()  # nvcc cross-compiles without a GPU; no-op when up to date
    return _lib.load()


def _spec_arrays(tuples):
    cells = np.zeros((len(tuples), 6), np.uint8)
    for i, t in enumerate(tuples):
        cells[i, :len(t)] = t
    return cells, np.array([len(t) for t in tuples], np.uint8)


def _random_tuples(rng, k: int, lengths=None):
    lengths = lengths if lengths is not None else rng.integers(1, 7, size=k)
    return tuple(tuple(int(c) for c in rng.permutation(16)[:n]) for n in lengths)


def _boards(rng, m: int) -> np.ndarray:
    """exponents 0..17 with many empty cells, plus arbitrary bytes in every fourth board"""
    b = np.where(rng.random((m, 16)) < 0.4, 0, rng.integers(1, 18, size=(m, 16))).astype(np.uint8)
    b[::4] = rng.integers(0, 256, size=b[::4].shape, dtype=np.uint8)
    return b


# ---- the reference against brute force ----------------------------------------------------------


def _brute_src(g: int, cell: int) -> int:
    r, c = divmod(cell, 4)
    rc = [(r, c), (r, 3 - c), (3 - r, c), (3 - r, 3 - c), (c, r), (c, 3 - r), (3 - c, r), (3 - c, 3 - r)][g]
    return 4 * rc[0] + rc[1]


def _brute_value(board, w, tuples, dtype):
    acc = dtype(0)
    off = 0
    for cells in tuples:
        for g in range(8):
            idx = 0
            for j, c in enumerate(cells):
                idx += min(int(board[_brute_src(g, c)]), 15) * 16 ** j
            acc = dtype(acc + dtype(w[off + idx]))
        off += 16 ** len(cells)
    return acc


def test_reference_against_brute_force():
    rng = np.random.default_rng(0)
    for g in range(8):
        assert [_brute_src(g, c) for c in range(16)] == list(ref.SRC[g])
    for k in (1, 2, 5):
        tuples = _random_tuples(rng, k, lengths=rng.integers(1, 4, size=k))
        w = rng.standard_normal(ref.num_weights(tuples)).astype(np.float32)
        boards = _boards(rng, 64)
        got = ref.value(boards, w, tuples)
        want = np.array([_brute_value(b, w, tuples, np.float32) for b in boards], np.float32)
        np.testing.assert_array_equal(got.view(np.uint32), want.view(np.uint32))


def test_reference_greedy_and_td_against_loops():
    rng = np.random.default_rng(1)
    tuples = ((0, 1, 2), (5, 9))
    n = ref.num_weights(tuples)
    w = np.round(rng.standard_normal(n) * 8).astype(np.float32)
    m = 200
    boards = _boards(rng, m)
    after = rng.integers(0, 6, size=(m, 4, 16)).astype(np.uint8)
    reward = rng.integers(0, 3, size=(m, 4)).astype(np.float32)
    valid = rng.integers(0, 2, size=(m, 4)).astype(np.uint8)
    valid[:20] = 0
    got = ref.greedy(boards, after, reward, valid, w, tuples)
    for i in range(m):
        qs = [(reward[i, a] + _brute_value(after[i, a], w, tuples, np.float32), a) for a in range(4) if valid[i, a]]
        if not qs:
            assert got["action"][i] == 0 and (got["state"][i] == boards[i]).all() and got["reward"][i] == 0 and got["value"][i] == 0
            continue
        best = max(qs, key=lambda qa: (qa[0], -qa[1]))[1]
        assert got["action"][i] == best
        assert (got["state"][i] == after[i, best]).all() and got["reward"][i] == reward[i, best]
    target = rng.standard_normal(m).astype(np.float32)
    mask = rng.integers(0, 2, m).astype(np.uint8)
    d = ref.td_delta(boards, target, w, tuples, 0.25, mask)
    w32 = ref.td_apply_f32(boards, d, w, tuples, mask)
    w64, cnt, _ = ref.td_apply_f64(boards, d, w, tuples, mask)
    loop = w.astype(np.float64).copy()
    adds = np.zeros(n, np.int64)
    for i in range(m):
        if not mask[i]:
            assert d[i] == 0
            continue
        assert d[i] == np.float32(np.float32(0.25) * np.float32(target[i] - _brute_value(boards[i], w, tuples, np.float32)))
        off = 0
        for cells in tuples:
            for g in range(8):
                e = off + sum(min(int(boards[i][_brute_src(g, c)]), 15) * 16 ** j for j, c in enumerate(cells))
                loop[e] += d[i]
                adds[e] += 1
            off += 16 ** len(cells)
    np.testing.assert_allclose(w64, loop, rtol=0, atol=1e-9)
    np.testing.assert_array_equal(cnt, adds)
    np.testing.assert_allclose(w32, loop, rtol=1e-5, atol=1e-4)  # float32 adds


def test_symmetries_are_the_dihedral_group():
    maps = {tuple(int(x) for x in row) for row in ref.SRC}
    assert len(maps) == 8
    for a, b in itertools.product(ref.SRC, ref.SRC):
        assert tuple(int(x) for x in a[b]) in maps  # closed under composition
    assert tuple(range(16)) in maps
    rng = np.random.default_rng(2)
    tuples = _random_tuples(rng, 6)
    w = rng.integers(-1000, 1000, size=ref.num_weights(tuples)).astype(np.float64)  # integers: float64 sums are exact
    boards = _boards(rng, 300)
    v = _value64(boards, w, tuples)
    for g in range(8):
        np.testing.assert_array_equal(_value64(ref.image(boards, g), w, tuples), v)


def _value64(boards, w, tuples):
    return w[ref.entries(boards, tuples)].sum(axis=1)


# ---- the product's arithmetic, compiled for the host ------------------------------------------------


def test_host_symmetry_map(shim):
    for g in range(8):
        assert [shim.nt_sym_src(g, c) for c in range(16)] == list(ref.SRC[g])


def test_host_expand_offsets(shim):
    rng = np.random.default_rng(3)
    for k in (1, 4, 16):
        tuples = _random_tuples(rng, k)
        cells, lens = _spec_arrays(tuples)
        offs = np.zeros(k, np.uint32)
        src4 = np.zeros((k, 8, 8), np.uint8)
        assert shim.nt_expand(cells.ctypes.data, lens.ctypes.data, k, offs.ctypes.data, src4.ctypes.data) == ref.num_weights(tuples)
        assert list(offs) == ref.offsets(tuples)
        for t, tup in enumerate(tuples):
            for g in range(8):
                assert list(src4[t, g, :len(tup)]) == [4 * ref.SRC[g][c] for c in tup]


def test_host_index_every_image_every_byte(shim):
    """every g, random tuples of every length, boards of arbitrary bytes (cells 0..255) and every byte in every cell"""
    rng = np.random.default_rng(4)
    every_byte = np.repeat(np.arange(256, dtype=np.uint8)[:, None], 16, axis=1)
    shifted = np.stack([np.roll(np.arange(256, dtype=np.uint8), 17 * c) for c in range(16)], axis=1)
    boards = np.concatenate([_boards(rng, 4096), rng.integers(0, 256, (4096, 16), dtype=np.uint8), every_byte, shifted])
    n = boards.shape[0]
    tuples = _random_tuples(rng, 12, lengths=[1, 2, 3, 4, 5, 6, 6, 5, 4, 3, 2, 1])
    cells, lens = _spec_arrays(tuples)
    out = np.zeros(n, np.uint32)
    for t, tup in enumerate(tuples):
        for g in range(8):
            shim.nt_index_batch(boards.ctypes.data, n, cells.ctypes.data, lens.ctypes.data, len(tuples), t, g, out.ctypes.data)
            want = ref.index(boards, tup, g)
            np.testing.assert_array_equal(out.astype(np.int64), want)
            assert (want < 16 ** len(tup)).all()


def test_host_value_bit_exact(shim):
    rng = np.random.default_rng(5)
    for tuples in (ref.STANDARD_4X6, _random_tuples(rng, 1, [6]), _random_tuples(rng, 16), _random_tuples(rng, 7, [1] * 7)):
        cells, lens = _spec_arrays(tuples)
        w = (rng.standard_normal(ref.num_weights(tuples)) * 100).astype(np.float32)
        boards = np.concatenate([_boards(rng, 2000), rng.integers(0, 256, (500, 16), dtype=np.uint8)])
        out = np.zeros(boards.shape[0], np.float32)
        shim.nt_value_batch(boards.ctypes.data, boards.shape[0], w.ctypes.data, cells.ctypes.data, lens.ctypes.data, len(tuples),
                            out.ctypes.data)
        np.testing.assert_array_equal(out.view(np.uint32), ref.value(boards, w, tuples).view(np.uint32))


# ---- spec and argument checks ------------------------------------------------------------------


def test_spec_validation():
    from ml2048_b200 import ops
    from ml2048_b200.ntuple import STANDARD_4X6

    assert STANDARD_4X6 == ref.STANDARD_4X6
    assert ops.ntuple_spec([[0, 1], (2,)]) == ((0, 1), (2,))
    assert ops.ntuple_num_weights(STANDARD_4X6) == 4 * 16 ** 6
    for bad in ([], [[]], [[0, 1, 2, 3, 4, 5, 6]], [[16]], [[-1]], [[3, 3]], [[0]] * 17, 5, [[0, "x"]], [1, 2]):
        with pytest.raises(ValueError):
            ops.ntuple_spec(bad)


def test_python_argument_errors_without_gpu():
    import torch

    from ml2048_b200 import ops

    b = torch.zeros((4, 16), dtype=torch.uint8)
    w = torch.zeros(16, dtype=torch.float32)
    with pytest.raises(ValueError):
        ops.ntuple_value(b, w, [[0]])  # CPU tensors
    with pytest.raises(ValueError):
        ops.ntuple_value(torch.zeros((4, 15), dtype=torch.uint8), w, [[0]])
    with pytest.raises(ValueError):
        ops.ntuple_greedy(b, w, [[0]], action_dtype=torch.int32)
    with pytest.raises(ValueError):
        ops.ntuple_greedy(b, w, [[0]], reward_fn=lambda s, p, m: 0.0)
    with pytest.raises(ValueError):
        ops.ntuple_td_update(b, torch.zeros(4), w, [[0, 0]], alpha=0.1)


def test_c_argument_errors_without_gpu(lib):
    """every check returns before a launch (the pointers below are never dereferenced)"""
    cells, lens = _spec_arrays(((0, 1), (5,)))
    n = 16 ** 2 + 16
    B, W, O = 0x10000, 0x20000, 0x30000
    c, ln = cells.ctypes.data, lens.ctypes.data

    def value(*, board=B, w=W, nw=n, cl=c, l=ln, k=2, out=O, m=8):
        return lib.ml2048_ntuple_value(board, w, nw, cl, l, k, out, m, None)

    assert value(m=0) == -3 and value(m=-1) == -3
    assert value(board=None) == -1 and value(w=None) == -1 and value(out=None) == -1 and value(cl=None) == -1 and value(l=None) == -1
    assert value(board=B + 4) == -2 and value(w=W + 2) == -2 and value(out=O + 1) == -2
    assert value(k=0) == -3 and value(k=17) == -3
    assert value(nw=n + 1) == -3 and value(nw=16 ** 2) == -3
    for tuples_cells, tuples_len, rc in ((((0, 1), (5,)), (7, 1), -3), (((0, 1), (5,)), (0, 1), -3), (((0, 16), (5,)), (2, 1), -4),
                                         (((0, 0), (5,)), (2, 1), -4), (((0, 255), (5,)), (2, 1), -4)):
        cc = np.zeros((2, 6), np.uint8)
        for i, t in enumerate(tuples_cells):
            cc[i, :len(t)] = t
        ll = np.array(tuples_len, np.uint8)
        assert value(cl=cc.ctypes.data, l=ll.ctypes.data) == rc

    def greedy(*, kind=0, u8=O, i64=None, after=0x40000, m=8, cl=c):
        return lib.ml2048_ntuple_greedy(B, W, n, cl, ln, 2, kind, u8, i64, after, 0x50000, 0x60000, m, None)

    assert greedy(m=0) == -3 and greedy(u8=None) == -1 and greedy(after=None) == -1
    assert greedy(u8=None, i64=O + 4) == -2 and greedy(after=0x40008) == -2
    assert greedy(kind=4) == -4 and greedy(kind=-1) == -4

    def td(*, mask=None, m=8, nw=n, delta=0x70000, target=0x80000):
        return lib.ml2048_ntuple_td_update(B, target, mask, 0.1, W, nw, c, ln, 2, delta, m, None)

    assert td(m=0) == -3 and td(delta=None) == -1 and td(target=None) == -1
    assert td(delta=0x70002) == -2 and td(nw=n - 1) == -3


def test_header_declarations_compile(tmp_path):
    """the new entries compile from C with their documented argument types, and _lib.SYMBOLS lists them"""
    from ml2048_b200 import _lib

    src = tmp_path / "nt.c"
    src.write_text(
        f'#include "{HEADER}"\n'
        "int f(void *b, float *w, uint8_t *c, uint8_t *l, float *v, uint8_t *a8, int64_t *a64, void *s) {\n"
        "  return ml2048_ntuple_value(b, w, 16, c, l, 1, v, 1, s) + ml2048_ntuple_greedy(b, w, 16, c, l, 1, 0, a8, a64, b, v, v, 1, s)\n"
        "       + ml2048_ntuple_td_update(b, v, a8, 0.5f, w, 16, c, l, 1, v, 1, s);\n}\n")
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "nt.o")], check=True)
    declared = set(re.findall(r"ML2048_API\s+[\w\s\*]+?\b(ml2048_ntuple_\w+)\s*\(", open(HEADER).read()))
    assert declared == {"ml2048_ntuple_value", "ml2048_ntuple_greedy", "ml2048_ntuple_td_update"}
    assert declared <= set(_lib.SYMBOLS)
    assert _lib.ABI_VERSION == 12
