"""
``TDAfterstateLearner`` on the GPU in lock step with the reference learner (tests/_learner_ref.py) over the C oracle.

The device learner runs on ``VecGame(M, kind, two_prob=..., output="torch", sync_free=True)`` in replay mode, which is bit
for bit the oracle's game; the reference runs on ``OracleVecGame`` from the same seed.  Before every device step the
device's weights, coherence and marks are read back and handed to the reference step, so that both choose their moves
on the same weights (no near tie can flip on the float32 rounding of the atomics), and after it:

- bit for bit: every field of the step result, the chosen action, ``learner.delta``, the promotion marks, and every
  weight and coherence entry that no masked-in x_0 touched (one comparison on the device);
- within the float32 bounds of the atomics (``_td_tolerance_check`` / ``_tc_tolerance_check``): the touched weights and
  coherence against the reference's float64 apply.

Rules TD(0), TC, TD(lambda) (h = 3, lambda = 0.5) and TC(lambda) (h = 2, lambda = 0.25), each on the 4 x 4-tuple network
SMALL with one stage, with stages (3, 5) and with stages (3, 5) and promotion (the storage behind every clear mark starts
as NaN), M = 257 games for 150 steps; the four reward kinds and two_prob 0.8 / 0.5 / 1 spread over the twelve runs.  Games
end inside every run and the updated afterstates cover every stage; one run per rule calls reset(seed) midway.  Also
alpha = 0 (nothing changes, the greedy policy's game) and the standard 4 x 6-tuple network at M = 1024 for 8 steps.
Measured on one B200 (power limit not recorded): 50 s for the file, 1.9-6.0 s per run; the host reference's oracle moves
and float64 applies take most of it.
"""

from __future__ import annotations

import numpy as np
import pytest
import torch

import _learner_ref as lr
import _stage_ref as sref
from _ntuple_gpu import _gpu, ops  # noqa: F401 (ops is a fixture)
from oracle.rollout import FIELDS
from test_ntuple import _td_tolerance_check
from test_stages import KINDS, SMALL, _same_bits
from test_tc import _tc_tolerance_check

RULES = {"td0": ("td0", 1, 0.5), "tc": ("tc", 1, 0.5), "td_lambda": ("td0", 3, 0.5), "tc_lambda": ("tc", 2, 0.25)}
NETS = {"single": ((), False), "staged": ((3, 5), False), "promoted": ((3, 5), True)}
DTYPES = {name: dt for name, dt, _ in FIELDS}


def _start_weights(net, seed: int, scale: float = 4.0) -> None:
    """random weights in every stage; with promotion every mark is clear, and the storage behind them NaN"""
    g = torch.Generator(device=net.device)
    g.manual_seed(seed)
    net.weights.copy_(torch.randn(net.weights.shape, device=net.device, generator=g) * scale)
    if net.promoted is not None:
        net.weights[net.promoted.numel():] = float("nan")


def _check_result(res, want: dict, t: int) -> None:
    for k in lr.RESULT_KEYS:
        got = np.ascontiguousarray(res[k].cpu().numpy(), DTYPES[k])
        exp = np.ascontiguousarray(want[k], DTYPES[k])
        if got.dtype.kind == "f":
            got, exp = got.view(np.uint32), exp.view(np.uint32)
        np.testing.assert_array_equal(got, exp, err_msg=f"result field {k!r} at step {t}")


def _check_update(net, upd, w_before, c_before, p_before, t: int) -> None:
    """the device's weights, coherence and marks after a step against the reference's expected update (None: no update)"""
    if p_before is not None:
        want_p = p_before.cpu().numpy() if upd is None else upd["marks"]
        np.testing.assert_array_equal(net.promoted.cpu().numpy(), want_p, err_msg=f"marks at step {t}")
    if upd is None:
        assert torch.equal(net.weights.view(torch.int32), w_before.view(torch.int32)), f"weights changed at step {t}"
        if c_before is not None:
            assert torch.equal(net.coherence.view(torch.int32), c_before.view(torch.int32))
        return
    touched = upd["adds"] > 0
    keep = torch.from_numpy(~touched).to(net.device)
    assert torch.equal(net.weights[keep].view(torch.int32), w_before[keep].view(torch.int32)), f"untouched weights at step {t}"
    idx = np.flatnonzero(touched)
    i_dev = torch.from_numpy(idx).to(net.device)
    got_w = net.weights[i_dev].cpu().numpy()
    if "e64" not in upd:
        _td_tolerance_check(got_w, upd["w0"][idx], upd["w64"][idx], upd["adds"][idx], upd["sabs"][idx])
        return
    c0 = torch.zeros((net.weights.numel(), 2), device=net.device) if c_before is None else c_before
    assert torch.equal(net.coherence[keep].view(torch.int32), c0[keep].view(torch.int32)), f"untouched coherence at step {t}"
    _tc_tolerance_check(got_w, net.coherence[i_dev].cpu().numpy(), upd["w0"][idx], upd["c0"][idx], upd["w64"][idx],
                        upd["e64"][idx], upd["a64"][idx], upd["adds"][idx], upd["sabs"][idx])
    assert not bool(net._tc_accum.view(torch.int32).any()), "the accumulator is not all zero bits"


def _lockstep(oracle, dev, *, tuples, stages, promotion, rule, h, lam, kind, two_prob, m, steps, seed, alpha=None,
              reset_at=None, start_seed=0):
    from ml2048_b200 import VecGame
    from ml2048_b200.ntuple import NTupleNetwork, TDAfterstateLearner

    net = NTupleNetwork(tuples, device=dev, stages=stages, promotion=promotion)
    _start_weights(net, start_seed)
    env = VecGame(m, kind, two_prob=two_prob, output="torch", sync_free=True)
    learner = TDAfterstateLearner(env, net, alpha=alpha, rule=rule, horizon=h, lam=lam)
    ref = lr.RefLearner(oracle, m, kind, two_prob, tuples, stages=stages, promotion=promotion, rule=rule, horizon=h, lam=lam,
                        alpha=learner.alpha)
    stats = {"ends": 0, "stages": set(), "updates": 0}
    since_reset = 0
    for t in range(steps):
        if t == 0 or t == reset_at:
            learner.reset(seed + t)
            ref.reset(seed + t)
            since_reset = 0
        w_before = net.weights.clone()
        c_before = None if net.coherence is None else net.coherence.clone()
        p_before = None if net.promoted is None else net.promoted.clone()
        want = ref.step(w_before.cpu().numpy(), None if c_before is None else c_before.cpu().numpy(),
                        None if p_before is None else p_before.cpu().numpy())
        res = learner.step()
        _check_result(res, want["result"], t)
        np.testing.assert_array_equal(learner._out["action"].cpu().numpy().astype(np.int64), want["action"])
        _same_bits(learner.delta.cpu().numpy(), want["delta"], f"delta at step {t}")
        _check_update(net, want["update"], w_before, c_before, p_before, t)
        if since_reset < h:  # nothing to update yet: no pending afterstate (h = 1) or a window still filling (h > 1)
            assert not bool(learner.delta.any())
            assert torch.equal(net.weights.view(torch.int32), w_before.view(torch.int32))
        upd = want["update"]
        if upd is not None and upd["adds"].any():
            stats["updates"] += 1
            stats["stages"] |= set(sref.stage(upd["x0"][upd["mask"]], stages).tolist())
        stats["ends"] += int(want["result"]["terminated"].sum())
        since_reset += 1
    return net, stats


CONFIGS = [(r, n) for r in RULES for n in NETS]


@pytest.mark.gpu
@pytest.mark.parametrize("rule,net", CONFIGS)
def test_learner_lockstep(ops, oracle, rule, net):
    i = CONFIGS.index((rule, net))
    r, h, lam = RULES[rule]
    stages, promotion = NETS[net]
    steps = 150
    reset_at = 100 if net == "staged" else None
    _, stats = _lockstep(oracle, _gpu(), tuples=SMALL, stages=stages, promotion=promotion, rule=r, h=h, lam=lam,
                         kind=KINDS[i % 4], two_prob=(0.8, 0.5, 1.0)[i % 3], m=257, steps=steps, seed=100 + i,
                         reset_at=reset_at, start_seed=i)
    assert stats["ends"] > 0
    assert stats["stages"] == set(range(len(stages) + 1)), stats["stages"]
    assert stats["updates"] == steps - h * (2 if reset_at else 1)


@pytest.mark.gpu
def test_learner_lockstep_alpha_zero(ops, oracle):
    """alpha = 0: no update at all (weights, coherence and marks as they were), and the game is the greedy policy's"""
    net, stats = _lockstep(oracle, _gpu(), tuples=SMALL, stages=(3, 5), promotion=True, rule="tc", h=2, lam=0.5,
                           kind="improved", two_prob=0.8, m=257, steps=60, seed=7, alpha=0.0, start_seed=3)
    assert stats["updates"] == 0 and net.coherence is None and not bool(net.promoted.any())


@pytest.mark.gpu
def test_learner_lockstep_standard_network(ops, oracle):
    """the standard 4 x 6-tuple network (256 MiB of weights), single stage, TD(0), M = 1024 for 8 steps"""
    from ml2048_b200.ntuple import STANDARD_4X6

    _, stats = _lockstep(oracle, _gpu(), tuples=STANDARD_4X6, stages=(), promotion=False, rule="td0", h=1, lam=0.5,
                         kind="normal", two_prob=0.8, m=1024, steps=8, seed=11, start_seed=5)
    assert stats["updates"] == 7
