"""tools/eval_cnn.py restates the reference's CNN actor (policy/_network.py, policy/actor_critic.py:240-284) so that
BASELINE configs[4] can run without the reference installed.  The restatement is held to what the repository records of the
reference -- its parameter count, probed from the live policy (SURVEY.md section 2, row 7) -- and its logits are pinned by
tests/golden/cnn_actor_logits.npz.  Given the ``src`` directory of a checkout of the reference in ML2048_REFERENCE_SRC, it
is also held to the reference itself: same parameter names (a reference state dict loads), same logits.  Caller context,
not product -- but the evaluation numbers quote it.

    python tests/test_eval_cnn_network.py      # rewrites tests/golden/cnn_actor_logits.npz from the restatement"""

from __future__ import annotations

import os
import sys
import types

import numpy as np
import torch

REF_SRC = os.environ.get("ML2048_REFERENCE_SRC")
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN_LOGITS = os.path.join(HERE, "golden", "cnn_actor_logits.npz")
# CNNActorCriticPolicy(share_encoder=True): encoder + actor + critic MLP 1024 -> 256 -> 64 -> 1, probed on the reference
REFERENCE_POLICY_PARAMS = 1_451_077
CRITIC_PARAMS = (1024 * 256 + 256) + (256 * 64 + 64) + (64 * 1 + 1)


def _load_tool():
    path = os.path.join(os.path.dirname(HERE), "tools", "eval_cnn.py")
    src = open(path).read().replace("import ml2048_b200\n", "")  # the networks need neither CUDA nor the extension
    mod = types.ModuleType("eval_cnn_under_test")
    mod.__file__ = path
    exec(compile(src, path, "exec"), mod.__dict__)
    return mod


def test_actor_restatement_matches_the_reference_policy():
    tool = _load_tool()
    mine = tool.ActorPolicy().eval()
    assert sum(p.numel() for p in mine.parameters()) + CRITIC_PARAMS == REFERENCE_POLICY_PARAMS
    if REF_SRC is None:
        return  # the reference's own policy is not at hand: the recorded parameter count is what can be checked
    sys.path.insert(0, REF_SRC)
    try:
        from ml2048.policy.actor_critic import CNNActorCriticPolicy
    finally:
        sys.path.remove(REF_SRC)
    torch.manual_seed(3)
    ref = CNNActorCriticPolicy(share_encoder=True).eval()
    assert sum(p.numel() for p in ref.parameters()) == REFERENCE_POLICY_PARAMS
    missing, unexpected = mine.load_state_dict(ref.state_dict(), strict=False)
    assert not missing
    assert all(k.startswith("_critic.") for k in unexpected), unexpected  # the evaluation only needs the actor
    boards = torch.randint(0, 16, (513, 16))
    valid = torch.ones((513, 4), dtype=torch.bool)
    with torch.no_grad():
        want = ref.action_logits(boards, valid)
        onehot = torch.nn.functional.one_hot(boards, 16).float().permute(0, 2, 1).contiguous()  # policy/_network.py:86-95
        got = mine(onehot)
    torch.testing.assert_close(got, want, rtol=0, atol=1e-6)  # fp32, same op order up to the fused input encoding


def _pinned_logits(tool):
    """The restated actor with weights drawn from a seeded NumPy generator (stable across torch versions, unlike
    torch's initialisers), scaled by 1/sqrt(fan-in), applied to 513 seeded boards."""
    rng = np.random.default_rng(2048)
    net = tool.ActorPolicy().eval()
    state = {}
    for name, t in net.state_dict().items():
        fan_in = t[0].numel() if t.dim() > 1 else 1
        state[name] = torch.from_numpy(rng.standard_normal(tuple(t.shape)).astype(np.float32) / np.float32(np.sqrt(fan_in)))
    net.load_state_dict(state)
    boards = torch.from_numpy(rng.integers(0, 16, (513, 16)))
    onehot = torch.nn.functional.one_hot(boards, 16).float().permute(0, 2, 1).contiguous()
    with torch.no_grad():
        logits = net(onehot)
    names = np.array(list(state))
    numels = np.array([state[k].numel() for k in state], np.int64)
    return names, numels, logits.numpy()


def test_actor_restatement_logits_are_pinned():
    """Names, sizes and logits of the restated actor stay what they were when the fixture was written (fp32 on the CPU:
    the tolerance covers a different convolution algorithm on another host)."""
    names, numels, logits = _pinned_logits(_load_tool())
    with np.load(GOLDEN_LOGITS, allow_pickle=False) as z:
        np.testing.assert_array_equal(names, z["names"])
        np.testing.assert_array_equal(numels, z["numels"])
        np.testing.assert_allclose(logits, z["logits"], rtol=1e-4, atol=1e-5)
    assert logits.shape == (513, 4) and np.all(logits.max(axis=1) == 0.0) and logits.min() < -0.1


def test_actor_restatement_shapes_without_the_reference():
    tool = _load_tool()
    torch.manual_seed(0)
    net = tool.ActorPolicy().eval()
    x = torch.zeros((7, 16, 16))
    x[:, 0, :] = 1.0  # empty boards
    with torch.no_grad():
        logits = net(x)
    assert logits.shape == (7, 4) and float(logits.max()) == 0.0  # translated so that max = 0 (policy/_network.py:181-185)


if __name__ == "__main__":
    names, numels, logits = _pinned_logits(_load_tool())
    np.savez_compressed(GOLDEN_LOGITS, names=names, numels=numels, logits=logits)
    print(GOLDEN_LOGITS, logits.shape)
