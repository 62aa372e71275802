"""The floating-point rollout ops on the GPU against plain high-precision references (tests/_rollout_ref.py):

    masked categorical sampler   stand-alone (ops.sample_masked_categorical) and inside the step kernel
                                 (VecGame.step_from_logits) vs the float64 inverse-CDF sample and log_softmax of the same
                                 uniform word, over logit classes, masks, sizes, slot bases and counters; exact edge cases
    GAE                          bit-exact vs the float32 recurrence at step counts on both sides of the 8-step unroll"""

from __future__ import annotations

import numpy as np
import pytest
import torch

import _rollout_ref as ref

pytestmark = pytest.mark.gpu

SEED = 0x9E3779B97F4A7C15  # both key words matter


@pytest.fixture(scope="module")
def ml():
    import ml2048_b200

    assert torch.cuda.is_available()
    return ml2048_b200


def _device_sampler(slot_base, counter, seed=SEED, dtype=torch.int64, valid_dtype=torch.uint8):
    from ml2048_b200.ops import sample_masked_categorical

    def sample(logits, valid):
        lg = torch.from_numpy(np.ascontiguousarray(logits, np.float32)).cuda()
        v = torch.from_numpy(np.ascontiguousarray(valid, np.uint8)).cuda().to(valid_dtype)
        a, lp = sample_masked_categorical(lg, v, seed=seed, counter=counter, slot_base=slot_base, dtype=dtype)
        return a.cpu().numpy(), lp.cpu().numpy()

    return sample


def _words(slot_base, n, counter, seed=SEED):
    return ref.policy_words(slot_base + np.arange(n, dtype=np.uint64), counter, seed)


SLOT_COUNTERS = [(0, 0), (5001, (3 << 32) + 1), ((1 << 34) + 17, 0), ((1 << 34) + 17, (3 << 32) + 1)]


def test_sampler_logit_classes_against_float64(ml):
    """Each logit class over 2^18 + 3 rows (masks: all 16 patterns, valid bytes 1..255; one class with bool masks): actions
    and log-probs within the rules of check_sampler; int64 and uint8 outputs give the same actions."""
    n = (1 << 18) + 3
    rng = np.random.default_rng(11)
    for i, name in enumerate(ref.LOGIT_CLASSES):
        base, counter = SLOT_COUNTERS[i % len(SLOT_COUNTERS)]
        words = _words(base, n, counter)
        logits = ref.sampler_logits(name, rng, words)
        valid = ref.random_masks(rng, n, wide=name != "ties")
        if name == "boundary":
            valid = ref.boundary_valid(valid)
        vdt = torch.bool if name == "ties" else torch.uint8
        a, lp = _device_sampler(base, counter, valid_dtype=vdt)(logits, valid)
        a8, lp8 = _device_sampler(base, counter, dtype=torch.uint8, valid_dtype=vdt)(logits, valid)
        assert a.dtype == np.int64 and a8.dtype == np.uint8
        np.testing.assert_array_equal(a8.astype(np.int64), a, err_msg=name)
        np.testing.assert_array_equal(lp8.view(np.uint32), lp.view(np.uint32), err_msg=name)
        stats = ref.check_sampler(logits, valid, words, a, lp, adversarial=name == "boundary", what=name)
        if name == "boundary":
            assert stats["boundary_rows"] > n // 4


@pytest.mark.parametrize("n", [1, 255, 256, 257])
def test_sampler_sizes_slot_bases_counters(ml, n):
    """Sizes that end inside, at and just past a 256-thread block (2^18 + 3: the class test above) x slot bases 0, odd and
    beyond 2^32 x counters 0 and beyond 2^32, both output dtypes: each row draws slot_word(slot_base + row, counter, seed),
    checked through the action."""
    rng = np.random.default_rng(n)
    for base in (0, 5001, (1 << 34) + 17):
        for counter in (0, (3 << 32) + 1):
            words = _words(base, n, counter)
            logits = ref.sampler_logits("randn3", rng, words)
            valid = ref.random_masks(rng, n)
            for dtype in (torch.int64, torch.uint8):
                a, lp = _device_sampler(base, counter, dtype=dtype)(logits, valid)
                ref.check_sampler(logits, valid, words, a, lp, what=f"n={n} base={base} counter={counter} {dtype}")
            # all four actions valid with equal logits: the action is the top two bits of the word, exactly
            a, _ = _device_sampler(base, counter)(np.zeros((n, 4), np.float32), np.ones((n, 4), np.uint8))
            np.testing.assert_array_equal(a, words.astype(np.int64) >> 30)


# at this counter and SEED, global slot 2^34 + 17 + 3224657 draws the word 0xAAAAAB76: u = 0xAAAAAB / 2^24 is 2^-24 above 2/3,
# so with three equal valid logits only the 24th bit of the uniform makes the action the third valid one
SLOT_ON_TWO_THIRDS = (1 << 34) + 17 + 3224657


def test_sampler_exact_cases(ml):
    """One valid / no valid action, equal logits, NaN / +-inf logits masked or valid: exact outcomes
    (_rollout_ref.check_sampler_exact), also for an odd slot base and a uniform on the 2/3 boundary."""
    counter = (3 << 32) + 1
    assert ref.policy_words(np.array([SLOT_ON_TWO_THIRDS], np.uint64), counter, SEED)[0] == 0xAAAAAB76
    for base, n in (((1 << 34) + 17, 4099), (SLOT_ON_TWO_THIRDS - 1, 2)):
        ref.check_sampler_exact(_device_sampler(base, counter), _words(base, n, counter), np.random.default_rng(5))


@pytest.mark.parametrize("rng_mode", ["replay", "philox"])
def test_step_from_logits_against_float64(ml, rng_mode):
    """The sampler inside the step kernel: 40 steps with resets, every logit class in turn, a batch at slot base 0 and one
    of 70 001 games at an odd slot base beyond 2^32.  Before each step the mask is observations()[1] and the word
    slot_word(slot_base + game, counter, seed) of the counter the kernel is about to use."""
    names = ref.LOGIT_CLASSES
    resets = 0
    for m, base in ((5000, 0), (70001, (1 << 33) + 1)):
        env = ml.VecGame(m, output="torch", rng_mode=rng_mode, slot_base=base, sync_free=True)
        env.reset(4)
        rng = np.random.default_rng(m)
        lp_out = torch.empty(m, device="cuda")
        for t in range(40):
            resets += int((env.observations()[1].sum(dim=1) == 0).sum())  # finished games: prepare() resets them
            env.prepare()
            valid = env.observations()[1].cpu().numpy()
            words = _words(base, m, env._philox_counter, env._philox_seed)
            name = names[t % len(names)]
            logits = ref.sampler_logits(name, rng, words)
            env.step_from_logits(torch.from_numpy(logits).cuda(), log_prob_out=lp_out)
            a, lp = env.sampled_actions.cpu().numpy(), lp_out.cpu().numpy()
            ref.check_sampler(logits, valid, words, a, lp, adversarial=name == "boundary", what=f"m={m} t={t} {name}")
    assert resets > 0


GAE_CASES = [  # (use, step, game): every step count, the games 1 / 255 / 257 / 4097 and uses 1 / 3 each appear
    (1, 1, 257), (3, 7, 1), (1, 8, 4097), (3, 9, 255), (1, 15, 257), (3, 17, 4097), (1, 65, 255), (3, 130, 257),
    (3, 1, 4097), (1, 9, 1),
]


@pytest.mark.parametrize("use,steps,games", GAE_CASES)
def test_gae_bit_exact_across_the_unroll(ml, use, steps, games):
    """GAE bit-exact against the float32 recurrence at step counts below, at and on both sides of multiples of the 8-step
    unroll; (gamma, lambda) = (0.997, 0.95), (1, 1), (0.9, 0); terminated as bool and as uint8 0 / 1 / 255, with
    terminations on the first and the last step; `out` pre-filled with NaN so that an element left unwritten fails."""
    from ml2048_b200.ops import gae_advantages

    g = torch.Generator(device="cuda").manual_seed(steps * 10007 + games)
    shape = (use, steps, games)
    v0 = torch.randn(shape, device="cuda", generator=g) * 30
    v1 = torch.randn(shape, device="cuda", generator=g) * 30
    reward = (torch.randint(0, 128, shape, device="cuda", generator=g) * 4).float()
    ended = torch.rand(shape, device="cuda", generator=g) < 0.1
    ended[:, 0, ::3] = True
    ended[:, -1, 1::3] = True
    for gamma, lam in ((0.997, 0.95), (1.0, 1.0), (0.9, 0.0)):
        wide = torch.where(ended, torch.randint(0, 2, shape, device="cuda", generator=g) * 254 + 1, 0).to(torch.uint8)
        for term in (ended, wide):  # uint8 holding 0, 1 and 255
            out = torch.full(shape, float("nan"), device="cuda")
            got = gae_advantages(v0, v1, reward, term, gamma=gamma, lambda_=lam, out=out)
            assert got.data_ptr() == out.data_ptr()
            want = ref.ref_gae(v0, v1, reward, term, gamma, lam)
            assert not torch.isnan(want).any()
            bad = (got.view(torch.int32) != want.view(torch.int32)).nonzero()
            assert bad.numel() == 0, (gamma, lam, term.dtype, bad[:4].tolist(), got[tuple(bad[0])].item(), want[tuple(bad[0])].item())
