"""Pins the float32 reward model (tests/_reward_f32.py) before the GPU tests compare reward bits with it: exact on
dyadic tables, within the float32 summation bound on uniform ones, and equal to the C oracle's rewards on the
reference's own tables (the envs test_gpu_packed.py::test_packed_equals_int8_bit_for_bit runs)."""
import numpy as np
import pytest

import _reward_f32 as RF
import _table_reference as TR
from gym_cellular_b200 import tables as T
from test_table_reference_cpu import reference_tables

N = 515


def _tables(rng, C, S, A, fam, noise):
    def rew():
        if fam == "dyadic":
            return rng.integers(-8 * 256, 8 * 256 + 1, (S, A)) / 256.0
        return rng.uniform(-1.0, 1.0, (S, A)).astype(np.float32).astype(np.float64)
    tabs = dict(n_cells=C, n_states=S, n_actions=A, move=rng.integers(0, S, (S, A)), reward=rew(),
                side_effects=np.zeros((C, S, S), np.int8), counted=np.ones(S, np.uint8))
    if noise:
        tabs.update(noisy=rng.integers(0, S, (S, A)), draws=rng.random((S, A)) < 0.5, reward_noisy=rew())
    return tabs


def _steps(tabs, n=N, steps=4, seed=0):
    rng = np.random.default_rng(seed)
    ref = TR.TableEnv(tabs, n, noise_prob=0.4, seed=seed, max_episode_steps=3)
    ref.set_state(rng.integers(0, ref.S, (ref.C, n)), rng.integers(0, 3, n))
    for _ in range(steps):
        ref.step(rng.integers(0, ref.A, (ref.C, n)))
        yield ref


CASES = [(C, noise) for C in (1, 2, 3, 4, 5, 7, 8, 9, 16) for noise in (False, True)]


@pytest.mark.parametrize("C,noise", CASES, ids=[f"C{C}-{'noise' if z else 'det'}" for C, z in CASES])
def test_model_exact_on_dyadic_tables(C, noise):
    tabs = _tables(np.random.default_rng(C), C, 4, 3, "dyadic", noise)
    fired = 0
    for ref in _steps(tabs, seed=C):
        fired += int(ref.last_fire.sum())
        for fam in (RF.PAIR, RF.SINGLE):
            got = RF.prelog(ref, fam)
            assert (got.astype(np.float64) == ref.reward_pre_log).all(), fam
            assert not np.signbit(got[got == 0]).any()
    assert fired > 0 or not noise


@pytest.mark.parametrize("C,noise", CASES, ids=[f"C{C}-{'noise' if z else 'det'}" for C, z in CASES])
def test_model_within_float32_bound_on_uniform_tables(C, noise):
    tabs = _tables(np.random.default_rng(100 + C), C, 4, 3, "uniform", noise)
    differs = 0
    for ref in _steps(tabs, seed=C):
        pair, single = RF.prelog(ref, RF.PAIR), RF.prelog(ref, RF.SINGLE)
        for got in (pair, single):
            assert (np.abs(got.astype(np.float64) - ref.reward_pre_log) <= RF.sum_bound(ref)).all()
        differs += int((RF.bits(pair) != RF.bits(single)).sum())
    if C >= 4:                                  # up to three cells the two orders are the same sum
        assert differs > 0                      # the two families round differently: the model tells them apart


def test_model_of_single_cell_is_the_entry():
    tabs = _tables(np.random.default_rng(7), 1, 4, 4, "uniform", True)
    for ref in _steps(tabs):
        want = np.where(ref.last_fire[0], ref.reward_noisy[ref.last_s[0], ref.last_a[0]],
                        ref.reward[ref.last_s[0], ref.last_a[0]]).astype(np.float32)
        for fam in (RF.PAIR, RF.SINGLE):
            assert (RF.bits(RF.prelog(ref, fam)) == RF.bits(want)).all()


def test_negative_zero_entries_sum_to_positive_zero():
    tabs = _tables(np.random.default_rng(3), 3, 4, 3, "dyadic", False)
    tabs["reward"] = np.where(np.arange(12).reshape(4, 3) % 2 == 0, -0.0, 0.25)
    zero = 0
    for ref in _steps(tabs):
        for fam in (RF.PAIR, RF.SINGLE):
            got = RF.prelog(ref, fam)
            assert (got.astype(np.float64) == ref.reward_pre_log).all()
            zero += int((got == 0).sum())
            assert (RF.bits(got[got == 0]) == 0).all()
    assert zero > 0


# The C oracle sums the reference's rules in float64; the model from the float32 tables the device receives must
# equal it within the float32 bound, and its log2(1 + .) within the accuracy the README states.
PACKED_ENVS = [(C, S, z) for C, S in [(16, 4), (3, 3), (2, 3), (7, 2), (13, 4)] for z in (False, True)]


@pytest.mark.parametrize("C,S,stochastic", PACKED_ENVS,
                         ids=[f"C{C}-S{S}-{'stochastic' if z else 'det'}" for C, S, z in PACKED_ENVS])
def test_model_reproduces_the_reference_envs(C, S, stochastic):
    from oracle import oracle as O
    reward = T.nonlinear_right_polarizing if stochastic else T.right_polarizing
    tabs = reference_tables(C, S, "easy", stochastic, False, reward)
    f32 = dict(tabs, reward=np.asarray(tabs["reward"], np.float32))
    ora = O.OracleEnv(n_envs=N, n_cells=C, n_states=S, reward="nonlinear_rp" if stochastic else "right_polarizing",
                      noise=stochastic, rng_episodic=True, seed=3, max_episode_steps=6)
    ref = TR.TableEnv(f32, N, seed=3, rng_episodic=True, max_episode_steps=6, reward_log2=reward.log2)
    rng = np.random.default_rng(C * 10 + S)
    for _ in range(5):
        a = rng.integers(0, S, (C, N)).astype(np.int8)
        ora.step(a)
        ref.step(a)
        assert (ref.state == ora.state).all()
        pre = RF.prelog(ref, RF.PAIR).astype(np.float64)
        bound = RF.sum_bound(ref) + C * 2.0 ** -24 * np.abs(reward.table(S, S)).max()   # + the tables' rounding
        if reward.log2:
            got = np.log2(1.0 + pre)
            assert (np.abs(got - ora.reward) <= bound / ((1 + pre) * np.log(2)) + 6e-7 * np.abs(ora.reward) + 1e-12).all()
        else:
            assert (np.abs(pre - ora.reward) <= bound).all()
