"""Pins the numpy table reference (tests/_table_reference.py) before any GPU test relies on it: on the table sets
`tables.py` lowers from the reference's rules it must equal the C oracle, and on the three debug MDPs the reference's
own outputs (tests/golden/debug.npz)."""
import numpy as np
import pytest

import _table_reference as TR
from gym_cellular_b200 import tables as T
from test_debug_envs import DET, _cases, _dexp_inputs

N = 515                          # not a multiple of 4 or 16
STEPS = 6
BIG_OFFSET = (1 << 32) + 4 * 1001
S_CHOICES = (2, 3, 4, 5, 8)
# noise mode: (noise, deadlock)
NOISE = ((False, False), (True, False), (True, True))
# C = 1..16 with S, difficulty, noise, counter, time limit and offset varied between rows (every S meets every noise
# mode and both counters across the 16 rows and the 32 wide rows below)
CASES = [(C, S_CHOICES[(C + k) % 5], T.DIFFICULTIES[(C + k) % 3], NOISE[(C + 2 * k) % 3], (C + k) % 2 == 0,
          3 if (C + k) % 4 < 2 else 0, BIG_OFFSET if (C + k) % 3 == 0 else 4 * C) for k in (0, 1) for C in range(1, 17)]


def _ids(case):
    C, S, diff, (noise, dead), epi, limit, off = case
    nz = "det" if not noise else ("deadlock" if dead else "noise")
    return f"C{C}-S{S}-{diff}-{nz}-{'epi' if epi else 'glob'}-lim{limit}-{'big' if off == BIG_OFFSET else 'small'}"


def reference_tables(C, S, difficulty, noise, deadlock, reward):
    if noise:
        move, noisy, draws = T.noise_tables(S, S, deadlock)
    else:
        move, noisy, draws = T.move_table(S, S), None, None
    return dict(n_cells=C, n_states=S, n_actions=S, move=move, noisy=noisy, draws=draws,
                reward=reward.table(S, S), side_effects=T.side_effect_tables(C, S, difficulty),
                counted=T.counted_levels(S))


@pytest.mark.parametrize("case", CASES, ids=[_ids(c) for c in CASES])
def test_reference_equals_oracle_on_reference_tables(case):
    from oracle import oracle as O
    C, S, diff, (noise, dead), epi, limit, off = case
    reward = T.nonlinear_right_polarizing if noise else (T.multiple_optima if C % 2 else T.right_polarizing)
    rid = "nonlinear_rp" if noise else reward.__name__
    seed, p = 0x9E3779B97F4A7C15 + C, 0.3
    ora = O.OracleEnv(n_envs=N, n_cells=C, n_states=S, reward=rid, difficulty=diff, noise=noise, deadlock=dead,
                      rng_episodic=epi, max_episode_steps=limit, noise_prob=p, seed=seed, env_id_offset=off)
    ref = TR.TableEnv(reference_tables(C, S, diff, noise, dead, reward), N, noise_prob=p, seed=seed, env_id_offset=off,
                      rng_episodic=epi, max_episode_steps=limit, reward_log2=reward.log2)
    rng = np.random.default_rng(C * 100 + S)
    cells = rng.integers(0, S, (C, N)).astype(np.int8)
    t0 = rng.integers(0, limit or 50, N).astype(np.int32)
    ora.state[:], ora.t[:], ora.index[:] = cells, t0, O.encode(cells, S)
    ref.set_state(cells, t0)
    ora.global_step = ref.global_step = 0xFFFFFFFE              # the global counter wraps at 2^32 on the way
    fired = 0
    for _ in range(STEPS):
        a = rng.integers(0, S, (C, N)).astype(np.int8)
        ora.step(a)
        ref.step(a)
        fired += int(ref.last_fire.sum())
        for k in ("state", "index", "t", "truncated", "unsafe", "count", "se_row"):
            assert (getattr(ref, k) == getattr(ora, k)).all(), k
        np.testing.assert_allclose(ref.reward_out, ora.reward, rtol=1e-12, atol=1e-15)
        assert (ref.stats == ora.stats).all()
    if noise:
        assert fired > 0
    assert ref.stats[1] > 0 or diff != "easy" or C == 1       # the easy tables report 'unsafe' at random states


@pytest.mark.parametrize("tag,make,S,A", DET)
def test_reference_on_deterministic_debug_mdps(golden_dbg, tag, make, S, A):
    g, tb = golden_dbg, make()
    s, a = _cases(S, A)
    ref = TR.TableEnv(tb, s.shape[1])
    ref.set_state(s)
    ref.step(a)
    assert (ref.state.T == g[f"{tag}_next"]).all()
    np.testing.assert_allclose(ref.reward_out, g[f"{tag}_reward"], rtol=0, atol=1e-15)
    assert (ref.se_row.T == g[f"{tag}_se"][:, 0, :]).all()
    assert (ref.unsafe == (g[f"{tag}_se"] == 2).any(axis=(1, 2))).all()
    assert (ref.count / 2 == g[f"{tag}_incidence"]).all()


def test_reference_on_deep_exploration(golden_dbg):
    """The reward_noisy case: the reward depends on whether the draw fired (replayed uniforms of the reference)."""
    g = golden_dbg
    s, a, u, ok = _dexp_inputs(g)
    ref = TR.TableEnv(T.deep_exploration_tables(), s.shape[1], replay=True)
    ref.set_state(s)
    ref.step(a, replay_u=np.nan_to_num(u, nan=0.0))
    assert (ref.state.T[ok] == g["dexp_next"][ok]).all()
    np.testing.assert_allclose(ref.reward_out[ok], g["dexp_reward"][ok], rtol=0, atol=1e-15)
    assert ref.last_fire.any() and (~ref.last_fire & ref.draws[s.astype(int), a.astype(int)]).any()


def test_reference_policies_equal_oracle():
    """Random and table actions of rollout / collect against the oracle's gco_policy_actions, on both counters."""
    from oracle import oracle as O
    C, S, n = 5, 4, 1030
    rng = np.random.default_rng(5)
    policy = rng.integers(0, S ** C, S ** C).astype(np.int32)
    for epi in (False, True):
        ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, rng_episodic=epi, seed=77, env_id_offset=BIG_OFFSET)
        ref = TR.TableEnv(reference_tables(C, S, "easy", False, False, T.right_polarizing), n, seed=77,
                          env_id_offset=BIG_OFFSET, rng_episodic=epi)
        cells = rng.integers(0, S, (C, n)).astype(np.int8)
        t0 = rng.integers(0, 50, n).astype(np.int32)
        ora.state[:], ora.t[:], ora.index[:] = cells, t0, O.encode(cells, S)
        ref.set_state(cells, t0)
        ora.global_step = ref.global_step = 12345
        for pol in (None, policy):
            assert (ref.policy_actions(pol) == ora.policy_actions(pol)).all()
