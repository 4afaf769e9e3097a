"""Policy stacks (GC_POLICY_TABLE_STACK) without a device: the argument checks of the Python layer, the ABI constants,
the numpy restatement the GPU tests drive the float64 table reference and the C oracle with, and the batched value
iteration of examples/posterior_sampling.py."""
import importlib.util
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

import _collect_oracle as CO
import _table_reference as TR
from conftest import REPO

torch = pytest.importorskip("torch")


# ---------------------------------------------------------------------------------------------
# the numpy restatement: env e takes the digits of policies[table_of_env[e]][index[e]]; exploration is the existing rule

class StackTableEnv(TR.TableEnv):
    """The float64 table reference whose table policy is a stack: `policy` is (policies [P, nS], table_of_env [n]).
    `policy_actions` / `collect` apply the reference's epsilon-greedy rule on top, unchanged."""

    def table_actions(self, policy):
        policies, m = policy
        p = np.asarray(policies, np.int64)[np.asarray(m, np.int64), self.index.astype(np.int64)]
        return np.stack([(p // self.A ** c) % self.A for c in range(self.C)]).astype(np.int8)


def oracle_stack_actions(ora, policies, m, epsilon):
    """int8 [C, n] actions of a policy stack for the C oracle's current step: each table's actions from the oracle's
    own table rule (gco_policy_actions), env e's taken from table m[e], then `_collect_oracle`'s explore rule."""
    per = np.stack([ora.policy_actions(np.asarray(p, np.int32)) for p in policies])          # [P, C, n]
    a = per[np.asarray(m, np.int64), :, np.arange(ora.n)].T.copy()
    view = SimpleNamespace(policy_actions=lambda _: a, global_step=ora.global_step, n=ora.n, cfg=ora.cfg, C=ora.C)
    return CO.explore_actions(view, None, epsilon)


def oracle_collect(ora, n_steps, policies, m, epsilon):
    """`_collect_oracle.collect` under a policy stack: (obs, action, reward, flags), each [n_steps, n]."""
    K, n = int(n_steps), ora.n
    obs, act = np.zeros((K, n), np.uint32), np.zeros((K, n), np.uint32)
    rew, flags = np.zeros((K, n), np.float64), np.zeros((K, n), np.uint8)
    radix = 5 if ora.cfg.kind == 1 else ora.cfg.n_actions
    place = np.array([radix ** c for c in range(ora.C)], np.uint64)
    for k in range(K):
        a = oracle_stack_actions(ora, policies, m, epsilon)
        obs[k] = ora.index
        act[k] = (a.astype(np.uint64) * place[:, None]).sum(0).astype(np.uint32)
        ora.step(a)
        rew[k] = ora.reward
        flags[k] = ora.unsafe | (ora.truncated << 1) | (ora.count << 2)
    return obs, act, rew, flags


def thread_mixed_map(n, P, seed):
    """Table ids [n] in [0, P) under which the 4 envs of a kernel thread (envs 4i .. 4i + 3) act by different tables
    (3 different ones at P = 3)."""
    shift = np.random.default_rng(seed).integers(0, P, (n + 3) // 4).repeat(4)[:n]
    return ((np.arange(n) % 4 + shift) % P).astype(np.int32)


def _tables(C, S, A, seed):
    from test_gpu_tables import make_tables
    return make_tables(seed, C, S, A, noise=True)


def _start(ref, seed):
    rng = np.random.default_rng(seed)
    ref.set_state((rng.random((ref.C, ref.n)) * ref.S).astype(np.int8), rng.integers(0, 3, ref.n).astype(np.int32))
    ref.global_step = 5


@pytest.mark.parametrize("eps", [0.0, 0.3])
def test_stack_of_one_is_the_table_policy(eps):
    from test_gpu_tables import f32_tables
    tabs = f32_tables(_tables(4, 3, 3, 1))
    n, K = 257, 6
    policy = np.random.default_rng(2).integers(0, 81, 81).astype(np.int32)
    one, stack = (cls(tabs, n, seed=9, max_episode_steps=3) for cls in (TR.TableEnv, StackTableEnv))
    _start(one, 3)
    _start(stack, 3)
    a, b = one.collect(K, policy, eps), stack.collect(K, (policy[None], np.zeros(n, np.int32)), eps)
    for k in a:
        assert (a[k] == b[k]).all(), k


@pytest.mark.parametrize("eps", [0.0, 0.3])
def test_mixed_stack_is_each_env_under_its_own_table(eps):
    """Env e of a stacked batch follows the trajectory of the same env under table m[e] alone."""
    from test_gpu_tables import f32_tables
    tabs = f32_tables(_tables(3, 3, 3, 4))
    n, K, P = 203, 7, 3
    policies = np.random.default_rng(5).integers(0, 27, (P, 27)).astype(np.int32)
    m = thread_mixed_map(n, P, 6)
    assert all(len(set(m[i:i + 4])) == 3 for i in range(0, n - 3, 4))
    stack = StackTableEnv(tabs, n, seed=9, env_id_offset=TR_BIG, max_episode_steps=3)
    _start(stack, 7)
    rec = stack.collect(K, (policies, m), eps)
    for j in range(P):
        one = TR.TableEnv(tabs, n, seed=9, env_id_offset=TR_BIG, max_episode_steps=3)
        _start(one, 7)
        want = one.collect(K, policies[j], eps)
        for k in rec:
            assert (rec[k][:, m == j] == want[k][:, m == j]).all(), (j, k)


TR_BIG = (1 << 32) + 4 * 12345


def test_oracle_stack_actions_match_table_reference():
    """The two restatements agree: the C oracle's table rule picked per env equals the table reference's stack on the
    reference's own tables (3 x 3 x 3 polarisation, noise)."""
    from oracle import oracle as O
    from gym_cellular_b200 import tables
    n, K, P = 64, 5, 4
    ora = O.OracleEnv(n_envs=n, noise=True, rng_episodic=True, seed=11, max_episode_steps=4)
    move, noisy, draws = tables.noise_tables(3, 3, False)
    tabs = dict(n_cells=3, n_states=3, n_actions=3, move=move, noisy=noisy, draws=draws,
                reward=tables.lower_reward(tables.right_polarizing, 3, 3, 3)[0],
                side_effects=tables.side_effect_tables(3, 3, "easy"), counted=tables.counted_levels(3))
    ref = StackTableEnv(tabs, n, seed=11, rng_episodic=True, max_episode_steps=4)
    policies = np.random.default_rng(1).integers(0, 27, (P, 27)).astype(np.int32)
    m = thread_mixed_map(n, P, 2)
    obs, act, _, flags = oracle_collect(ora, K, policies, m, 0.3)
    rec = ref.collect(K, (policies, m), 0.3)
    assert (obs == rec["obs"]).all() and (act == rec["action"]).all() and (flags == rec["flags"]).all()


# ---------------------------------------------------------------------------------------------
# argument checks of the Python layer (no device: CPU tensors against device "cpu")

def _check(*a):
    from gym_cellular_b200.vector_env import _check_policy_stack
    return _check_policy_stack(*a)


def test_argument_checks_need_no_device():
    cpu = torch.device("cpu")
    m = torch.zeros(10, dtype=torch.int32)
    out = _check(torch.zeros(3, 27, dtype=torch.int64), m, 27, 10, cpu)
    assert out.dtype == torch.int32 and out.shape == (3, 27) and out.is_contiguous()
    assert _check(np.zeros((1, 27), np.int16), m.to(torch.int64), 27, 10, cpu).shape == (1, 27)
    bad = [((None, m), "random policy"),
           ((torch.zeros(27, dtype=torch.int32), m), r"\[n_tables, 27\]"),
           ((torch.zeros(0, 27, dtype=torch.int32), m), r"\[n_tables, 27\]"),
           ((torch.zeros(2, 26, dtype=torch.int32), m), r"\[n_tables, 27\]"),
           ((torch.zeros(2, 27), m), "integer tabular actions"),
           ((torch.zeros(2, 27, dtype=torch.int32), m.numpy()), "torch tensor"),
           ((torch.zeros(2, 27, dtype=torch.int32), m.float()), "integer tensor"),
           ((torch.zeros(2, 27, dtype=torch.int32), m[:9]), r"shape \(10,\)"),
           ((torch.zeros(2, 27, dtype=torch.int32), m.view(2, 5)), r"shape \(10,\)")]
    for (policy, mp), msg in bad:
        with pytest.raises(ValueError, match=msg):
            _check(policy, mp, 27, 10, cpu)
    with pytest.raises(ValueError, match="lives on cpu"):
        _check(torch.zeros(2, 27, dtype=torch.int32), m, 27, 10, torch.device("meta"))


def test_abi_constant_and_export():
    from gym_cellular_b200 import _lib
    header = open(os.path.join(REPO, "include", "gym_cellular_b200.h")).read()
    assert int(re.search(r"#define GC_POLICY_TABLE_STACK\s+(\d+)", header).group(1)) == _lib.POLICY_TABLE_STACK == 2
    assert "gc_set_policy_stack" in _lib.EXPORTS and _lib.ABI_VERSION == 2


def test_set_policy_stack_rejects_a_null_handle():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    L = _lib.load()
    assert L.gc_set_policy_stack(None, None, 1) == _lib.ERR_INVALID and b"NULL" in L.gc_last_error()


# ---------------------------------------------------------------------------------------------
# the example's planner

def _example():
    spec = importlib.util.spec_from_file_location("posterior_sampling", os.path.join(REPO, "examples", "posterior_sampling.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_batched_value_iteration_plans_each_model():
    ex = _example()
    g = torch.Generator().manual_seed(0)
    nS, nA, M = 9, 4, 5
    P = torch.rand(M, nS, nA, nS, generator=g, dtype=torch.float64)
    P /= P.sum(-1, keepdim=True)
    R = torch.rand(nS, nA, generator=g, dtype=torch.float64)
    got = ex.plan(P, R)
    assert got.shape == (M, nS) and got.dtype == torch.int32
    for m in range(M):
        assert torch.equal(got[m], ex.value_iteration(P[m], R))


def test_posterior_samples_are_distributions_near_the_counts():
    ex = _example()
    torch.manual_seed(0)
    nxt = torch.zeros(3, 2, 3, dtype=torch.int64)
    nxt[0, 0] = torch.tensor([10 ** 6, 0, 0])
    counts = SimpleNamespace(next=nxt)
    P = ex.sample_models(counts, 7, prior=1.0)
    assert P.shape == (7, 3, 2, 3) and torch.allclose(P.sum(-1), torch.ones(7, 3, 2, dtype=torch.float64))
    assert (P[:, 0, 0, 0] > 0.999).all() and (P >= 0).all()


def test_reward_samples_narrow_with_visits():
    ex = _example()
    torch.manual_seed(1)
    visits = torch.tensor([[0, 10 ** 6]])
    counts = SimpleNamespace(visits=visits, reward_q24=torch.tensor([[0, 3 * 10 ** 6 * 2 ** 24]]))
    R = ex.sample_rewards(counts, 4000)
    assert R.shape == (4000, 1, 2)
    assert abs(float(R[:, 0, 0].std()) - 1.0) < 0.05 and abs(float(R[:, 0, 0].mean())) < 0.05
    assert (R[:, 0, 1] - 3.0).abs().max() < 0.01
