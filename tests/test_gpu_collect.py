"""Experience collection (gc_collect / `collect`): the fused K-step rollout that records every transition, with
epsilon-greedy table policies.  Against the oracle step by step, against the step kernel replayed with the recorded
actions, against `rollout()`, and across layouts, shards and large record strides."""
import ctypes as C
import importlib.util
import os

import numpy as np
import pytest
from scipy import stats as sps

import _collect_oracle as CO
from conftest import REPO

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

REWARD_RTOL = 1e-6
REWARD_ATOL = 1e-7


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def host(t):
    return t.cpu().numpy()


def u32(t):
    return host(t).view(np.uint32)


def _flags(unsafe, truncated, count):
    return unsafe.astype(np.uint8) | (truncated.astype(np.uint8) << 1) | (count.astype(np.uint8) << 2)


def _check_collect(env, ora, K, policy=None, eps=0.0, reps=2):
    n = env.num_envs
    for _ in range(reps):
        tr = env.collect(K, policy, eps)
        obs, act, rew, flags = CO.collect(ora, K, policy, eps)
        assert tr.obs.shape == (K, n) and tr.next_obs is None
        assert (u32(tr.obs) == obs).all()
        assert (u32(tr.action) == act).all()
        assert (host(tr.flags) == flags).all()
        np.testing.assert_allclose(host(tr.reward), rew, rtol=REWARD_RTOL, atol=REWARD_ATOL)
        assert (host(env.state) == ora.state).all()
        assert (host(env.time_step) == ora.t).all()
        assert (u32(env.tabular_state(torch.int32)) == ora.index).all()
    s = env.stats()
    assert s["env_steps"] == ora.stats[0] == reps * K * n and s["unsafe_steps"] == ora.stats[1]
    assert s["count_sum"] == ora.stats[2] and s["episodes_truncated"] == ora.stats[3]
    assert abs(s["reward_sum"] * 2 ** 24 - ora.stats[4]) <= reps * K * n


CELL_CASES = {                     # name: (env kwargs, oracle kwargs)
    "det1": (dict(n_cells=1), dict(n_cells=1, rng_episodic=True)),
    "det3": (dict(), dict(rng_episodic=True)),
    "det5": (dict(n_cells=5), dict(n_cells=5, rng_episodic=True)),
    "det8": (dict(n_cells=8), dict(n_cells=8, rng_episodic=True)),
    "stoch3_episodic_deadlock": (dict(stochastic=True, deadlock=True, rng_episodic=True),
                                 dict(noise=True, deadlock=True, rng_episodic=True, reward="nonlinear_rp")),
    "stoch3_global": (dict(stochastic=True, rng_episodic=False), dict(noise=True, rng_episodic=False, reward="nonlinear_rp")),
    "stoch16x4_hard": (dict(n_cells=16, n_states=4, stochastic=True, difficulty="hard"),
                       dict(n_cells=16, n_states=4, noise=True, rng_episodic=True, difficulty="hard", reward="nonlinear_rp")),
}


@pytest.mark.parametrize("case", sorted(CELL_CASES))
@pytest.mark.parametrize("pol", ["random", "table", "eps"])
def test_collect_cellular_vs_oracle(B, O, case, pol):
    ekw, okw = CELL_CASES[case]
    n = 10007
    C = ekw.get("n_cells", 3)
    S = ekw.get("n_states", 3)
    if pol != "random" and S ** C > 10 ** 5:
        pytest.skip("no tabular policy for 4^16 states")
    env = B.CellularVectorEnv(num_envs=n, env_seed=21, max_episode_steps=5, **ekw)
    ora = O.OracleEnv(n_envs=n, seed=21, max_episode_steps=5, **okw)
    policy = None if pol == "random" else np.random.default_rng(C).integers(0, S ** C, S ** C).astype(np.int32)
    _check_collect(env, ora, 12, policy, 0.3 if pol == "eps" else 0.0)


def _gw_policy(golden_gw):
    policy = np.zeros(400, np.int32)
    st, pol = golden_gw["gw_states"].astype(int), golden_gw["gw_initial_policy"].astype(int)
    policy[st[:, 0] + 20 * st[:, 1]] = pol[:, 0] + 5 * pol[:, 1]
    return policy


@pytest.mark.parametrize("pol", ["random", "table", "eps"])
def test_collect_gridworld_vs_oracle(B, O, golden_gw, pol):
    n = 10007
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=9, dispersal_prob=0.05, max_episode_steps=7)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=9, dispersal_prob=0.05, max_episode_steps=7)
    policy = None if pol == "random" else _gw_policy(golden_gw)
    _check_collect(env, ora, 16, policy, 0.3 if pol == "eps" else 0.0)
    env.check_actions()


# ---------------------------------------------------------------------------------------------
# replay: the recorded actions fed to the step kernel reproduce the record bit for bit

@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_replay_equals_step_kernel(B, golden_gw, kind):
    n, K = 10007, 11
    kw = dict(stochastic=True, rng_episodic=False) if kind == "cellular" else dict(dispersal_prob=0.2)
    env = B.CellularVectorEnv(kind=kind, num_envs=n, env_seed=4, max_episode_steps=4, **kw)
    twin = B.CellularVectorEnv(kind=kind, num_envs=n, env_seed=4, max_episode_steps=4, emit_final_obs=True, **kw)
    policy = (np.random.default_rng(0).integers(0, 27, 27).astype(np.int32) if kind == "cellular" else _gw_policy(golden_gw))
    tr = env.collect(K, policy, 0.4, next_obs=True)
    for k in range(K):
        _, reward, _, trunc, infos = twin.step(twin.detabularize(tr.action[k], "action"))
        nxt = tr.obs[k + 1] if k + 1 < K else env.tabular_state(torch.int32)
        assert torch.equal(twin.tabular_state(torch.int32), nxt)
        assert torch.equal(reward.view(torch.int32), tr.reward[k].view(torch.int32))
        assert torch.equal(_flags_t(infos["unsafe"], trunc, infos["count"]), tr.flags[k])
        fin = twin.tabularize(torch.stack(infos["final_obs"]))
        assert torch.equal(fin.to(torch.int32), tr.next_obs[k])
        assert bool(trunc.any()) or k % 4 != 3
    assert torch.equal(twin.state, env.state) and torch.equal(twin.time_step, env.time_step)


def _flags_t(unsafe, trunc, count):
    return unsafe.to(torch.uint8) | (trunc.to(torch.uint8) << 1) | (count.to(torch.uint8) << 2)


# ---------------------------------------------------------------------------------------------
# recording changes nothing

@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
@pytest.mark.parametrize("pol", ["random", "table"])
def test_collect_advances_like_rollout(B, golden_gw, kind, pol):
    n, K = 10007, 19
    kw = dict(stochastic=True) if kind == "cellular" else {}
    envs = [B.CellularVectorEnv(kind=kind, num_envs=n, env_seed=8, max_episode_steps=6, **kw) for _ in range(2)]
    policy = None
    if pol == "table":
        policy = (np.random.default_rng(1).integers(0, 27, 27).astype(np.int32) if kind == "cellular" else _gw_policy(golden_gw))
    tr = envs[0].collect(K, policy)
    envs[1].rollout(K, policy)
    a, b = envs
    assert torch.equal(a.state, b.state) and torch.equal(a.time_step, b.time_step)
    assert torch.equal(a.tabular_state(torch.int32), b.tabular_state(torch.int32))
    assert a.stats() == b.stats() and a.launch_count == b.launch_count
    if policy is not None and kind == "cellular":
        assert (u32(tr.action) == policy[u32(tr.obs)]).all()


# ---------------------------------------------------------------------------------------------
# epsilon statistics

def _pvalue_uniform(counts):
    return sps.chisquare(counts, np.full(len(counts), counts.sum() / len(counts))).pvalue


def test_epsilon_one_is_uniform(B, golden_gw):
    env = B.CellularVectorEnv(num_envs=1 << 16, stochastic=True, env_seed=31)
    tr = env.collect(16, np.zeros(27, np.int32), 1.0)
    assert _pvalue_uniform(np.bincount(u32(tr.action).ravel(), minlength=27)) > 1e-4
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=1 << 16, env_seed=31)
    tr = gw.collect(16, _gw_policy(golden_gw), 1.0)
    counts = np.bincount(u32(tr.action).ravel(), minlength=25)
    codes = [4 + 5 * p for p in range(4)] + [p + 20 for p in range(4)]
    assert counts[codes].sum() == tr.action.numel()
    assert _pvalue_uniform(counts[codes]) > 1e-4


def test_epsilon_quarter_fraction(B):
    eps, N = 0.25, (1 << 16) * 16
    policy = np.random.default_rng(2).integers(0, 27, 27).astype(np.int32)
    env = B.CellularVectorEnv(num_envs=1 << 16, stochastic=True, env_seed=32)
    tr = env.collect(16, policy, eps)
    frac = (u32(tr.action) != policy[u32(tr.obs)]).mean()
    p = eps * (1 - 1 / 27)
    assert abs(frac - p) < 5 * np.sqrt(p * (1 - p) / N)


def test_exploration_uses_the_global_step(B):
    """Episodic noise replays every episode; exploration must not: the non-greedy steps of an env differ between two
    consecutive episodes (a deterministic env restarts from the same state, so with episode-keyed draws they would not)."""
    n, T = 4096, 16
    policy = np.zeros(27, np.int32)
    env = B.CellularVectorEnv(num_envs=n, rng_episodic=True, env_seed=33, max_episode_steps=T)
    tr = env.collect(2 * T, policy, 0.5)
    nongreedy = host(tr.action) != 0
    assert (nongreedy[:T] != nongreedy[T:]).any(axis=0).mean() > 0.99


# ---------------------------------------------------------------------------------------------
# packed layout and shards

@pytest.mark.parametrize("shape", [(3, 3), (16, 4)])
def test_packed_equals_int8(B, shape):
    C, S = shape
    n = 10007
    kw = dict(num_envs=n, n_cells=C, n_states=S, stochastic=True, env_seed=6, max_episode_steps=5,
              difficulty="hard" if C == 16 else "easy")
    a, p = B.CellularVectorEnv(**kw), B.PackedCellularVectorEnv(**kw)
    policy, eps = (np.random.default_rng(3).integers(0, 27, 27).astype(np.int32), 0.3) if C == 3 else (None, 0.0)
    for _ in range(2):
        ta, tp = a.collect(9, policy, eps, next_obs=True), p.collect(9, policy, eps, next_obs=True)
        for f in ("obs", "action", "reward", "flags", "next_obs"):
            assert torch.equal(getattr(ta, f), getattr(tp, f)), f
    assert torch.equal(p.unpack(p._state)[:, :n], a.state)
    assert torch.equal(p.tabular_state(torch.int32), a.tabular_state(torch.int32))
    assert torch.equal(p.time_step, a.time_step) and p.stats() == a.stats()


def test_shards_reproduce_one_handle(B):
    n, h = 20008, 10004
    policy = np.random.default_rng(5).integers(0, 27, 27).astype(np.int32)
    kw = dict(stochastic=True, rng_episodic=False, env_seed=7, max_episode_steps=6)
    whole = B.CellularVectorEnv(num_envs=n, **kw).collect(14, policy, 0.3, next_obs=True)
    parts = [B.CellularVectorEnv(num_envs=h, env_id_offset=o, **kw).collect(14, policy, 0.3, next_obs=True) for o in (0, h)]
    for f in ("obs", "action", "reward", "flags", "next_obs"):
        assert torch.equal(torch.cat([getattr(p, f) for p in parts], 1), getattr(whole, f)), f


# ---------------------------------------------------------------------------------------------
# large strides, NULL fields, status

def test_large_record_stride_flags_only(B):
    """2^24 envs x 129 steps: the record spans more than 2^31 elements; only flags are recorded."""
    from gym_cellular_b200 import _lib
    n, K = 1 << 24, 129
    kw = dict(num_envs=n, n_cells=16, n_states=4, stochastic=True, env_seed=41, max_episode_steps=50,
              emit_side_effects=False)
    env = B.CellularVectorEnv(**kw)
    assert K * env.ld > 2 ** 31
    flags = torch.zeros(K, env.ld, dtype=torch.uint8, device=env.device)
    rec = _lib.GcRecord(C.sizeof(_lib.GcRecord), None, None, None, flags.data_ptr(), None)
    _lib.check(env._lib.gc_collect(env._h, K, _lib.POLICY_RANDOM, None, 0.0, C.c_void_p(env._state.data_ptr()),
                                   C.c_void_p(env._t.data_ptr()), C.c_void_p(env._index.data_ptr()), C.byref(rec),
                                   C.c_void_p(env._stats.data_ptr()), env._stream()))
    first = B.CellularVectorEnv(**kw).collect(1).flags[0]
    assert torch.equal(flags[0, :n], first)
    del first
    last = B.CellularVectorEnv(**kw)
    last.rollout(128)
    assert torch.equal(flags[128, :n], last.collect(1).flags[0])
    assert torch.equal(last.state, env.state) and torch.equal(last.time_step, env.time_step)


def test_gridworld_no_position_action_is_reported(B):
    env = B.CellularVectorEnv(kind="gridworld", num_envs=1001, env_seed=1)
    env.collect(3, np.full(400, 24, np.int32))
    with pytest.raises(KeyError, match="position"):
        env.check_actions()


def test_errors(B):
    from gym_cellular_b200 import _lib
    env = B.CellularVectorEnv(num_envs=100, env_seed=1)
    policy = np.zeros(27, np.int32)

    def invalid(fn, text):
        with pytest.raises(_lib.GcError) as ei:
            fn()
        assert ei.value.code == _lib.ERR_INVALID and text in ei.value.message

    invalid(lambda: env.collect(0), "n_steps")
    for eps in (-0.1, 1.5, float("nan")):
        invalid(lambda: env.collect(4, policy, eps), "epsilon")
    invalid(lambda: env.collect(4, None, 0.1), "epsilon")
    ptab = torch.zeros(27, dtype=torch.int32, device=env.device)
    buf = torch.zeros(4 * env.ld + 4, dtype=torch.int32, device=env.device)

    def raw(kind, rec, pol=ptab):
        p = lambda t: C.c_void_p(t.data_ptr())                     # noqa: E731
        _lib.check(env._lib.gc_collect(env._h, 4, kind, p(pol), 0.0, p(env._state), p(env._t), p(env._index),
                                       C.byref(rec), None, env._stream()))
    ok = _lib.GcRecord(C.sizeof(_lib.GcRecord), buf.data_ptr())
    invalid(lambda: raw(7, ok), "policy kind")
    invalid(lambda: raw(_lib.POLICY_TABLE, _lib.GcRecord(C.sizeof(_lib.GcRecord), buf.data_ptr() + 4)), "aligned")
    invalid(lambda: raw(_lib.POLICY_TABLE, _lib.GcRecord(8, buf.data_ptr())), "struct_size")
    raw(_lib.POLICY_TABLE, ok)
    wide = B.CellularVectorEnv(num_envs=100, n_cells=2, n_states=6, env_seed=1)
    invalid(lambda: wide.collect(4), "n_states, n_actions <= 4")


# ---------------------------------------------------------------------------------------------
# the example learns

def test_collect_and_learn_example(B):
    spec = importlib.util.spec_from_file_location("collect_and_learn", os.path.join(REPO, "examples", "collect_and_learn.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.learn(envs=16384)
    assert out["collect_launches"] == 40
    assert out["greedy_return"] > out["random_return"], out
