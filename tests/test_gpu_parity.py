"""GPU parity tests: the CUDA path (through the C ABI, via ctypes) against
  (1) the golden vectors produced by executing the unmodified reference, and
  (2) the CPU oracle on seeded random rollouts,
bit-exact for states / indices / flags, rewards within 1e-6 relative (BASELINE.json north_star).
"""
import numpy as np
import pytest

from conftest import detab

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

REWARD_RTOL = 1e-6      # north_star: "rewards within 1e-6 relative"
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


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def assert_matches_oracle(env, ora, check_se=True):
    n = env.num_envs
    assert (host(env.state) == ora.state).all()
    assert (host(env.tabular_state()) == ora.index).all()
    assert (host(env.time_step) == ora.t).all()
    assert (host(env._terminated[:n]) == ora.terminated).all()
    assert (host(env._truncated[:n]) == ora.truncated).all()
    assert (host(env._unsafe[:n]) == ora.unsafe).all()
    assert (host(env._count[:n]) == ora.count).all()
    if check_se:
        assert (host(env._se_row[:, :n]) == ora.se_row).all()
    np.testing.assert_allclose(host(env._reward[:n]), ora.reward, rtol=REWARD_RTOL, atol=REWARD_ATOL)


# ---------------------------------------------------------------------------------------------
# (1) golden vectors from the reference

@pytest.mark.parametrize("tag,C", [("c3", 3), ("c2", 2)])
@pytest.mark.parametrize("difficulty", ["easy", "hard", "impossible"])
@pytest.mark.parametrize("reward", ["right_polarizing", "multiple_optima", "nonlinear"])
def test_polarisation_exhaustive_vs_reference(B, golden_pol, tag, C, difficulty, reward):
    g = golden_pol
    n_s = 3 ** C
    pairs = np.arange(n_s * n_s)
    env = B.CellularVectorEnv(num_envs=len(pairs), n_cells=C, difficulty=difficulty,
                              reward_func=getattr(B.tables, reward))
    env.set_state(detab(pairs // n_s, C, 3))
    obs, rew, term, trunc, info = env.step(dev(detab(pairs % n_s, C, 3)))
    assert (host(torch.stack(obs)).T == g[f"{tag}_next"]).all()
    assert (host(env.tabular_state()) == g[f"{tag}_next_tab"]).all()
    np.testing.assert_allclose(host(rew), g[f"{tag}_reward_{reward}"], rtol=REWARD_RTOL, atol=REWARD_ATOL)
    se = g[f"{tag}_se_{difficulty}"]
    assert (host(info["side_effects"]).T == se[:, 0, :]).all()
    assert (host(info["unsafe"]) == (se == 2).any(axis=(1, 2))).all()
    np.testing.assert_allclose(host(env.side_effects_incidence()), g[f"{tag}_incidence"], rtol=1e-6)
    assert not host(term).any() and not host(trunc).any() and (host(info["time_step"]) == 1).all()


@pytest.mark.parametrize("mode", ["rs", "dl"])
def test_polarisation_noise_exhaustive_vs_reference(B, golden_pol, mode):
    g = golden_pol
    sa, u = g[f"noise_{mode}_sa"], g[f"noise_{mode}_u"]
    n = len(sa)
    for reward, rf in (("nonlinear", B.nonlinear_right_polarizing), ("right_polarizing", B.right_polarizing)):
        env = B.CellularVectorEnv(num_envs=n, stochastic=True, deadlock=(mode == "dl"), reward_func=rf)
        env.set_state(detab(sa[:, 0], 3, 3))
        obs, rew, _, _, info = env.step(dev(detab(sa[:, 1], 3, 3)), replay_u=np.where(np.isnan(u), 0.0, u))
        assert (host(env.state).T == g[f"noise_{mode}_next"]).all()
        np.testing.assert_allclose(host(rew), g[f"noise_{mode}_reward_{reward}"], rtol=REWARD_RTOL, atol=REWARD_ATOL)
        assert (host(info["side_effects"]).T == g[f"noise_{mode}_se_easy"][:, 0, :]).all()
        assert (host(info["count"]) / 3 == g[f"noise_{mode}_incidence"]).all()


@pytest.mark.parametrize("mode", ["rs", "dl"])
@pytest.mark.parametrize("seed", [12345, 7])
def test_polarisation_trajectory_real_mt19937(B, golden_pol, mode, seed):
    """The reference's own MT19937 draws, recorded, replayed into the kernel step by step."""
    g = golden_pol
    tag = f"traj_{mode}_{seed}"
    acts, states, rewards, u = (g[f"{tag}_{k}"] for k in ("actions", "states", "rewards", "u"))
    T = min(len(acts), 400)
    env = B.CellularVectorEnv(num_envs=1, stochastic=True, deadlock=(mode == "dl"))
    got_s, got_r = [], []
    for t in range(T):
        env.step_device(dev(acts[t].reshape(3, 1)), replay_u=np.where(np.isnan(u[t]), 0.0, u[t]).reshape(1, 3))
        got_s.append(env.state.clone())
        got_r.append(env._reward[:1].clone())
    assert (host(torch.cat(got_s, 1)).T == states[:T]).all()
    np.testing.assert_allclose(host(torch.cat(got_r)), rewards[:T], rtol=REWARD_RTOL, atol=REWARD_ATOL)


def _gw_replay(u0, bits, k):
    u = np.zeros((len(u0), 6))
    u[:, 0] = u0
    u[:, 1:5] = bits * 0.5 + 0.25
    u[:, 5] = k * 0.5 + 0.25
    return u


def test_gridworld_exhaustive_vs_reference(B, golden_gw):
    g = golden_gw
    s, a = g["gw_case_state"], g["gw_case_action"]
    n = len(s)
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n)
    assert (host(env.state)[:, 0] == g["gw_reset_cell"]).all() and host(env.tabular_state())[0] == g["gw_reset_tab"]
    env.set_state(s.T.copy())
    obs, rew, term, trunc, info = env.step(dev(a.T), replay_u=_gw_replay(g["gw_case_u0"], g["gw_case_bits"], g["gw_case_k"]))
    assert (host(env.state).T == g["gw_case_next"]).all()
    assert (host(env.tabular_state()) == g["gw_case_tab"]).all()
    assert (host(rew) == g["gw_case_reward"]).all()
    assert (host(info["count"]) / 2 == g["gw_case_incidence"]).all()
    assert (host(info["side_effects"]).T == g["gw_case_se"][:, 0, :]).all() and not host(info["unsafe"]).any()
    env.check_actions()
    # both-barren states: nothing is drawn, a would-be trigger must be ignored
    s, a = g["gw_barren_state"], g["gw_barren_action"]
    env = B.CellularVectorEnv(kind="gridworld", num_envs=len(s))
    env.set_state(s.T.copy())
    _, rew, _, _, info = env.step(dev(a.T), replay_u=np.zeros((len(s), 6)))
    assert (host(env.state).T == g["gw_barren_next"]).all() and (host(env.tabular_state()) == g["gw_barren_tab"]).all()
    assert (host(rew) == g["gw_barren_reward"]).all() and (host(info["count"]) == 2).all()


def test_gridworld_no_position_action_is_reported(B):
    env = B.CellularVectorEnv(kind="gridworld", num_envs=40)
    a = np.full((2, 40), 4, np.int8)
    a[0, :39] = 1
    env.step(dev(a))
    with pytest.raises(KeyError):        # the reference raises KeyError('position'), grid_world.py:143
        env.check_actions()
    env.check_actions()                  # cleared by the poll


def test_gridworld_trajectory_real_mt19937(B, golden_gw):
    g = golden_gw
    ep_len = int(g["gwtraj_ep_len"])
    T = ep_len * 40
    acts = g["gwtraj_actions"]
    u = _gw_replay(np.nan_to_num(g["gwtraj_u0"], nan=0.0), np.maximum(g["gwtraj_bits"], 0), np.maximum(g["gwtraj_k"], 0))
    env = B.CellularVectorEnv(kind="gridworld", num_envs=1, max_episode_steps=ep_len)
    cells, tabs, rews, cnts, truncs = [], [], [], [], []
    for t in range(T):
        env.step_device(dev(acts[t].reshape(2, 1)), replay_u=u[t:t + 1])
        cells.append(env.state.clone()); tabs.append(env.tabular_state().clone())
        rews.append(env._reward[:1].clone()); cnts.append(env._count[:1].clone()); truncs.append(env._truncated[:1].clone())
    cells, tabs = host(torch.cat(cells, 1)).T, host(torch.cat(tabs))
    last = (np.arange(T) + 1) % ep_len == 0
    assert (host(torch.cat(truncs)).astype(bool) == last).all()
    assert (cells[~last] == g["gwtraj_cells"][:T][~last]).all() and (tabs[~last] == g["gwtraj_tab"][:T][~last]).all()
    assert (cells[last] == g["gw_reset_cell"]).all()
    assert (host(torch.cat(rews)) == g["gwtraj_reward"][:T]).all()
    assert (host(torch.cat(cnts)) / 2 == g["gwtraj_incidence"][:T]).all()


# ---------------------------------------------------------------------------------------------
# (2) seeded random rollouts against the oracle (Philox draws on both sides)

def _rollout(env, ora, T, rng, gridworld=False, check_every=1):
    n, C = env.num_envs, env.n_cells
    for t in range(T):
        if gridworld:
            a = np.full((2, n), 4, np.int8)
            a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        else:
            a = rng.integers(0, env.n_actions, size=(C, n)).astype(np.int8)
        env.step_device(dev(a))
        ora.step(a)
        if (t + 1) % check_every == 0 or t == T - 1:
            assert_matches_oracle(env, ora)


@pytest.mark.parametrize("n", [1, 5, 17, 1000, 65536])
def test_config2_polarisation_rollout(B, O, n):
    """BASELINE config 2: default polarisation env, 65,536 envs (plus ragged sizes), deterministic."""
    env = B.CellularVectorEnv(num_envs=n)
    ora = O.OracleEnv(n_envs=n)
    _rollout(env, ora, 30, np.random.default_rng(n))
    s = env.stats()
    assert s["env_steps"] == 30 * n == ora.stats[0] and s["unsafe_steps"] == ora.stats[1] and s["count_sum"] == ora.stats[2]
    assert abs(s["reward_sum"] * 2 ** 24 - ora.stats[4]) <= 30 * n


@pytest.mark.parametrize("deadlock", [False, True])
@pytest.mark.parametrize("episodic", [True, False])
def test_stochastic_polarisation_rollout_philox(B, O, deadlock, episodic):
    n = 20011
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, deadlock=deadlock, env_seed=99, rng_episodic=episodic,
                              max_episode_steps=7, env_id_offset=123456789012)
    ora = O.OracleEnv(n_envs=n, noise=True, deadlock=deadlock, seed=99, rng_episodic=episodic, max_episode_steps=7,
                      env_id_offset=123456789012, reward="nonlinear_rp")
    _rollout(env, ora, 25, np.random.default_rng(1))
    s = env.stats()
    assert s["episodes_truncated"] == ora.stats[3] == (25 // 7) * n


def test_config3_gridworld_rollout_autoreset(B, O):
    """BASELINE config 3 (scaled to what the oracle steps in seconds): stochastic + fused auto-reset."""
    n = 1 << 17
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=5, max_episode_steps=16, dispersal_prob=0.05)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=5, max_episode_steps=16, dispersal_prob=0.05)
    _rollout(env, ora, 40, np.random.default_rng(2), gridworld=True, check_every=5)
    s = env.stats()
    assert s["env_steps"] == ora.stats[0] and s["count_sum"] == ora.stats[2] and s["episodes_truncated"] == ora.stats[3]
    assert s["reward_sum"] * 2 ** 24 == ora.stats[4]           # integer rewards: exact
    env.check_actions()


@pytest.mark.parametrize("stochastic", [False, True])
@pytest.mark.parametrize("difficulty,reward", [("easy", "right_polarizing"), ("hard", "multiple_optima")])
def test_config4_16cells_4levels_rollout(B, O, stochastic, difficulty, reward):
    """BASELINE config 4 shape (16 cells x 4 levels, 32-bit index) at a size the oracle handles."""
    n = 30000
    env = B.CellularVectorEnv(num_envs=n, n_cells=16, n_states=4, stochastic=stochastic, difficulty=difficulty,
                              reward_func=getattr(B.tables, reward), env_seed=11)
    ora = O.OracleEnv(n_envs=n, n_cells=16, n_states=4, noise=stochastic, rng_episodic=True, difficulty=difficulty,
                      reward=reward, seed=11)
    _rollout(env, ora, 20, np.random.default_rng(3), check_every=4)
    assert host(env.tabular_state()).max() > 2 ** 31          # the index really needs 32 unsigned bits


@pytest.mark.parametrize("C,S", [(1, 2), (4, 5), (7, 3), (10, 8), (13, 4), (16, 2)])
def test_other_shapes(B, O, C, S):
    n = 4099
    env = B.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=True, env_seed=S)
    ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=True, rng_episodic=True, seed=S, reward="nonlinear_rp")
    _rollout(env, ora, 10, np.random.default_rng(C))


@pytest.mark.parametrize("C", list(range(1, 17)))
def test_every_cell_count_deterministic_and_stochastic(B, O, C):
    """Every instantiation of the pair-table kernel (1..16 cells: full groups, ragged tail groups, the
    three-block register budgets), deterministic and with Philox noise, with the fused auto-reset."""
    n = 3001
    for stochastic in (False, True):
        S = 4 if C % 2 else 3
        difficulty = "hard" if (C >= 3 and C % 3) else "easy"
        env = B.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=stochastic, env_seed=C, max_episode_steps=5,
                                  difficulty=difficulty)
        ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=stochastic, rng_episodic=True, seed=C, max_episode_steps=5,
                          difficulty=difficulty, reward="nonlinear_rp" if stochastic else "right_polarizing")
        _rollout(env, ora, 8, np.random.default_rng(100 + C), check_every=4)


@pytest.mark.parametrize("C,S,stochastic", [(3, 3, True), (2, 3, False), (16, 4, True), (16, 4, False), (1, 4, True)])
def test_generic_kernel_equals_oracle(B, O, C, S, stochastic):
    """The generic per-cell kernel (used for 5-8 levels or per-cell side-effect tables) on shapes the
    pair-table fast path normally takes: both must agree with the oracle, including side-effect rows."""
    n = 9001
    env = B.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=stochastic, env_seed=8, difficulty="hard",
                              max_episode_steps=6, force_generic_kernel=True)
    ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=stochastic, seed=8, rng_episodic=True, difficulty="hard",
                      max_episode_steps=6, reward="nonlinear_rp" if stochastic else "right_polarizing")
    _rollout(env, ora, 14, np.random.default_rng(C * S), check_every=2)
    s = env.stats()
    assert s["env_steps"] == ora.stats[0] and s["unsafe_steps"] == ora.stats[1] and s["episodes_truncated"] == ora.stats[3]
    obs, rew, *_ = env.step(np.zeros((C, n), np.int8))               # host path through the generic kernel
    ora.step(np.zeros((C, n), np.int8))
    assert (np.stack(obs) == ora.state).all()


def test_custom_reward_table_and_callable(B, O):
    n = 2048
    tab = np.random.default_rng(0).random((3, 3))
    env = B.CellularVectorEnv(num_envs=n, reward_func=tab)
    env2 = B.CellularVectorEnv(num_envs=n, reward_func=lambda s, a, ns: float(sum(tab[x, y] for x, y in zip(s, a))))
    ora = O.OracleEnv(n_envs=n, reward_table=tab)
    rng = np.random.default_rng(1)
    for _ in range(5):
        a = rng.integers(0, 3, size=(3, n)).astype(np.int8)
        env.step_device(dev(a)); env2.step_device(dev(a)); ora.step(a)
        assert_matches_oracle(env, ora)
        assert_matches_oracle(env2, ora)
    with pytest.raises(ValueError):
        B.CellularVectorEnv(num_envs=4, reward_func=lambda s, a, ns: float(s[0] * s[1]))
    with pytest.raises(ValueError, match="Difficulty must be one of"):
        B.CellularVectorEnv(num_envs=4, difficulty="nope")


def test_host_path_equals_device_path(B, O):
    """gc_step_host (numpy in / numpy out, chunked H2D-kernel-D2H pipeline) against the oracle."""
    n = 100003
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=4, max_episode_steps=9, host_chunk_envs=16384)
    ora = O.OracleEnv(n_envs=n, noise=True, rng_episodic=True, seed=4, max_episode_steps=9, reward="nonlinear_rp")
    rng = np.random.default_rng(4)
    for t in range(12):
        a = rng.integers(0, 3, size=(3, n)).astype(np.int8)
        if t % 2:
            obs, rew, term, trunc, info = env.step(a)
        else:
            obs, rew, term, trunc, info = env.step(tuple(a))
        ora.step(a)
        assert (np.stack(obs) == ora.state).all() and (info["tabular_state"] == ora.index).all()
        assert (trunc == ora.truncated.astype(bool)).all() and not term.any()
        assert (info["unsafe"] == ora.unsafe.astype(bool)).all() and (info["count"] == ora.count).all()
        np.testing.assert_allclose(rew, ora.reward, rtol=REWARD_RTOL, atol=REWARD_ATOL)
    assert_matches_oracle(env, ora, check_se=False)
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=8, host_chunk_envs=50000)
    gwo = O.OracleEnv(kind="gridworld", n_envs=n, seed=8)
    for t in range(6):
        a = np.full((2, n), 4, np.int8)
        a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        obs, rew, term, trunc, info = gw.step(a)
        gwo.step(a)
        assert (np.stack(obs) == gwo.state).all() and (info["tabular_state"] == gwo.index).all() and (rew == gwo.reward).all()


def test_cuda_graph_replay_advances_rng(B, O):
    """A graph of 8 captured steps replayed 3 times = 24 distinct steps: the global-step RNG counter
    lives on the device and is advanced by the kernels, so replays do not repeat their draws."""
    n = 50000
    rng = np.random.default_rng(3)
    acts = np.full((8, 2, n), 4, np.int8)
    for k in range(8):
        acts[k, rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=17, dispersal_prob=0.2, max_episode_steps=10)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=17, dispersal_prob=0.2, max_episode_steps=10)
    ring = []
    for k in range(8):
        a = torch.zeros(2, env.ld, dtype=torch.int8, device="cuda")
        a[:, :n] = dev(acts[k])
        ring.append(a)
    graph = env.capture_steps(ring)
    for rep in range(3):
        graph.replay()
        for k in range(8):
            ora.step(acts[k])
        assert_matches_oracle(env, ora, check_se=True)
    assert env.sync_step_counter() == 24
    env.step_device(dev(acts[0]))                       # ordinary launches continue from the same counter
    ora.step(acts[0])
    assert_matches_oracle(env, ora)
    obs, rew, term, trunc, info = env.step(acts[1])     # and so does the host path
    ora.step(acts[1])
    assert (np.stack(obs) == ora.state).all() and (rew == ora.reward).all()
    assert env.stats()["env_steps"] == 26 * n


def test_cuda_graph_replay_stochastic_polarisation(B, O):
    """The same for the pair-table kernel (global-step counter: blocks arrive at kernel start, the last
    one advances it), small and multi-wave batches."""
    for n in (300, 700001):
        rng = np.random.default_rng(n)
        acts = rng.integers(0, 3, size=(8, 3, n)).astype(np.int8)
        env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=5, rng_episodic=False, noise_prob=0.3)
        ora = O.OracleEnv(n_envs=n, noise=True, rng_episodic=False, seed=5, noise_prob=0.3, reward="nonlinear_rp")
        ring = []
        for k in range(8):
            a = torch.zeros(3, env.ld, dtype=torch.int8, device="cuda")
            a[:, :n] = dev(acts[k])
            ring.append(a)
        graph = env.capture_steps(ring)
        for rep in range(2):
            graph.replay()
            for k in range(8):
                ora.step(acts[k])
            assert_matches_oracle(env, ora, check_se=True)
        assert env.sync_step_counter() == 16


def test_bound_step_on_pinned_stream(B, O):
    """bind_step(stream=s): launches go to s whatever stream is current; two handles on two streams."""
    n = 40000
    rng = np.random.default_rng(12)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=2)
    ora = O.OracleEnv(n_envs=n, noise=True, rng_episodic=True, seed=2, reward="nonlinear_rp")
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=3, max_episode_steps=6)
    gwo = O.OracleEnv(kind="gridworld", n_envs=n, seed=3, max_episode_steps=6)
    a1 = torch.zeros(3, env.ld, dtype=torch.int8, device="cuda")
    a2 = torch.full((2, gw.ld), 4, dtype=torch.int8, device="cuda")
    c1, c2 = env.bind_step(a1, stream=s1), gw.bind_step(a2, stream=s2)
    for t in range(10):
        x1 = rng.integers(0, 3, size=(3, n)).astype(np.int8)
        x2 = np.full((2, n), 4, np.int8)
        x2[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        a1[:, :n] = dev(x1)
        a2[:, :n] = dev(x2)
        s1.wait_stream(torch.cuda.current_stream())
        s2.wait_stream(torch.cuda.current_stream())
        c1()
        c2()
        torch.cuda.current_stream().wait_stream(s1)
        torch.cuda.current_stream().wait_stream(s2)
        ora.step(x1)
        gwo.step(x2)
    assert_matches_oracle(env, ora)
    assert_matches_oracle(gw, gwo)
    with pytest.raises(ValueError):
        env.bind_step(torch.zeros(3, 8, dtype=torch.int8, device="cuda"), stream=s1)


def test_zero_noise_probability_is_the_deterministic_env(B, O):
    """noise_prob = 0 dispatches the draw-free kernels; the deadlock rule still applies."""
    n = 5000
    rng = np.random.default_rng(1)
    for C, S in ((3, 3), (9, 4)):
        env = B.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=True, deadlock=True, noise_prob=0.0, env_seed=1)
        ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=True, deadlock=True, rng_episodic=True, seed=1,
                          noise_prob=0.0, reward="nonlinear_rp")
        for t in range(12):
            a = rng.integers(0, S, size=(C, n)).astype(np.int8)
            env.step_device(dev(a))
            ora.step(a)
        assert_matches_oracle(env, ora)
        assert bool((env.state == S - 1).any())


def test_shard_invariance(B):
    """Results for env i do not depend on which shard owns it (Philox keyed by global env id)."""
    n, T = 40000, 12
    rng = np.random.default_rng(9)
    acts = rng.integers(0, 3, size=(T, 3, n)).astype(np.int8)
    full = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=21, rng_episodic=False)
    cut = 16384 + 16
    parts = [B.CellularVectorEnv(num_envs=cut, stochastic=True, env_seed=21, rng_episodic=False),
             B.CellularVectorEnv(num_envs=n - cut, stochastic=True, env_seed=21, rng_episodic=False, env_id_offset=cut)]
    for t in range(T):
        full.step_device(dev(acts[t]))
        parts[0].step_device(dev(acts[t][:, :cut]))
        parts[1].step_device(dev(acts[t][:, cut:]))
    assert (host(full.state) == np.concatenate([host(p.state) for p in parts], 1)).all()
    assert (host(full._reward[:n]) == np.concatenate([host(p._reward[:p.num_envs]) for p in parts])).all()
    sf, sp = full.stats(), [p.stats() for p in parts]
    for k in sf:
        assert sf[k] == sum(s[k] for s in sp), k      # integer / fixed-point statistics add exactly


def test_reset_and_masked_reset(B):
    env = B.CellularVectorEnv(num_envs=1003, n_cells=5, n_states=4)
    rng = np.random.default_rng(0)
    for _ in range(3):
        env.step_device(dev(rng.integers(0, 4, size=(5, 1003)).astype(np.int8)))
    before = host(env.state).copy()
    mask = rng.random(1003) < 0.3
    env.reset_envs(dev(mask))
    after, t = host(env.state), host(env.time_step)
    assert (after[:, mask] == 0).all() and (after[:, ~mask] == before[:, ~mask]).all()
    assert (t[mask] == 0).all() and (t[~mask] == 3).all() and (host(env.tabular_state())[mask] == 0).all()
    obs, info = env.reset()
    assert (host(env.state) == 0).all() and (host(env.time_step) == 0).all()
    assert (host(info["side_effects"])[0] == 1).all() and (host(info["side_effects"])[1:] == 0).all()


def test_codec_kernels(B, O, golden_pol):
    import ctypes as C
    from gym_cellular_b200 import _lib
    L = _lib.load()
    rng = np.random.default_rng(0)
    for n_cells, radix, n in ((16, 4, 100000), (3, 3, 27), (2, 20, 400), (5, 7, 4097), (1, 2, 1)):
        ld = (n + 15) // 16 * 16
        cells = np.zeros((n_cells, ld), np.int8)
        cells[:, :n] = rng.integers(0, radix, size=(n_cells, n))
        d_cells, d_idx = dev(cells), torch.zeros(ld, dtype=torch.int32, device="cuda")
        _lib.check(L.gc_encode(0, n, ld, n_cells, radix, C.c_void_p(d_cells.data_ptr()), C.c_void_p(d_idx.data_ptr()), None))
        want = O.encode(cells[:, :n].copy(), radix)
        assert (host(d_idx)[:n].view(np.uint32) == want).all()
        d_back = torch.zeros_like(d_cells)
        _lib.check(L.gc_decode(0, n, ld, n_cells, radix, C.c_void_p(d_idx.data_ptr()), C.c_void_p(d_back.data_ptr()), None))
        assert (host(d_back)[:, :n] == cells[:, :n]).all()
    g = golden_pol
    c16 = np.zeros((16, 4096), np.int8)
    c16[:] = g["codec_c16_cells"].T
    d_idx = torch.zeros(4096, dtype=torch.int32, device="cuda")
    _lib.check(L.gc_encode(0, 4096, 4096, 16, 4, C.c_void_p(dev(c16).data_ptr()), C.c_void_p(d_idx.data_ptr()), None))
    assert (host(d_idx).view(np.uint32).astype(np.uint64) == g["codec_c16_tab"]).all()


# ---------------------------------------------------------------------------------------------
# (3) full BASELINE sizes: size-independent properties

def test_config4_full_size_properties(B):
    """16 cells x 4 levels, 16M envs: index <-> state round trip, count/unsafe consistency, move rule."""
    import ctypes as C
    from gym_cellular_b200 import _lib
    n = 1 << 24
    env = B.CellularVectorEnv(num_envs=n, n_cells=16, n_states=4, emit_side_effects=False)
    g = torch.Generator(device="cuda").manual_seed(0)
    prev = env.state.clone()
    for _ in range(3):
        a = torch.randint(0, 4, (16, n), dtype=torch.int8, device="cuda", generator=g)
        env.step_device(a)
        st = env.state
        assert bool((st == prev + torch.sign(a - prev)).all())                 # one step towards the action
        assert bool((env._count[:n] == (st == 3).sum(0)).all())
        prev = st.clone()
    back = torch.zeros_like(env._state)
    _lib.check(_lib.load().gc_decode(0, n, env.ld, 16, 4, C.c_void_p(env._index.data_ptr()), C.c_void_p(back.data_ptr()), None))
    assert bool((back[:, :n] == env.state).all())
    # tabular index equals the 2-bit packing of the cells
    packed = torch.zeros(n, dtype=torch.int64, device="cuda")
    for c in range(16):
        packed |= env.state[c].to(torch.int64) << (2 * c)
    assert bool((packed == env.tabular_state()).all())
    assert env.stats()["env_steps"] == 3 * n


def test_config3_full_size_properties(B):
    """Grid world, 1M envs, auto-reset: valid codes, exactly one agent, reward in {0..3}, truncation cadence."""
    n = 1 << 20
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, max_episode_steps=8, env_seed=1)
    g = torch.Generator(device="cuda").manual_seed(1)
    for t in range(16):
        jur = torch.randint(0, 2, (n,), device="cuda", generator=g)
        pos = torch.randint(0, 4, (n,), device="cuda", generator=g).to(torch.int8)
        a = torch.full((2, n), 4, dtype=torch.int8, device="cuda")
        a[jur, torch.arange(n, device="cuda")] = pos
        env.step_device(a)
        st = env.state
        assert bool(((st >= 0) & (st < 20)).all())
        assert bool((((st[0] >> 2) < 4) ^ ((st[1] >> 2) < 4)).all())           # exactly one jurisdiction holds the agent
        assert bool(((env._reward[:n] >= 0) & (env._reward[:n] <= 3)).all())
        assert bool((env._truncated[:n] == (1 if (t + 1) % 8 == 0 else 0)).all())
        assert bool((env.tabular_state() == st[0].to(torch.int64) + 20 * st[1].to(torch.int64)).all())
    env.check_actions()
    assert env.stats()["episodes_truncated"] == 2 * n


# ---------------------------------------------------------------------------------------------
# SURVEY 8(f1), (f4): batched codec both ways, reference-typed materialisation, exact model export

def test_batched_codec_and_materialise(B, O, golden_gw):
    env = B.CellularVectorEnv(kind="gridworld", num_envs=128)
    st = golden_gw["gw_states"]
    env.set_state(st.T.copy())
    tab = env.tabularize(env.state)
    assert (host(tab) == st[:, 0].astype(int) + 20 * st[:, 1].astype(int)).all()
    assert (host(env.detabularize(tab)) == st.T).all()
    acts = golden_gw["gw_actions"]                                    # 24 actions: ragged (not a multiple of 16)
    assert (host(env.tabularize(dev(acts.T), "action")) == golden_gw["gw_action_tab"]).all()
    assert (host(env.detabularize(dev(golden_gw["gw_action_tab"]), "action")) == acts.T).all()
    obj = env.materialise(5)
    dec = golden_gw["gw_states_decoded"][5]
    J = int(dec[0])
    assert (obj[J]["agt"]["position"] == dec[1:3]).all() and (obj[0]["living_trees"].reshape(-1) == dec[3:7]).all()
    pol = B.CellularVectorEnv(num_envs=20, n_cells=16, n_states=4)
    cells = np.random.default_rng(0).integers(0, 4, (16, 20)).astype(np.int8)
    pol.set_state(cells)
    assert (host(pol.tabularize(pol.state)).astype(np.uint32) == O.encode(cells, 4)).all()
    assert pol.materialise(3) == tuple(int(x) for x in cells[:, 3])


def test_exact_model_export(B, golden_pol, golden_gw):
    from gym_cellular_b200.model import exact_model
    # deterministic 3-cell env: a permutation-like 0/1 model that reproduces the reference's table
    P, R, valid = exact_model("cellular")
    assert P.shape == (27, 27, 27) and valid.all() and ((P == 0) | (P == 1)).all() and (P.sum(2) == 1).all()
    assert (P.reshape(729, 27).argmax(1) == golden_pol["c3_next_tab"]).all()
    np.testing.assert_allclose(R.reshape(-1), golden_pol["c3_reward_right_polarizing"], rtol=1e-6)
    # stochastic env: probabilities of the reference's enumerated noise patterns
    P, R, _ = exact_model("cellular", stochastic=True)
    np.testing.assert_allclose(P.sum(2), 1.0, atol=1e-12)
    sa, u, nxt = golden_pol["noise_rs_sa"], golden_pol["noise_rs_u"], golden_pol["noise_rs_next"]
    want = np.zeros_like(P)
    for (si, ai), uu, ns in zip(sa, u, nxt):
        w = np.prod([1.0 if np.isnan(x) else (0.1 if x < 0.1 else 0.9) for x in uu])
        want[si, ai, ns[0] + 3 * ns[1] + 9 * ns[2]] += w
    np.testing.assert_allclose(P, want, atol=1e-12)
    # grid world: 9 outcomes per (state, action); compare with the reference's enumeration
    P, R, valid = exact_model("gridworld")
    assert valid.sum() == 128
    np.testing.assert_allclose(P[valid].sum(2), 1.0, atol=1e-12)
    g = golden_gw
    s_tab = g["gw_case_state"][:, 0].astype(int) + 20 * g["gw_case_state"][:, 1].astype(int)
    a_tab = g["gw_case_action"][:, 0].astype(int) + 5 * g["gw_case_action"][:, 1].astype(int)
    w = np.where(g["gw_case_u0"] < 0.01, 0.01 / 32, 0.99)            # 16 bit patterns x 2 jurisdictions
    want = np.zeros_like(P)
    np.add.at(want, (s_tab, a_tab, g["gw_case_tab"]), w)
    Rw = np.zeros_like(R)
    np.add.at(Rw, (s_tab, a_tab), w * g["gw_case_reward"])
    covered = np.zeros(P.shape[:2], bool)
    covered[s_tab, a_tab] = True
    np.testing.assert_allclose(P[covered], want[covered], atol=1e-9)
    np.testing.assert_allclose(R[covered], Rw[covered], atol=1e-6)


def test_make_vec_entry_point(B):
    from gym_cellular_b200._gym import gym
    env = gym.make_vec("gym_cellular/GridWorld-v0", num_envs=64, max_episode_steps=128)
    obs, info = env.reset()
    assert env.num_envs == 64 and len(obs) == 2 and (host(info["tabular_state"]) == 375).all()
    env.close()


# ---------------------------------------------------------------------------------------------
# SURVEY 8(f2): K-step fused rollout == K x (generate actions, step), against the oracle

def _check_rollout(env, ora, K, policy=None, reps=2):
    n = env.num_envs
    for _ in range(reps):
        ret, uns = env.rollout(K, policy)
        oret, ouns = ora.rollout(K, None if policy is None else host(policy) if hasattr(policy, "cpu") else policy)
        assert (host(env.state) == ora.state).all()
        assert (host(env.time_step) == ora.t).all()
        assert (host(env.tabular_state()) == ora.index).all()
        assert (host(uns) == ouns).all()
        np.testing.assert_allclose(host(ret), oret, rtol=1e-5, atol=1e-6)
    s = env.stats()
    assert s["env_steps"] == ora.stats[0] == reps * K * n and s["unsafe_steps"] == ora.stats[1]
    assert s["count_sum"] == ora.stats[2] and s["episodes_truncated"] == ora.stats[3]
    assert abs(s["reward_sum"] * 2 ** 24 - ora.stats[4]) <= reps * K * n


@pytest.mark.parametrize("n", [5, 10007])
def test_rollout_deterministic_polarisation(B, O, n):
    env = B.CellularVectorEnv(num_envs=n, env_seed=12, env_id_offset=4096, max_episode_steps=11)
    ora = O.OracleEnv(n_envs=n, seed=12, env_id_offset=4096, max_episode_steps=11, rng_episodic=True)
    _check_rollout(env, ora, 17)


@pytest.mark.parametrize("episodic", [True, False])
def test_rollout_stochastic_polarisation(B, O, episodic):
    n = 6007
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, deadlock=True, env_seed=5, rng_episodic=episodic, max_episode_steps=9)
    ora = O.OracleEnv(n_envs=n, noise=True, deadlock=True, seed=5, rng_episodic=episodic, max_episode_steps=9, reward="nonlinear_rp")
    _check_rollout(env, ora, 13)
    # ordinary steps continue from the state and the counters the rollout left behind
    a = np.random.default_rng(0).integers(0, 3, (3, n)).astype(np.int8)
    env.step_device(dev(a)); ora.step(a)
    assert_matches_oracle(env, ora)


def test_rollout_16_cells(B, O):
    n = 3001
    env = B.CellularVectorEnv(num_envs=n, n_cells=16, n_states=4, stochastic=True, env_seed=2, difficulty="hard")
    ora = O.OracleEnv(n_envs=n, n_cells=16, n_states=4, noise=True, seed=2, rng_episodic=True, difficulty="hard", reward="nonlinear_rp")
    _check_rollout(env, ora, 6)


def test_rollout_gridworld_random_and_policy(B, O, golden_gw):
    n = 20011
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=9, dispersal_prob=0.05, max_episode_steps=24)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=9, dispersal_prob=0.05, max_episode_steps=24)
    _check_rollout(env, ora, 30)
    env.check_actions()
    # tabular policy: the reference's initial_policy (grid_world.py:423-438) as a 400-entry table
    policy = np.zeros(400, np.int32)
    st, pol = golden_gw["gw_states"].astype(int), golden_gw["gw_initial_policy"].astype(int)
    policy[st[:, 0] + 20 * st[:, 1]] = pol[:, 0] + 5 * pol[:, 1]
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=10, max_episode_steps=16)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=10, max_episode_steps=16)
    _check_rollout(env, ora, 20, policy=policy)


def test_rollout_tabular_policy_polarisation(B, O):
    n = 4099
    policy = np.random.default_rng(4).integers(0, 27, 27).astype(np.int32)
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=3)
    ora = O.OracleEnv(n_envs=n, noise=True, seed=3, rng_episodic=True, reward="nonlinear_rp")
    _check_rollout(env, ora, 25, policy=policy)


# ---------------------------------------------------------------------------------------------
# Full BASELINE sizes against the oracle itself (all host cores), not only through properties

def _threads():
    import os
    return max(1, min(32, os.cpu_count() or 1))


def _full_size_compare(env, ora, steps, gridworld=False):
    n = env.num_envs
    g = torch.Generator(device="cuda").manual_seed(123)
    for _ in range(steps):
        if gridworld:
            a = torch.full((2, n), 4, dtype=torch.int8, device="cuda")
            jur = torch.randint(0, 2, (n,), device="cuda", generator=g)
            pos = torch.randint(0, 4, (n,), device="cuda", generator=g).to(torch.int8)
            a[0] = torch.where(jur == 0, pos, a[0]); a[1] = torch.where(jur == 1, pos, a[1])
        else:
            a = torch.randint(0, env.n_actions, (env.n_cells, n), dtype=torch.int8, device="cuda", generator=g)
        env.step_device(a)
        ora.step_parallel(a.cpu().numpy(), _threads())
    assert bool((env.state.cpu() == torch.from_numpy(ora.state)).all())
    assert (host(env.tabular_state()) == ora.index).all()
    assert (host(env.time_step) == ora.t).all()
    assert (host(env._truncated[:n]) == ora.truncated).all() and (host(env._unsafe[:n]) == ora.unsafe).all()
    assert (host(env._count[:n]) == ora.count).all()
    np.testing.assert_allclose(host(env._reward[:n]), ora.reward, rtol=REWARD_RTOL, atol=REWARD_ATOL)


def test_config3_full_size_vs_oracle(B, O):
    n = 1 << 20
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=0, max_episode_steps=128, emit_side_effects=False)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=0, max_episode_steps=128)
    _full_size_compare(env, ora, 12, gridworld=True)


def test_config4_full_size_vs_oracle(B, O):
    n = 1 << 24
    env = B.CellularVectorEnv(num_envs=n, n_cells=16, n_states=4, emit_side_effects=False)
    ora = O.OracleEnv(n_envs=n, n_cells=16, n_states=4)
    _full_size_compare(env, ora, 2)


def test_config5_mixed_shard_vs_oracle(B, O):
    """One GPU's share of BASELINE config 5 at 8 GPUs: 4M stochastic polarisation + 4M grid-world envs,
    global ids as rank 3 of 8 would own them."""
    n = 1 << 22
    off = 3 * (1 << 23)
    pol = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=0, max_episode_steps=128, env_id_offset=off, emit_side_effects=False)
    opol = O.OracleEnv(n_envs=n, noise=True, seed=0, rng_episodic=True, max_episode_steps=128, env_id_offset=off, reward="nonlinear_rp")
    _full_size_compare(pol, opol, 3)
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=0, max_episode_steps=128, env_id_offset=off + n, emit_side_effects=False)
    ogw = O.OracleEnv(kind="gridworld", n_envs=n, seed=0, max_episode_steps=128, env_id_offset=off + n)
    _full_size_compare(gw, ogw, 3, gridworld=True)


# ---------------------------------------------------------------------------------------------
# Largest sizes, resume, DLPack, argument errors

def test_config5_all_64m_envs_on_one_gpu(B, O):
    """All 2^26 envs of BASELINE config 5 on a single GPU (32M stochastic polarisation + 32M grid
    world), one step against the oracle plus global-id bookkeeping at the 2^25 boundary."""
    n = 1 << 25
    pol = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=0, max_episode_steps=128, emit_side_effects=False)
    opol = O.OracleEnv(n_envs=n, noise=True, seed=0, rng_episodic=True, max_episode_steps=128, reward="nonlinear_rp")
    _full_size_compare(pol, opol, 2)
    del pol, opol
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=0, max_episode_steps=128, env_id_offset=n, emit_side_effects=False)
    ogw = O.OracleEnv(kind="gridworld", n_envs=n, seed=0, max_episode_steps=128, env_id_offset=n)
    _full_size_compare(gw, ogw, 2, gridworld=True)


def test_state_dict_resume(B):
    n = 30000
    rng = np.random.default_rng(0)
    acts = [dev(rng.integers(0, 3, (3, n)).astype(np.int8)) for _ in range(12)]
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=6, rng_episodic=False, max_episode_steps=5)
    for a in acts[:4]:
        env.step_device(a)
    sd = env.state_dict()
    for a in acts[4:]:
        env.step_device(a)
    want_state, want_stats = env.state.clone(), env.stats()
    env2 = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=6, rng_episodic=False, max_episode_steps=5)
    env2.load_state_dict(sd)
    assert bool((env2.tabular_state() == env2.tabularize(env2.state)).all())
    for a in acts[4:]:
        env2.step_device(a)
    assert bool((env2.state == want_state).all()) and env2.stats() == want_stats
    with pytest.raises(ValueError):
        B.CellularVectorEnv(num_envs=n + 16, stochastic=True, env_seed=6).load_state_dict(sd)


def test_dlpack_exchange(B):
    """Device buffers cross framework boundaries over DLPack: actions come in as any __dlpack__ exporter,
    observations go out as capsules."""
    class Foreign:                                   # stands for a cupy / jax array
        def __init__(self, t):
            self._t = t

        def __dlpack__(self, stream=None):
            return self._t.__dlpack__()

        def __dlpack_device__(self):
            return self._t.__dlpack_device__()
    n = 1024
    env = B.CellularVectorEnv(num_envs=n)
    a = torch.randint(0, 3, (3, n), dtype=torch.int8, device="cuda")
    obs, rew, term, trunc, info = env.step(Foreign(a))
    back = torch.from_dlpack(torch.utils.dlpack.to_dlpack(env.state))
    assert back.data_ptr() == env.state.data_ptr() and bool((back == torch.sign(a)).all())
    assert term.dtype == torch.bool and trunc.dtype == torch.bool and info["tabular_state"].dtype == torch.int32


def test_argument_errors_on_gpu(B):
    import ctypes as C
    from gym_cellular_b200 import _lib
    env = B.CellularVectorEnv(num_envs=100)
    L, p = env._lib, lambda t: C.c_void_p(t.data_ptr())
    args = (p(env._actions), p(env._state), p(env._t), p(env._reward), p(env._index), p(env._terminated),
            p(env._truncated), p(env._unsafe), p(env._count), None, None, None, None)
    assert L.gc_step(env._h, 8, 16, *args) == _lib.ERR_INVALID and b"multiple of 16" in L.gc_last_error()
    assert L.gc_step(env._h, 0, 200, *args) == _lib.ERR_INVALID and b"outside" in L.gc_last_error()
    assert L.gc_step(env._h, 0, 100, None, *args[1:]) == _lib.ERR_INVALID
    assert L.gc_step(env._h, 0, 100, *args) == 0 and L.gc_step(env._h, 16, 84, *args) == 0     # ragged tail chunk
    with pytest.raises(ValueError):
        env.step(torch.zeros(5, 100, dtype=torch.int8, device="cuda"))
    with pytest.raises(ValueError, match="levels"):
        env.set_state(np.full((3, 100), 3, np.int8))
    env.set_state(np.full((3, 100), 2, np.int8))
    assert (host(env.tabular_state()) == 26).all()
    with pytest.raises(_lib.GcError):
        B.CellularVectorEnv(num_envs=16, n_cells=17)
    with pytest.raises(_lib.GcError):
        B.CellularVectorEnv(num_envs=16, n_cells=16, n_states=8)                                # 8^16 > 2^32
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=16)
    assert L.gc_rollout(gw._h, 0, 0, None, p(gw._state), p(gw._t), p(gw._index), p(gw._reward), p(gw._index), None, None) == _lib.ERR_INVALID
    with pytest.raises(_lib.GcError):
        B.CellularVectorEnv(num_envs=16, n_cells=3, n_states=6, stochastic=True).rollout(3)     # fast path only


def test_rejected_tables_leave_the_previous_ones_in_force(B, O):
    """gc_set_tables validates before it commits: after a rejected call the env steps by its old rules."""
    import ctypes as C
    from gym_cellular_b200 import _lib
    n = 1000
    env = B.CellularVectorEnv(num_envs=n, env_seed=3)
    ora = O.OracleEnv(n_envs=n, seed=3, rng_episodic=True)
    move = np.zeros((3, 3), np.int8); move[2, 2] = 3                   # level 3 does not exist
    ok = [np.zeros((3, 3), np.float32), np.zeros((3, 3, 3), np.int8), np.zeros(3, np.uint8), np.zeros(3, np.int8)]
    t = _lib.GcCellTables(move.ctypes.data, None, None, *[a.ctypes.data for a in ok], None, None)
    assert env._lib.gc_set_tables(env._h, C.byref(t)) == _lib.ERR_INVALID and b"outside" in env._lib.gc_last_error()
    _rollout(env, ora, 6, np.random.default_rng(0))


def test_second_device_leaves_current_device_alone(B, O):
    """A handle on cuda:1 runs there without changing the caller's current device."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    assert torch.cuda.current_device() == 0
    n = 5000
    env = B.CellularVectorEnv(num_envs=n, stochastic=True, env_seed=1, device="cuda:1")
    ora = O.OracleEnv(n_envs=n, noise=True, seed=1, rng_episodic=True, reward="nonlinear_rp")
    rng = np.random.default_rng(0)
    for _ in range(4):
        a = rng.integers(0, 3, (3, n)).astype(np.int8)
        env.step(torch.from_numpy(a).to("cuda:1"))
        ora.step(a)
        assert torch.cuda.current_device() == 0
    assert env.state.device.index == 1
    assert_matches_oracle(env, ora)
    obs, rew, *_ = env.step(a)                        # host path on the second device
    ora.step(a)
    assert (np.stack(obs) == ora.state).all() and torch.cuda.current_device() == 0


def test_example_plan_and_rollout(B):
    """examples/plan_and_rollout.py: value iteration on the exported model beats random play."""
    import importlib.util
    from conftest import REPO
    spec = importlib.util.spec_from_file_location("plan_and_rollout", REPO + "/examples/plan_and_rollout.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    import sys
    argv, sys.argv = sys.argv, ["x", "--env", "polarisation", "--envs", "65536", "--steps", "64"]
    try:
        res = mod.main()
    finally:
        sys.argv = argv
    assert res["planned"][0] > res["random"][0] * 1.5


def test_gridworld_episodes_after_reset_draw_fresh_noise(B, O):
    """The reference never re-seeds grid world (grid_world.py:97-104): after reset() the dispersal events
    must NOT replay the previous episode's.  The global step keeps counting across reset(), as the oracle's."""
    n = 4096
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=3, dispersal_prob=0.2)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=3, dispersal_prob=0.2)
    rng = np.random.default_rng(8)
    acts = []
    for _ in range(6):
        a = np.full((2, n), 4, np.int8)
        a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        acts.append(a)
    episodes = []
    for ep in range(2):
        env.reset()
        ora.reset()
        traj = []
        for a in acts:
            env.step_device(dev(a))
            ora.step(a)
            assert_matches_oracle(env, ora)
            traj.append(host(env.state).copy())
        episodes.append(np.stack(traj))
    assert env.sync_step_counter() == 12
    assert (episodes[0] != episodes[1]).any()          # same actions, different dispersal draws


def test_gridworld_staged_table_on_second_device(B, O):
    """The staged-table grid-world kernel (> 48 KB of dynamic shared memory: a per-device opt-in) on two
    devices of one process."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    n = 1 << 21                                            # above the staging threshold
    rng = np.random.default_rng(9)
    a = np.full((2, n), 4, np.int8)
    a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=4)
    ora.step_parallel(a, __import__("os").cpu_count() or 1)
    for d in ("cuda:0", "cuda:1"):
        env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=4, device=d)
        env.step_device(torch.from_numpy(a).to(d))
        assert (host(env.state) == ora.state).all() and (host(env._reward[:n]) == ora.reward).all()


def test_mixed_radix_codec_on_device(B, O, golden_pol):
    """gc_encode_mixed / gc_decode_mixed: the reference's codec with its per-cell space list (arbitrary min
    and length per cell), against the reference's own outputs (codec_ragged_* fixtures) and the oracle."""
    g = golden_pol
    lens, mins, cells = g["codec_ragged_lens"], g["codec_ragged_mins"], g["codec_ragged_cells"]
    spaces = [range(int(m), int(m) + int(l)) for m, l in zip(mins, lens)]
    n = len(cells)                                             # row i of the fixture encodes to i
    idx = B.encode_mixed(dev(cells.T.astype(np.int8)), spaces)
    assert (host(idx) == np.arange(n)).all()
    back = B.decode_mixed(torch.arange(n, device="cuda"), spaces)
    assert (host(back).T == cells).all()
    for i in (0, 17, n - 1):
        assert O.encode_mixed_radix(cells[i], mins, lens) == int(idx[i]) and (O.decode_mixed_radix(i, mins, lens) == host(back)[:, i]).all()
    # 16 cells x 4 levels through the mixed entry points: the full unsigned 32-bit range
    sp16 = [range(0, 4)] * 16
    c16, t16 = g["codec_c16_cells"], g["codec_c16_tab"]
    assert (host(B.encode_mixed(dev(c16.T.copy()), sp16)).astype(np.uint64) == t16).all()
    assert (host(B.decode_mixed(dev(t16.astype(np.int64)), sp16)).T == c16).all()
    # a large ragged batch against the host codec
    rng = np.random.default_rng(0)
    spaces = [range(-1, 2), range(0, 5), range(3, 5), range(-4, 3), range(0, 1), range(10, 17)]
    cells = np.stack([rng.integers(min(s), max(s) + 1, 10007) for s in spaces]).astype(np.int8)
    want = np.array([B.generalized_cellular2tabular([int(x) for x in cells[:, i]], spaces) for i in range(0, 10007, 97)])
    got = B.encode_mixed(dev(cells), spaces)
    assert (host(got)[::97] == want).all()
    assert (host(B.decode_mixed(got, spaces)) == cells).all()
    from gym_cellular_b200 import _lib
    with pytest.raises(_lib.GcError, match="32-bit"):
        B.encode_mixed(dev(np.zeros((9, 16), np.int8)), [range(0, 16)] * 9)


def test_ragged_state_space_index_in_step(B, O):
    """Per-cell level counts (gc_cell_tables.radix): the step's tabular index is the reference's mixed-radix
    index of a ragged space list, everything else is unchanged."""
    n, radix = 5003, [2, 4, 3, 4, 2]
    spaces = [range(0, r) for r in radix]
    env = B.CellularVectorEnv(num_envs=n, n_cells=5, n_states=4, cell_radix=radix, max_episode_steps=6)
    ora = O.OracleEnv(n_envs=n, n_cells=5, n_states=4, max_episode_steps=6)
    rng = np.random.default_rng(4)
    for t in range(10):
        a = np.stack([rng.integers(0, r, n) for r in radix]).astype(np.int8)      # actions keep cell c below radix[c]
        env.step_device(dev(a))
        ora.step(a)
        st = host(env.state)
        assert (st == ora.state).all() and (st < np.array(radix)[:, None]).all()
        want = host(B.encode_mixed(env.state, spaces))
        assert (host(env.tabular_state()) == want).all()
        assert int(want[7]) == O.encode_mixed_radix(st[:, 7], np.zeros(5, np.int64), np.array(radix, np.int64))
        np.testing.assert_allclose(host(env._reward[:n]), ora.reward, rtol=REWARD_RTOL, atol=REWARD_ATOL)


@pytest.mark.parametrize("kind", ["cellular3", "cellular16", "generic", "gridworld"])
def test_final_observation_int8_layout(B, O, kind):
    """emit_final_obs: for every truncated env `final_obs` is the oracle's next state BEFORE the auto-reset
    (an oracle without time limit, re-synchronised every step); elsewhere it equals the observation."""
    n = 6007
    gw = kind == "gridworld"
    C, S = {"cellular3": (3, 3), "cellular16": (16, 4), "generic": (4, 6), "gridworld": (2, 20)}[kind]
    if gw:
        env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=3, max_episode_steps=4, emit_final_obs=True, dispersal_prob=0.1)
        mk = lambda lim: O.OracleEnv(kind="gridworld", n_envs=n, seed=3, max_episode_steps=lim, dispersal_prob=0.1)
    else:
        env = B.CellularVectorEnv(num_envs=n, n_cells=C, n_states=S, stochastic=True, env_seed=3, max_episode_steps=4,
                                  emit_final_obs=True)
        mk = lambda lim: O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=True, rng_episodic=True, seed=3,
                                     max_episode_steps=lim, reward="nonlinear_rp")
    lim, free = mk(4), mk(0)
    rng = np.random.default_rng(6)
    seen = 0
    for t in range(9):
        if gw:
            a = np.full((2, n), 4, np.int8)
            a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        else:
            a = rng.integers(0, S, size=(C, n)).astype(np.int8)
        free.state[:], free.t[:], free.global_step = lim.state, lim.t, lim.global_step
        obs, rew, term, trunc, infos = env.step(dev(a))
        free.step(a)
        lim.step(a)
        assert_matches_oracle(env, lim, check_se=False)
        fin = host(torch.stack(infos["final_obs"]))
        assert (fin == free.state).all()
        tr = host(infos["_final_obs"])
        assert (tr == lim.truncated.astype(bool)).all()
        assert (fin[:, ~tr] == lim.state[:, ~tr]).all()
        assert (host(infos["final_info"]["tabular_state"]) == free.index).all()
        seen += int(tr.sum())
    assert seen == 2 * n


def test_step_many_int8_layout(B, O):
    """gc_step_many on the int8 layout: steps over a ring of 8 bound action buffers in one foreign call (plain launches and graph replay),
    grid world (global-step RNG counter, read from device memory by every launch)."""
    n = 20011
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=5, max_episode_steps=7, dispersal_prob=0.1)
    ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=5, max_episode_steps=7, dispersal_prob=0.1)
    rng = np.random.default_rng(11)
    acts = []
    for _ in range(8):
        a = np.full((2, n), 4, np.int8)
        a[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
        acts.append(a)
    ring = []
    for a in acts:
        t = torch.zeros(2, env.ld, dtype=torch.int8, device="cuda")
        t[:, :n] = dev(a)
        ring.append(t)
    slots = [env._bind(t) for t in ring]
    env.step_many(slots, 19)                               # plain launches (fewer steps than one cached graph holds)
    for i in range(19):
        ora.step(acts[i % 8])
    assert_matches_oracle(env, ora, check_se=False)
    assert env.sync_step_counter() == 19
    env.prepare_step_many(slots)
    env.step_many(slots, 77)                               # 4 replays of the cached 16-step graph + 13 plain launches
    for i in range(77):
        ora.step(acts[i % 8])
    assert_matches_oracle(env, ora, check_se=False)
    assert env.sync_step_counter() == 96 and env.stats()["env_steps"] == 96 * n


def test_log2_reward_max_relative_error(B, golden_pol):
    """`nonlinear` rewards: the in-kernel log2(1 + r) against the reference's float64 np.log2 values over ALL
    reachable reward sums of the 3- and 2-cell envs, as a pure relative error (no absolute slack): the
    contract is 1e-6, the series is built for ~4e-7."""
    g = golden_pol
    worst = 0.0
    for tag, C in (("c3", 3), ("c2", 2)):
        n_s = 3 ** C
        pairs = np.arange(n_s * n_s)
        for rf, key in ((B.tables.nonlinear, "nonlinear"),):
            env = B.CellularVectorEnv(num_envs=len(pairs), n_cells=C, reward_func=rf)
            env.set_state(detab(pairs // n_s, C, 3))
            env.step_device(dev(detab(pairs % n_s, C, 3)))
            got, want = host(env._reward[:len(pairs)]).astype(np.float64), g[f"{tag}_reward_{key}"]
            assert (got[want == 0] == 0).all()
            nz = want != 0
            worst = max(worst, float(np.abs(got[nz] / want[nz] - 1).max()))
    # the stochastic env's variant (log2 over right_polarizing) on every noise case
    sa = g["noise_rs_sa"]
    env = B.CellularVectorEnv(num_envs=len(sa), stochastic=True)
    env.set_state(detab(sa[:, 0], 3, 3))
    env.step_device(dev(detab(sa[:, 1], 3, 3)), replay_u=np.where(np.isnan(g["noise_rs_u"]), 0.0, g["noise_rs_u"]))
    got, want = host(env._reward[:len(sa)]).astype(np.float64), g["noise_rs_reward_nonlinear"]
    nz = want != 0
    worst = max(worst, float(np.abs(got[nz] / want[nz] - 1).max()))
    assert (got[~nz] == 0).all()
    # 16 cells x 4 levels: sums beyond 1 take the log1pf path
    n = 50000
    env = B.CellularVectorEnv(num_envs=n, n_cells=16, n_states=4, reward_func=B.tables.nonlinear_right_polarizing.for_shape(4, 4))
    rng = np.random.default_rng(0)
    s, a = rng.integers(0, 4, (16, n)).astype(np.int8), rng.integers(0, 4, (16, n)).astype(np.int8)
    env.set_state(dev(s))
    env.step_device(dev(a))
    tab = B.tables.right_polarizing.table(4, 4)
    want = np.log2(1.0 + tab[s, a].sum(axis=0))
    got = host(env._reward[:n]).astype(np.float64)
    worst = max(worst, float(np.abs(got / want - 1).max()))
    print(f"max relative error of log2(1 + r): {worst:.3e}")
    assert worst <= 6e-7, worst


@pytest.mark.parametrize("layout", ["int8", "packed"])
def test_host_path_at_bench_size(B, layout):
    """The host path at the size it is benchmarked (2^24 envs, 16 cells x 4 levels, 1 M-env chunks on three
    streams): bit-identical to the device path fed the same actions."""
    n = 1 << 24
    cls = B.CellularVectorEnv if layout == "int8" else B.PackedCellularVectorEnv
    kw = dict(num_envs=n, n_cells=16, n_states=4, stochastic=True, rng_episodic=False, env_seed=2, emit_side_effects=False,
              max_episode_steps=3)
    hp, dp = cls(host_chunk_envs=1 << 20, **kw), cls(**kw)
    gen = torch.Generator(device="cuda").manual_seed(3)
    for t in range(4):
        a = torch.randint(0, 4, (16, n), dtype=torch.int8, device="cuda", generator=gen)
        if layout == "packed":
            a = dp.pack(a)
        obs, rew, term, trunc, info = hp.step(a.cpu().numpy())
        dp.step_device(a)
        if layout == "packed":
            assert (torch.from_numpy(obs.view(np.int32)) == dp.packed_state.cpu()).all()
            assert (torch.from_numpy(info["flags"]) == dp._flags[:n].cpu()).all()
        else:
            assert (torch.from_numpy(np.stack(obs)) == dp.state.cpu()).all()
            assert (torch.from_numpy(info["tabular_state"].view(np.int32)) == dp._index[:n].cpu()).all()
            assert (torch.from_numpy(info["unsafe"]) == dp._unsafe[:n].cpu().bool()).all()
            assert (torch.from_numpy(trunc) == dp._truncated[:n].cpu().bool()).all()
        assert (torch.from_numpy(rew).view(torch.int32) == dp._reward[:n].cpu().view(torch.int32)).all()
    assert hp.stats() == dp.stats()


@pytest.mark.parametrize("C,S", [(1, 5), (2, 8), (3, 6), (5, 5), (10, 8), (9, 7), (13, 5), (4, 8)])
def test_pair8_kernel_vs_oracle(B, O, C, S):
    """5..8 levels, deterministic: the 3-bit pair-table kernel (gc_cell_pair8.cu) against the oracle, with the
    fused auto-reset, the final observation and ragged batch sizes; and against the generic per-cell kernel.
    A third handle also writes the side-effect rows (the WITH_SE instantiation)."""
    n = 5003
    difficulty = "hard" if C % 2 else "easy"
    reward = "multiple_optima" if S % 2 else "right_polarizing"
    kw = dict(num_envs=n, n_cells=C, n_states=S, difficulty=difficulty, reward_func=getattr(B.tables, reward),
              max_episode_steps=5, emit_side_effects=False)
    env = B.CellularVectorEnv(emit_final_obs=True, **kw)
    gen = B.CellularVectorEnv(force_generic_kernel=True, **kw)
    wse = B.CellularVectorEnv(**dict(kw, emit_side_effects=True))
    ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, difficulty=difficulty, reward=reward, max_episode_steps=5)
    free = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, difficulty=difficulty, reward=reward)
    rng = np.random.default_rng(C * 10 + S)
    for t in range(12):
        a = rng.integers(0, S, size=(C, n)).astype(np.int8)
        free.state[:], free.t[:] = ora.state, ora.t
        env.step_device(dev(a))
        gen.step_device(dev(a))
        wse.step_device(dev(a))
        ora.step(a)
        free.step(a)
        assert_matches_oracle(env, ora, check_se=False)
        assert_matches_oracle(wse, ora, check_se=True)
        assert (host(env._final[:, :n]) == free.state).all()
        # (pair sums are rounded once per pair, the generic kernel adds cell by cell: rewards agree to rounding)
        np.testing.assert_allclose(host(env._reward[:n]), host(gen._reward[:n]), rtol=REWARD_RTOL, atol=REWARD_ATOL)
        assert torch.equal(env.state, gen.state) and torch.equal(env._unsafe[:n], gen._unsafe[:n])
        assert torch.equal(env._count[:n], gen._count[:n]) and torch.equal(env._index[:n], gen._index[:n])
    s = env.stats()
    assert s["env_steps"] == 12 * n == ora.stats[0] and s["unsafe_steps"] == ora.stats[1] and s["count_sum"] == ora.stats[2]



@pytest.mark.parametrize("episodic", [True, False])
@pytest.mark.parametrize("C,S", [(1, 5), (2, 8), (3, 6), (4, 8), (5, 5), (10, 8), (9, 7), (13, 5)])
def test_pair8_kernel_with_noise_vs_oracle(B, O, C, S, episodic):
    """5..8 levels with Philox noise: the single-cell-table variant of gc_cell_pair8.cu (32-bit draws up to four
    cells, 16-bit halves with the tie rule beyond) against the oracle and against the generic per-cell kernel, with
    the fused auto-reset, the final observation, a shard offset and a ragged batch size."""
    n = 5003
    difficulty = "hard" if C % 2 else "easy"
    deadlock = bool(S % 2)
    off = 987654321096 if C > 4 else 0
    kw = dict(num_envs=n, n_cells=C, n_states=S, difficulty=difficulty, stochastic=True, deadlock=deadlock, env_seed=C + S,
              rng_episodic=episodic, max_episode_steps=5, emit_side_effects=False, noise_prob=0.2, env_id_offset=off)
    env = B.CellularVectorEnv(emit_final_obs=True, **kw)
    gen = B.CellularVectorEnv(force_generic_kernel=True, **kw)
    wse = B.CellularVectorEnv(**dict(kw, emit_side_effects=True))
    okw = dict(n_envs=n, n_cells=C, n_states=S, difficulty=difficulty, noise=True, deadlock=deadlock, seed=C + S,
               rng_episodic=episodic, reward="nonlinear_rp", noise_prob=0.2, env_id_offset=off)
    ora, free = O.OracleEnv(max_episode_steps=5, **okw), O.OracleEnv(**okw)
    rng = np.random.default_rng(C * 10 + S)
    for t in range(12):
        a = rng.integers(0, S, size=(C, n)).astype(np.int8)
        free.state[:], free.t[:], free.global_step = ora.state, ora.t, ora.global_step
        env.step_device(dev(a))
        gen.step_device(dev(a))
        wse.step_device(dev(a))
        ora.step(a)
        free.step(a)
        assert_matches_oracle(env, ora, check_se=False)
        assert_matches_oracle(wse, ora, check_se=True)
        assert (host(env._final[:, :n]) == free.state).all()
        np.testing.assert_allclose(host(env._reward[:n]), host(gen._reward[:n]), rtol=REWARD_RTOL, atol=REWARD_ATOL)
        assert torch.equal(env.state, gen.state) and torch.equal(env._unsafe[:n], gen._unsafe[:n])
        assert torch.equal(env._count[:n], gen._count[:n]) and torch.equal(env._index[:n], gen._index[:n])
    s = env.stats()
    assert s["env_steps"] == 12 * n == ora.stats[0] and s["unsafe_steps"] == ora.stats[1] and s["count_sum"] == ora.stats[2]
    assert s["episodes_truncated"] == ora.stats[3]
