"""`value_iteration` on the device (libgymcellular_b200_plan.so) against the numpy restatement of its arithmetic
(tests/_plan_reference.py), bit for bit: exact models, sampled dense models and real `collect_counts` output, grouped
and not, through both row paths (compacted in shared memory, and dense from global memory); the grouping and input-kind
identities, edge cases, the kernel inventory of the planner library, no synchronisation, and the example."""
import functools
import importlib.util
import os
import subprocess

import numpy as np
import pytest

import _plan_reference as PR
from conftest import REPO
from test_gpu_every_kernel import _cuda_tool, _demangle, normalise

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

GAMMA, ITERS = 0.95, 300
GRID_RANDOM = np.array([4, 9, 14, 19, 20, 21, 22, 23], np.int32)      # a_0 + 5 a_1 of the reference sampler's actions


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@functools.lru_cache(maxsize=None)
def plan_inventory():
    """Every __global__ function of libgymcellular_b200_plan.so, normalised as in test_gpu_every_kernel."""
    from gym_cellular_b200 import build as _build
    sass = subprocess.run([_cuda_tool("cuobjdump"), "-sass", _build.PLAN_LIB_PATH], capture_output=True, text=True,
                          check=True)
    mangled = [line.split("Function :", 1)[1].strip() for line in sass.stdout.splitlines() if "Function :" in line]
    return frozenset(normalise(n) for n in _demangle(mangled))


COUNTS_KERNEL, MODEL_KERNEL = ("plan_kernel", (1,)), ("plan_kernel", (0,))


def np_counts(counts):
    return tuple(t.cpu().numpy() for t in (counts.visits, counts.next, counts.reward_q24))


def assert_bits(plan, pi, V):
    got_pi, got_V = plan.policy.cpu().numpy(), plan.value.cpu().numpy()
    assert got_pi.dtype == np.int32 and got_pi.shape == pi.shape
    assert np.array_equal(got_pi, pi), np.argwhere(got_pi != pi)[:5]
    assert np.array_equal(got_V.view(np.int64), V.view(np.int64)), np.argwhere(got_V != V)[:5]


def check_counts(B, counts, gamma=GAMMA, iters=ITERS):
    plan = B.value_iteration(counts, gamma, iters)
    pi, V, _ = PR.value_iteration(*PR.estimate(*np_counts(counts)), gamma, iters)
    assert_bits(plan, pi, V)
    return plan


def check_model(B, P, R, gamma=GAMMA, iters=ITERS):
    plan = B.value_iteration((P, R), gamma, iters)
    pi, V, _ = PR.value_iteration(P.cpu().numpy(), R.cpu().numpy(), gamma, iters)
    assert_bits(plan, pi, V)
    return plan


def dirichlet(M, nS, nA, seed):
    torch.manual_seed(seed)
    alpha = torch.rand(nS, nA, nS, dtype=torch.float64, device="cuda") + 0.2
    P = torch.distributions.Dirichlet(alpha).sample((M,))
    R = torch.randn(M, nS, nA, dtype=torch.float64, device="cuda")
    return P.contiguous(), R


# ---------------------------------------------------------------------------------------------
# explicit models

@pytest.mark.parametrize("stochastic", [False, True])
def test_exact_model_three_cells(B, stochastic):
    from gym_cellular_b200.model import exact_model
    P, R, _ = exact_model(stochastic=stochastic)
    check_model(B, torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda())


def test_exact_model_gridworld(B):
    from gym_cellular_b200.model import exact_model
    P, R, _ = exact_model(kind="gridworld")
    check_model(B, torch.from_numpy(P).cuda(), torch.from_numpy(R).cuda())


def test_dirichlet_dense_config2_batch(B):
    P, R = dirichlet(8, 27, 27, 1)
    plan = check_model(B, P, R)
    assert plan.policy.shape == (8, 27)


def test_dense_rows_from_global_memory(B):
    """Dirichlet-dense grid world: 400 x 25 x 400 nonzeros cannot fit in the cluster's shared memory (2.5 MB per CTA
    even at 16 CTAs), so every CTA reads its rows densely from global memory; the bits are the contract's."""
    P, R = dirichlet(1, 400, 25, 2)
    check_model(B, P[0], R[0], iters=60)


# ---------------------------------------------------------------------------------------------
# real collect_counts output, with unvisited rows

def _cellular_counts(B, groups, n=1 << 14, seed=3):
    env = B.CellularVectorEnv(num_envs=n, n_cells=3, n_states=3, stochastic=True, env_seed=seed, max_episode_steps=20)
    nS, nA = env._joint_sizes()
    G = groups or 1
    pol = torch.randint(0, nA, (G, nS), generator=torch.Generator().manual_seed(seed), dtype=torch.int32).cuda()
    m = (torch.arange(n, device="cuda") % G).to(torch.int32)
    counts = env.zero_counts(groups=groups)
    env.collect_counts(16, pol if groups else pol[0], 0.1, counts, **({"policy_of_env": m} if groups else {}))
    env.close()
    return counts


def _gridworld_counts(B, groups, n=1 << 14, seed=4):
    env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=seed, max_episode_steps=40)
    G = groups or 1
    rng = np.random.default_rng(seed)
    pol = torch.from_numpy(GRID_RANDOM[rng.integers(0, 8, (G, 400))]).cuda()
    m = (torch.arange(n, device="cuda") % G).to(torch.int32)
    counts = env.zero_counts(groups=groups)
    env.collect_counts(32, pol if groups else pol[0], 0.2, counts, **({"policy_of_env": m} if groups else {}))
    env.close()
    return counts


def _packed_counts(B, groups, n=1 << 14, seed=5):
    env = B.PackedCellularVectorEnv(num_envs=n, n_cells=4, n_states=3, stochastic=True, env_seed=seed,
                                    max_episode_steps=20)
    G = groups or 1
    counts = env.zero_counts(groups=groups)
    nS, nA = counts.visits.shape[-2:]
    pol = torch.randint(0, nA, (G, nS), generator=torch.Generator().manual_seed(seed), dtype=torch.int32).cuda()
    m = (torch.arange(n, device="cuda") % G).to(torch.int32)
    env.collect_counts(16, pol if groups else pol[0], 0.2, counts, **({"policy_of_env": m} if groups else {}))
    env.close()
    return counts


@pytest.mark.parametrize("source", ["cellular", "gridworld", "packed"])
@pytest.mark.parametrize("groups", [None, 8])
def test_collected_counts(B, source, groups):
    counts = {"cellular": _cellular_counts, "gridworld": _gridworld_counts, "packed": _packed_counts}[source](B, groups)
    assert bool((counts.visits == 0).any()) and bool((counts.visits > 0).any())       # unvisited and visited rows
    plan = check_counts(B, counts)
    assert plan.policy.shape == counts.visits.shape[:-1]


@pytest.mark.parametrize("P", [8, 64])
def test_groups_plan_alone(B, P):
    counts = _cellular_counts(B, P, n=1 << 16)
    whole = B.value_iteration(counts)
    for g in range(P):
        one = B.value_iteration(counts.group(g))
        assert torch.equal(one.policy, whole.policy[g])
        assert torch.equal(one.value.view(torch.int64), whole.value[g].view(torch.int64))


@pytest.mark.parametrize("source", ["cellular", "gridworld"])
def test_counts_input_equals_model_input(B, source):
    cp = _example("count_and_plan")
    counts = (_cellular_counts if source == "cellular" else _gridworld_counts)(B, 8)
    a = B.value_iteration(counts)
    P, R = cp.estimate(counts)
    b = B.value_iteration((P.contiguous(), R.contiguous()))
    assert torch.equal(a.policy, b.policy) and torch.equal(a.value.view(torch.int64), b.value.view(torch.int64))


# ---------------------------------------------------------------------------------------------
# edge cases

def test_ties_gamma_zero_and_one_iteration(B):
    g = torch.Generator(device="cuda").manual_seed(7)
    nS, nA = 40, 37                                         # more actions than lanes: two per lane for some
    P, _ = dirichlet(1, nS, nA, 8)
    P, R = P[0], torch.randint(0, 3, (nS, nA), generator=g, device="cuda").double()
    P[:, 33] = P[:, 2]                                      # action 33 duplicates action 2: an exact tie, 2 wins
    R[:, 33] = R[:, 2]
    plan = check_model(B, P, R)
    assert not bool((plan.policy == 33).any())
    z = check_model(B, P, R, gamma=0.0)
    assert torch.equal(z.policy.long(), R.argmax(1)) and torch.equal(z.value, R.max(1).values)
    one = check_model(B, P, R, iters=1)
    assert torch.equal(one.policy.long(), R.argmax(1))


def test_gamma_one_chain_counts_steps(B):
    nS, nA, iters = 50, 3, 37
    P = torch.zeros(nS, nA, nS, dtype=torch.float64, device="cuda")
    s = torch.arange(nS, device="cuda")
    P[s, :, (s + 1).clamp(max=nS - 1)] = 1.0
    R = torch.ones(nS, nA, dtype=torch.float64, device="cuda")
    plan = check_model(B, P, R, gamma=1.0, iters=iters)
    assert bool((plan.value == float(iters)).all()) and bool((plan.policy == 0).all())


def test_two_sizes_on_one_stream(B):
    a_P, a_R = dirichlet(3, 27, 27, 9)
    b = _gridworld_counts(B, None)
    pa = B.value_iteration((a_P, a_R), GAMMA, ITERS)
    pb = B.value_iteration(b, GAMMA, ITERS)
    pa2 = B.value_iteration((a_P[1:2].contiguous(), a_R[1:2].contiguous()), GAMMA, ITERS)
    pi, V, _ = PR.value_iteration(a_P.cpu().numpy(), a_R.cpu().numpy(), GAMMA, ITERS)
    assert_bits(pa, pi, V)
    assert_bits(pa2, pi[1:2], V[1:2])
    pi, V, _ = PR.value_iteration(*PR.estimate(*np_counts(b)), GAMMA, ITERS)
    assert_bits(pb, pi, V)


def test_no_synchronisation(B):
    counts = _cellular_counts(B, 8)
    P, R = dirichlet(2, 27, 27, 10)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        a = B.value_iteration(counts, GAMMA, ITERS)
        b = B.value_iteration((P, R), GAMMA, ITERS)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert a.policy.shape == (8, 27) and b.policy.shape == (2, 27)


PROFILED = r"""
import json, sys
sys.path[:0] = [{tests!r}, {repo!r}]
import numpy as np, torch
import gym_cellular_b200 as B
from test_gpu_every_kernel import launches
from test_gpu_plan import _cellular_counts, _gridworld_counts, dirichlet
calls = {"counts": _cellular_counts(B, None), "grouped counts": _gridworld_counts(B, 8),
         "model": tuple(t[0] for t in dirichlet(1, 27, 27, 1)), "model batch": dirichlet(8, 27, 27, 2)}
out = {}
for name, model in calls.items():
    torch.cuda.synchronize()
    with launches() as L:
        B.value_iteration(model, 0.95, 300)
    out[name] = [[e[0][0], list(e[0][1])] for e in L.events]
print(json.dumps(out))
"""


def test_one_kernel_per_call_and_inventory():
    """Exactly one kernel launches per call, and every instantiation of the planner library launches (torch.profiler,
    in a fresh process: the calls' kernels are then the only ones of each profiled window)."""
    import json
    import sys
    assert plan_inventory() == {COUNTS_KERNEL, MODEL_KERNEL}
    script = PROFILED.replace("{tests!r}", repr(os.path.join(REPO, "tests"))).replace("{repo!r}", repr(REPO))
    flags = ["-s"] if sys.flags.no_user_site else []
    res = subprocess.run([sys.executable, *flags, "-c", script], cwd=os.path.join(REPO, "tests"), capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    want = {"counts": COUNTS_KERNEL, "grouped counts": COUNTS_KERNEL, "model": MODEL_KERNEL, "model batch": MODEL_KERNEL}
    for name, events in got.items():
        assert [(n, tuple(v)) for n, v in events] == [want[name]], (name, events)
    assert {want[n] for n in got} == plan_inventory()


# ---------------------------------------------------------------------------------------------
# the example

def _example(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REPO, "examples", name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_device_planning_example(B):
    ex = _example("device_planning")
    out = ex.learn(agents=4, envs=1 << 13, rounds=3, steps=32)
    assert min(out["learned_return"]) > out["random_return"], out
    assert len(out["plan_ms"]) == 3 and all(t > 0 for t in out["plan_ms"])


def test_device_planning_first_round_matches_torch(B):
    ia = _example("independent_agents")
    agents, envs = 8, 1 << 14
    env = B.CellularVectorEnv(num_envs=envs, env_seed=1, max_episode_steps=50, emit_side_effects=False, **ia.ENV)
    agent = (torch.arange(envs, device=env.device) % agents).to(torch.int32)
    counts = env.zero_counts(groups=agents)
    nS, nA = counts.visits.shape[1:]
    env.collect_counts(64, ia.initial_policies(agents, nS, nA, env.device), 0.2, counts, policy_of_env=agent)
    env.close()
    dev = B.value_iteration(counts).policy.cpu().numpy()
    ref = torch.stack([ia.value_iteration(*ia.estimate(counts.group(j))) for j in range(agents)]).cpu().numpy()
    _, _, Q = PR.value_iteration(*PR.estimate(*np_counts(counts)), GAMMA, ITERS)
    clear = PR.greedy_gap(Q) > 1e-9
    assert clear.mean() > 0.5
    assert np.array_equal(dev[clear], ref[clear])
