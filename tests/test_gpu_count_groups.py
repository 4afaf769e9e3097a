"""Grouped experience counts (gc_collect_counts_grouped, `collect_counts` with `zero_counts(groups=P)` and
`policy_of_env=`): one launch of the COUNT kernels in which each env adds into the counts of its own table.

  per group  group g equals the histogram of the stacked `collect` record over the envs of table g (same start state and
             global step), for every C and noise mode, grid world and the packed layout; cellular cases also against the
             float64 table reference driven by the stack restatement
  sum        the sum over the groups equals the ungrouped stacked counts bit for bit, and the handle advances as the
             ungrouped call advances it; one group under a map of zeros equals GC_POLICY_TABLE
  geometry   256-thread blocks with a wrapping grid-stride loop, and two shards that add up to the whole batch
  bounds     wild map ids write only groups [0, P); a bin past 2^32 in one group stays exact
  errors     refused calls change nothing
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_counts import FIELDS, _gw_policy, hist, record
from test_gpu_every_kernel import EPS, K, ROLL_SA, _count_tables, assert_launched, assert_wraps, \
    launches, roll_declared
from test_gpu_tables import BIG, G0, SEED, build, dev, f32_tables, host, make_tables, start
from test_policy_stack_cpu import StackTableEnv, thread_mixed_map

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@pytest.fixture(scope="module")
def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _lib():
    from gym_cellular_b200 import _lib as lib
    return lib


def snapshot(env):
    return dict(state=host(env.state), t=host(env.time_step), index=host(env.tabular_state(torch.int32)),
                stats=host(env._stats), step=env.sync_step_counter(), launches=env.launch_count)


def assert_snap(a, b):
    for k in a:
        assert (np.asarray(a[k]) == np.asarray(b[k])).all(), k


def per_group(rec, m, P, nS, nA, shape, **kw):
    """The histogram of the record over the envs of each group: {field: [P, ...] or None}."""
    hs = [hist({k: v[:, m == g] for k, v in rec.items()}, nS, nA, shape, **kw) for g in range(P)]
    return {f: None if hs[0][f] is None else np.stack([h[f] for h in hs]) for f in FIELDS}


def assert_grouped(counts, want):
    for f in FIELDS:
        got = getattr(counts, f)
        assert (got is None) == (want[f] is None), f
        if got is not None:
            g = host(got)
            assert g.shape == want[f].shape, f
            assert (g == want[f]).all(), (f, np.argwhere(g != want[f])[:5])


def assert_sum_is_ungrouped(grouped, plain):
    for f in FIELDS:
        g, p = getattr(grouped, f), getattr(plain, f)
        assert (g is None) == (p is None), f
        if g is not None:
            assert torch.equal(g.sum(0), p), f


# ---------------------------------------------------------------------------------------------
# 1. every C and noise mode: group g = the histogram of the stacked record over the envs of table g

@pytest.mark.parametrize("noise", [False, True], ids=["det", "noise"])
@pytest.mark.parametrize("C", range(1, 17))
def test_groups_equal_histogram_every_c(B, C, noise):
    S, A = ROLL_SA[C]
    P = 3
    tabs = make_tables(9173 * C + noise, C, S, A, noise=noise)      # the every-kernel sweep's tables
    policies = np.random.default_rng(C + 7).integers(0, A ** C, (P, S ** C)).astype(np.int32)
    epi, off = (C + noise) % 2 == 0, BIG if C % 3 == 1 else 0
    nS, nA, joint, trans = _count_tables(S, A, C)
    ckw = dict(joint=joint, transitions=trans)
    runs = {}
    with launches() as L:
        for what in ("record", "grouped", "plain"):
            env, ref = build(B, tabs, "dyadic", epi=epi, off=off)
            start(env, ref, np.random.default_rng(C))
            m = thread_mixed_map(env.num_envs, P, C)
            mm = dev(m)
            if what == "record":
                out = record(env.collect(K, dev(policies), EPS, next_obs=True, policy_of_env=mm))
            else:
                out = env.collect_counts(K, dev(policies), EPS, env.zero_counts(groups=P if what == "grouped" else None,
                                                                                 **ckw), policy_of_env=mm)
            runs[what] = (out, snapshot(env), ref)
    assert_launched(L, {k for k in roll_declared(C, noise) if k[1][2] != 0})          # record and count
    rec, grouped, plain = runs["record"][0], runs["grouped"][0], runs["plain"][0]
    assert_grouped(grouped, per_group(rec, m, P, nS, nA, (C, S, A), **ckw))
    assert_sum_is_ungrouped(grouped, plain)
    assert_snap(runs["grouped"][1], runs["plain"][1])
    assert_snap(runs["grouped"][1], runs["record"][1])
    # the float64 table reference driven by the stack restatement, from the same start state
    ref = runs["grouped"][2]
    sref = StackTableEnv(f32_tables(tabs), ref.n, seed=SEED, env_id_offset=off, rng_episodic=epi, max_episode_steps=3)
    sref.set_state(ref.state, ref.t)
    sref.global_step = G0
    want = sref.collect(K, (policies, m), EPS)
    assert_grouped(grouped, per_group(want, m, P, nS, nA, (C, S, A), **ckw))
    assert (runs["grouped"][1]["state"] == sref.state).all() and (runs["grouped"][1]["t"] == sref.t).all()


# ---------------------------------------------------------------------------------------------
# 2. grid world and the packed layout

def test_groups_gridworld(B, golden_gw):
    n, P = 10007, 4
    kw = dict(kind="gridworld", num_envs=n, env_seed=9, dispersal_prob=0.05, max_episode_steps=7, env_id_offset=BIG)
    rng = np.random.default_rng(4)
    grid_random = np.array([4, 9, 14, 19, 20, 21, 22, 23], np.int32)
    policies = np.stack([_gw_policy(golden_gw)] + [grid_random[rng.integers(0, 8, 400)] for _ in range(P - 1)])
    m = thread_mixed_map(n, P, 5)
    envs = [B.CellularVectorEnv(**kw) for _ in range(3)]
    for e in envs:
        e.rollout(3)                                                # away from the reset state
    with launches() as L:
        rec = record(envs[0].collect(K, dev(policies), EPS, next_obs=True, policy_of_env=dev(m)))
        grouped = envs[1].collect_counts(K, dev(policies), EPS, envs[1].zero_counts(groups=P), policy_of_env=dev(m))
        plain = envs[2].collect_counts(K, dev(policies), EPS, policy_of_env=dev(m))
    assert_launched(L, {("grid_rollout_kernel", (2,))})
    assert_grouped(grouped, per_group(rec, m, P, 400, 25, None))
    assert_sum_is_ungrouped(grouped, plain)
    assert_snap(snapshot(envs[1]), snapshot(envs[2]))
    assert_snap(snapshot(envs[1]), snapshot(envs[0]))
    for e in envs:
        e.check_actions()


@pytest.mark.parametrize("shape", [(3, 3), (8, 4)])
def test_groups_packed_equals_int8(B, shape):
    Cn, S = shape
    kw = dict(num_envs=10007, n_cells=Cn, n_states=S, stochastic=True, env_seed=6, max_episode_steps=5)
    a, p = B.CellularVectorEnv(**kw), B.PackedCellularVectorEnv(**kw)
    P = 5
    policies = dev(np.random.default_rng(3).integers(0, S ** Cn, (P, S ** Cn)).astype(np.int32))
    m = dev(thread_mixed_map(a.num_envs, P, 1))
    joint = Cn == 3
    ca, cp = (e.zero_counts(joint=joint, groups=P) for e in (a, p))
    for _ in range(2):
        a.collect_counts(K, policies, EPS, ca, policy_of_env=m)
        p.collect_counts(K, policies, EPS, cp, policy_of_env=m)
    for f in FIELDS:
        assert (getattr(ca, f) is None) == (getattr(cp, f) is None)
        if getattr(ca, f) is not None:
            assert torch.equal(getattr(ca, f), getattr(cp, f)), f
    assert int(ca.cell_next.sum()) == 2 * K * a.num_envs * Cn
    assert torch.equal(p.unpack(p._state)[:, :a.num_envs], a.state)
    assert torch.equal(p.time_step, a.time_step) and p.stats() == a.stats()


# ---------------------------------------------------------------------------------------------
# 3. one group under a map of zeros is GC_POLICY_TABLE

@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_one_group_equals_table_policy(B, golden_gw, kind):
    kw = dict(stochastic=True, rng_episodic=False) if kind == "cellular" else dict(dispersal_prob=0.05)
    a, b = (B.CellularVectorEnv(kind=kind, num_envs=10007, env_seed=23, max_episode_steps=5, **kw) for _ in range(2))
    policy = np.random.default_rng(6).integers(0, 27, 27).astype(np.int32) if kind == "cellular" else _gw_policy(golden_gw)
    zeros = torch.zeros(a.num_envs, dtype=torch.int32, device=a.device)
    ca, cb = a.zero_counts(), b.zero_counts(groups=1)
    for _ in range(2):
        a.collect_counts(7, dev(policy), 0.3, ca)
        b.collect_counts(7, dev(policy[None]), 0.3, cb, policy_of_env=zeros)
    for f in FIELDS:
        if getattr(ca, f) is not None:
            assert torch.equal(getattr(cb, f)[0], getattr(ca, f)), f
    assert_snap(snapshot(a), snapshot(b))


# ---------------------------------------------------------------------------------------------
# 4. geometry: 256-thread blocks with a wrapping grid-stride loop; two shards

N_BIG = (1 << 19) + 5


@pytest.mark.parametrize("C,S,A,noise", [(5, 2, 4, True), (13, 2, 2, False)], ids=["C5-noise", "C13-det"])
def test_groups_256_threads(B, n_sm, C, S, A, noise):
    n, P = N_BIG, 5
    assert (n + 3) // 4 >= n_sm * 512
    tabs = make_tables(811 * C, C, S, A, noise=noise)
    policies = dev(np.random.default_rng(C).integers(0, A ** C, (P, S ** C)).astype(np.int32))
    nS, nA, joint, trans = _count_tables(S, A, C)
    ckw = dict(joint=joint, transitions=trans)
    m = thread_mixed_map(n, P, C + 1)
    key = ("cell_rollout_kernel", (C, int(noise), 2))

    def fresh():
        env, ref = build(B, tabs, "dyadic", n=n, epi=noise, off=BIG if noise else 0)
        start(env, ref, np.random.default_rng(1))
        return env

    rec_env = fresh()
    rec = record(rec_env.collect(K, policies, EPS, next_obs=True, policy_of_env=dev(m)))
    with launches() as L:
        g_env = fresh()
        grouped = g_env.collect_counts(K, policies, EPS, g_env.zero_counts(groups=P, **ckw), policy_of_env=dev(m))
        p_env = fresh()
        plain = p_env.collect_counts(K, policies, EPS, p_env.zero_counts(**ckw), policy_of_env=dev(m))
    assert_launched(L, {key})
    assert_wraps(L, [key], n, 256)
    assert_grouped(grouped, per_group(rec, m, P, nS, nA, (C, S, A), **ckw))
    assert_sum_is_ungrouped(grouped, plain)
    assert_snap(snapshot(g_env), snapshot(p_env))
    assert torch.equal(g_env.state, rec_env.state)


@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_groups_of_two_shards_add_up(B, golden_gw, kind):
    n, h, P = 20008, 10004, 3
    kw = dict(stochastic=True, rng_episodic=False) if kind == "cellular" else dict(dispersal_prob=0.1)
    kw.update(kind=kind, env_seed=7, max_episode_steps=6)
    whole = B.CellularVectorEnv(num_envs=n, **kw)
    nS, nA = whole._joint_sizes()
    policies = dev(np.random.default_rng(5).integers(0, nA, (P, nS)).astype(np.int32))
    if kind == "gridworld":
        policies[0] = dev(_gw_policy(golden_gw))
    m = dev(thread_mixed_map(n, P, 2))
    cw = whole.collect_counts(14, policies, 0.3, whole.zero_counts(groups=P), policy_of_env=m)
    parts = []
    for i, o in enumerate((0, h)):
        e = B.CellularVectorEnv(num_envs=h, env_id_offset=o, **kw)
        parts.append(e.collect_counts(14, policies, 0.3, e.zero_counts(groups=P), policy_of_env=m[i * h:(i + 1) * h].clone()))
    for f in FIELDS:
        if getattr(cw, f) is not None:
            assert torch.equal(getattr(parts[0], f) + getattr(parts[1], f), getattr(cw, f)), f


# ---------------------------------------------------------------------------------------------
# 5. bounds

def _raw_grouped(env, policies, counts_ptrs, eps=0.0, n_steps=4):
    lib = _lib()
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())          # noqa: E731
    cs = lib.GcCounts(C.sizeof(lib.GcCounts), *counts_ptrs)
    return env._lib.gc_collect_counts_grouped(env._h, n_steps, p(policies), eps, p(env._state), p(env._t), p(env._index),
                                              C.byref(cs), p(env._stats), env._stream())


def test_wild_ids_write_only_the_groups(B):
    """Through the C ABI a map may hold any int32: each id is clamped into [0, P) (negative ids, read as unsigned, to
    P - 1), so only groups [0, P) are written: a guard region after each table stays zero."""
    lib, n, P, K_ = _lib(), 4099, 3, 6
    kw = dict(num_envs=n, stochastic=True, env_seed=12, max_episode_steps=5)
    raw_env, py_env = B.CellularVectorEnv(**kw), B.CellularVectorEnv(**kw)
    stack = dev(np.random.default_rng(2).integers(0, 27, (P, 27)).astype(np.int32))
    wild = np.random.default_rng(3).choice(np.array([0, 1, 2, -1, 3, 7, -(2 ** 31), 2 ** 31 - 1], np.int32), n)
    clamped = np.minimum(wild.astype(np.int64) & 0xFFFFFFFF, P - 1).astype(np.int32)
    amap = torch.zeros(raw_env.ld, dtype=torch.int32, device=raw_env.device)
    amap[:n] = dev(wild)
    lib.check(raw_env._lib.gc_set_policy_stack(raw_env._h, C.c_void_p(amap.data_ptr()), P))
    want = py_env.collect_counts(K_, stack, 0.3, py_env.zero_counts(groups=P), policy_of_env=dev(clamped))
    guard = 4096
    bufs = [torch.zeros(t.numel() + guard, dtype=torch.int64, device=raw_env.device) for t in want]
    lib.check(_raw_grouped(raw_env, stack, [b.data_ptr() for b in bufs], eps=0.3, n_steps=K_))
    for f, b, w in zip(FIELDS, bufs, want):
        assert torch.equal(b[:w.numel()].view(w.shape), w), f
        assert not b[w.numel():].any(), f
    assert torch.equal(raw_env.state, py_env.state) and raw_env.stats() == py_env.stats()


def test_hot_bin_above_2_32_in_one_group(B):
    """3 x 3 polarisation from the all-zero state under action 0 (a fixed point): every env-step of group 1 lands on
    visits[1, 0, 0] and cell_next[1, c, 0, 0, 0]; group 0 holds no env and stays zero."""
    n, K_ = 1 << 22, 1025
    env = B.CellularVectorEnv(num_envs=n, n_cells=3, n_states=3, env_seed=5, emit_side_effects=False)
    assert (host(env.tabular_state()) == 0).all()
    ones = torch.ones(n, dtype=torch.int32, device=env.device)
    counts = env.collect_counts(K_, torch.zeros(2, 27, dtype=torch.int32, device=env.device), 0.0,
                                env.zero_counts(groups=2), policy_of_env=ones)
    total = K_ * n
    assert total > 2 ** 32
    v, nx, cell = host(counts.visits), host(counts.next), host(counts.cell_next)
    assert v[1, 0, 0] == total and v.sum() == total and not v[0].any()
    assert nx[1, 0, 0, 0] == total and not nx[0].any()
    assert (cell[1, :, 0, 0, 0] == total).all() and (cell[1].sum((1, 2, 3)) == total).all() and not cell[0].any()


# ---------------------------------------------------------------------------------------------
# 6. errors: refused before any launch, nothing changes

def test_errors(B):
    lib = _lib()
    env = B.CellularVectorEnv(num_envs=100, stochastic=True, env_seed=1)
    P = 3
    stack = torch.zeros(P, 27, dtype=torch.int32, device=env.device)
    counts = env.zero_counts(groups=P)
    ptrs = [t.data_ptr() for t in counts]

    def refused(call, code, text):
        before = snapshot(env)
        kept = [t.clone() for t in counts]
        assert call() == code and text in env._lib.gc_last_error().decode(), env._lib.gc_last_error()
        assert_snap(before, snapshot(env))
        assert all(torch.equal(a, b) for a, b in zip(kept, counts))

    refused(lambda: _raw_grouped(env, stack, ptrs), lib.ERR_STATE, "gc_set_policy_stack")       # no map
    amap = torch.zeros(env.ld, dtype=torch.int32, device=env.device)
    lib.check(env._lib.gc_set_policy_stack(env._h, C.c_void_p(amap.data_ptr()), P))
    refused(lambda: _raw_grouped(env, stack, [p + 4 for p in ptrs]), lib.ERR_INVALID, "8-byte aligned")
    refused(lambda: _raw_grouped(env, stack, [None] * 5), lib.ERR_INVALID, "NULL")
    refused(lambda: _raw_grouped(env, None, ptrs), lib.ERR_INVALID, "GC_POLICY_TABLE_STACK")
    refused(lambda: _raw_grouped(env, stack, ptrs, n_steps=0), lib.ERR_INVALID, "n_steps")
    refused(lambda: _raw_grouped(env, stack, ptrs, eps=1.5), lib.ERR_INVALID, "epsilon")
    assert _raw_grouped(env, stack, ptrs) == lib.OK
    assert int(counts.visits.sum()) == 4 * 100
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=100, env_seed=1)
    gmap = torch.zeros(gw.ld, dtype=torch.int32, device=gw.device)
    lib.check(gw._lib.gc_set_policy_stack(gw._h, C.c_void_p(gmap.data_ptr()), 2))
    cell = torch.zeros(64, dtype=torch.int64, device=gw.device)
    gstack = torch.full((2, 400), 4, dtype=torch.int32, device=gw.device)
    before = snapshot(gw)
    assert _raw_grouped(gw, gstack, [None, None, None, None, cell.data_ptr()]) == lib.ERR_INVALID
    assert b"cell_next" in gw._lib.gc_last_error()
    assert_snap(before, snapshot(gw))
    # P x a table's size past 2^31: 8 cells x 4 levels x 2 actions have nS nA = 2^24 (state, action) entries and
    # C S A S = 2^8 per-cell entries a group
    mid = B.CellularVectorEnv(num_envs=100, n_cells=8, n_states=4, n_actions=2, env_seed=1)
    mmap = torch.zeros(mid.ld, dtype=torch.int32, device=mid.device)
    v = torch.zeros(16, dtype=torch.int64, device=mid.device)
    for groups, table in ((2 ** 7 + 1, "(state, action)"), (2 ** 23 + 1, "'cell_next'")):
        lib.check(mid._lib.gc_set_policy_stack(mid._h, C.c_void_p(mmap.data_ptr()), groups))
        before = snapshot(mid)
        ptr = [v.data_ptr(), None, None, None, None] if table.startswith("(") else [None] * 4 + [v.data_ptr()]
        assert _raw_grouped(mid, torch.zeros(1, 65536, dtype=torch.int32, device=mid.device), ptr) == lib.ERR_INVALID
        assert table in mid._lib.gc_last_error().decode() and "2^31" in mid._lib.gc_last_error().decode()
        assert_snap(before, snapshot(mid))
        assert not v.any()
    # the Python layer: grouped counts without a map, or with another number of groups
    m = torch.zeros(100, dtype=torch.int32, device=env.device)
    for call, msg in ((lambda: env.collect_counts(2, stack, 0.0, counts), "need policy_of_env"),
                      (lambda: env.collect_counts(2, stack[:2], 0.0, counts, policy_of_env=m), "3 groups; the policy stack has 2"),
                      (lambda: env.collect_counts(2, stack, 0.0, env.zero_counts(groups=4), policy_of_env=m), "4 groups")):
        before = snapshot(env)
        kept = [t.clone() for t in counts]
        with pytest.raises(ValueError, match=msg):
            call()
        assert_snap(before, snapshot(env))
        assert all(torch.equal(a, b) for a, b in zip(kept, counts))


# ---------------------------------------------------------------------------------------------
# 7. the example

def test_independent_agents_example(B):
    import importlib.util
    import os
    from conftest import REPO
    spec = importlib.util.spec_from_file_location("independent_agents", os.path.join(REPO, "examples", "independent_agents.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.learn(agents=4, envs=16384, rounds=4)
    assert out["count_launches"] == 4
    assert out["counted_transitions"] == [4 * 64 * 16384 // 4] * 4
    assert min(out["learned_return"]) > out["random_return"], out
