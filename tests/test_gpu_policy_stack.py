"""Policy stacks (GC_POLICY_TABLE_STACK, `policy_of_env=`): rollout, collect and collect_counts with a table per env, in
the existing rollout-family kernels.

  identity   a stack of one table under a map of zeros equals GC_POLICY_TABLE bit for bit, every C and noise mode and
             grid world, launching the kernels the every-kernel sweep declares
  mixed      env e of a stacked batch equals the same env under table map[e] alone (GPU runs per table, same start state
             and global step) and the float64 table reference driven by the numpy restatement of the stack
             (tests/test_policy_stack_cpu.py); 64- and 256-thread blocks, the grid-stride loop wrapping; grid world
             against the C oracle
  counts     the stacked counts are the histogram of the stacked record; packed equals int8
  errors     refused calls change nothing; the kernels read only the rows [0, n_tables) whatever the map holds
"""
import ctypes as C

import numpy as np
import pytest

from test_gpu_counts import _gw_policy, assert_counts, hist, record
from test_gpu_every_kernel import EPS, GRID_ROLL_DECLARED, K, ROLL_SA, _check_end, _count_tables, \
    assert_launched, assert_wraps, launches, roll_declared, slices
from test_gpu_tables import BIG, G0, SEED, build, dev, f32_tables, host, make_tables, start
from test_policy_stack_cpu import StackTableEnv, oracle_collect, oracle_stack_actions, thread_mixed_map

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


def run_modes(env, policy, eps, counts_kw, table_of_env=None):
    """rollout, collect and collect_counts in turn on one handle, K steps each; every output and the handle's state
    after each call.  table_of_env=None: GC_POLICY_TABLE with `policy`; else the stack `policy` [P, nS]."""
    kw = {} if table_of_env is None else dict(policy_of_env=table_of_env)
    out = {}
    ret, uns = env.rollout(K, policy, **kw)
    out.update(ret=host(ret).view(np.uint32), uns=host(uns), after_rollout=snapshot(env))
    tr = env.collect(K, policy, eps, next_obs=True, **kw)
    out.update(record=record(tr), after_collect=snapshot(env))
    counts = env.collect_counts(K, policy, eps, env.zero_counts(**counts_kw), **kw)
    out.update(counts={f: None if getattr(counts, f) is None else host(getattr(counts, f)) for f in counts._fields},
               after_counts=snapshot(env))
    return out


def assert_same(a, b, path=""):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), path
        for k in a:
            assert_same(a[k], b[k], f"{path}.{k}")
    elif a is None or isinstance(a, (int, float)):
        assert a == b, (path, a, b)
    else:
        assert a.dtype == b.dtype and a.shape == b.shape and (a.view(np.uint8) == b.view(np.uint8)).all(), path


# ---------------------------------------------------------------------------------------------
# 1. identity: one table, a map of zeros

@pytest.mark.parametrize("noise", [False, True], ids=["det", "noise"])
@pytest.mark.parametrize("C", range(1, 17))
def test_stack_of_one_equals_table_policy(B, C, noise):
    S, A = ROLL_SA[C]
    tabs = make_tables(7919 * C + noise, C, S, A, noise=noise)
    policy = np.random.default_rng(C).integers(0, A ** C, S ** C).astype(np.int32)
    epi, off = (C + noise) % 2 == 1, BIG if C % 3 == 0 else 0
    _, _, joint, trans = _count_tables(S, A, C)
    outs = []
    with launches() as L:
        for stacked in (False, True):
            env, ref = build(B, tabs, "dyadic", epi=epi, off=off)
            start(env, ref, np.random.default_rng(C + 50))
            zeros = torch.zeros(env.num_envs, dtype=torch.int32, device=env.device)
            outs.append(run_modes(env, dev(policy[None]) if stacked else dev(policy), EPS,
                                  dict(joint=joint, transitions=trans), zeros if stacked else None))
    assert_launched(L, roll_declared(C, noise))
    assert_same(outs[0], outs[1])
    assert outs[1]["after_counts"]["launches"] - outs[1]["after_rollout"]["launches"] == 2     # one launch per call


def test_stack_of_one_equals_table_policy_gridworld(B, golden_gw):
    policy = _gw_policy(golden_gw)
    outs = []
    with launches() as L:
        for stacked in (False, True):
            env = B.CellularVectorEnv(kind="gridworld", num_envs=10007, env_seed=9, dispersal_prob=0.05,
                                      max_episode_steps=7, env_id_offset=BIG)
            env.rollout(3)                                          # away from the reset state
            zeros = torch.zeros(env.num_envs, dtype=torch.int32, device=env.device)
            outs.append(run_modes(env, dev(policy[None]) if stacked else dev(policy), EPS, {}, zeros if stacked else None))
            env.check_actions()
    assert_launched(L, GRID_ROLL_DECLARED)
    assert_same(outs[0], outs[1])


# ---------------------------------------------------------------------------------------------
# 2. mixed maps: each env is the env under its own table

def _stack_ref(tabs, ref, n, epi, off, s=0):
    """The stacked float64 reference of envs [s, s + n) of a batch whose table reference `ref` holds the start state."""
    r = StackTableEnv(f32_tables(tabs), n, seed=SEED, env_id_offset=off + s, rng_episodic=epi, max_episode_steps=3)
    r.set_state(ref.state[:, s:s + n], ref.t[s:s + n])
    r.global_step = G0
    return r


def _ref_rollout(r, stack):
    ret, uns = np.zeros(r.n), np.zeros(r.n, np.int64)
    for _ in range(K):
        r.collect(1, stack)
        ret += r.reward_out
        uns += r.unsafe
    return ret, uns


MIX_C = [3, 5, 8, 11, 2, 7, 13, 4]
MIX_ROWS = [dict(C=C, S=ROLL_SA[C][0], A=ROLL_SA[C][1], noise=i % 3 != 2, P=P, eps=eps, epi=epi, off=BIG if i % 2 else 0)
            for i, (C, (P, eps, epi)) in enumerate(zip(MIX_C, [(P, eps, epi) for P in (3, 5) for eps in (0.0, EPS)
                                                                for epi in (True, False)]))]


def _mix_id(r):
    return f"C{r['C']}-P{r['P']}-eps{r['eps']}-{'epi' if r['epi'] else 'glob'}-{'off' if r['off'] else 'zero'}"


@pytest.mark.parametrize("r", MIX_ROWS, ids=[_mix_id(r) for r in MIX_ROWS])
def test_mixed_map_equals_each_table_alone(B, r):
    C, S, A, P, eps, epi, off = (r[k] for k in ("C", "S", "A", "P", "eps", "epi", "off"))
    tabs = make_tables(311 * C + P, C, S, A, noise=r["noise"])
    policies = np.random.default_rng(C + P).integers(0, A ** C, (P, S ** C)).astype(np.int32)
    nS, nA, joint, trans = _count_tables(S, A, C)
    ckw = dict(joint=joint, transitions=trans)

    env, ref = build(B, tabs, "dyadic", epi=epi, off=off)
    start(env, ref, np.random.default_rng(C))
    m = thread_mixed_map(env.num_envs, P, C)
    got = run_modes(env, dev(policies), eps, ckw, dev(m))

    # the float64 reference driven by the numpy restatement of the stack
    sref = _stack_ref(tabs, ref, ref.n, epi, off)
    ret, uns = _ref_rollout(sref, (policies, m))
    assert (got["ret"].view(np.float32).astype(np.float64) == ret).all() and (got["uns"] == uns).all()
    rec = sref.collect(K, (policies, m), eps)
    for k in rec:
        want = rec[k]
        assert (got["record"][k].astype(np.float64) == want).all() if k == "reward" else (got["record"][k] == want).all(), k
    rec = sref.collect(K, (policies, m), eps)
    assert_same(got["counts"], {f: v for f, v in hist(rec, nS, nA, (C, S, A), **ckw).items()})
    _check_end(env, sref)
    assert (rec["flags"] & 2).any()

    # each table alone, from the same start state and global step
    for j in range(P):
        tj, rj = build(B, tabs, "dyadic", epi=epi, off=off)
        start(tj, rj, np.random.default_rng(C))
        one = run_modes(tj, dev(policies[j]), eps, ckw)
        sel = m == j
        assert sel.sum() > 0
        assert (one["ret"][sel] == got["ret"][sel]).all() and (one["uns"][sel] == got["uns"][sel]).all()
        for k, v in one["record"].items():
            assert (v[:, sel] == got["record"][k][:, sel]).all(), (j, k)
        for when in ("after_rollout", "after_collect", "after_counts"):
            for k in ("state", "t", "index"):
                assert (one[when][k][..., sel] == got[when][k][..., sel]).all(), (j, when, k)
            assert one[when]["step"] == got[when]["step"]


STACK_BIG = [dict(C=5, S=2, A=4, noise=True, epi=True, off=BIG, P=5, eps=EPS),
             dict(C=13, S=2, A=2, noise=False, epi=False, off=0, P=3, eps=0.0)]
N_BIG = (1 << 19) + 5


@pytest.mark.parametrize("r", STACK_BIG, ids=[f"C{r['C']}-P{r['P']}" for r in STACK_BIG])
def test_mixed_map_256_threads(B, n_sm, r):
    """256-thread blocks and a wrapping grid-stride loop: each mode from the same start state, against the reference on
    slices, against each table alone on every env, and the counts against the histogram of the stacked record."""
    C, S, A, P, eps, epi, off, n = r["C"], r["S"], r["A"], r["P"], r["eps"], r["epi"], r["off"], N_BIG
    assert (n + 3) // 4 >= n_sm * 512
    tabs = make_tables(6007 * C, C, S, A, noise=r["noise"])
    policies = np.random.default_rng(C).integers(0, A ** C, (P, S ** C)).astype(np.int32)
    nS, nA, joint, trans = _count_tables(S, A, C)
    m = thread_mixed_map(n, P, C + 1)
    keys = [("cell_rollout_kernel", (C, int(r["noise"]), mode)) for mode in (0, 1, 2)]

    def fresh():
        env, ref = build(B, tabs, "dyadic", n=n, epi=epi, off=off)
        start(env, ref, np.random.default_rng(1))
        return env, ref

    with launches() as L:
        env, ref = fresh()
        g_ret, g_uns = (host(x) for x in env.rollout(K, dev(policies), policy_of_env=dev(m)))
        rec_env, _ = fresh()
        got_rec = record(rec_env.collect(K, dev(policies), eps, next_obs=True, policy_of_env=dev(m)))
        cnt_env, _ = fresh()
        counts = cnt_env.collect_counts(K, dev(policies), eps, cnt_env.zero_counts(joint=joint, transitions=trans),
                                        policy_of_env=dev(m))
    assert_launched(L, set(keys))
    assert_wraps(L, keys, n, 256)
    stride = L.of(keys[0])[0][1][0] * 256 * 4
    for s, e in slices(n, stride):
        ret, uns = _ref_rollout(_stack_ref(tabs, ref, e - s, epi, off, s), (policies, m[s:e]))
        assert (g_ret[s:e].astype(np.float64) == ret).all() and (g_uns[s:e] == uns).all()
        want = _stack_ref(tabs, ref, e - s, epi, off, s).collect(K, (policies, m[s:e]), eps)
        for k in want:
            g = got_rec[k][:, s:e]
            assert (g.astype(np.float64) == want[k]).all() if k == "reward" else (g == want[k]).all(), (s, k)
    assert_counts(counts, hist(got_rec, nS, nA, (C, S, A), joint=joint, transitions=trans))
    assert torch.equal(cnt_env.state, rec_env.state) and cnt_env.stats() == rec_env.stats()
    for j in range(P):
        tj, _ = fresh()
        one = record(tj.collect(K, dev(policies[j]), eps, next_obs=True))
        sel = m == j
        for k, v in one.items():
            assert (v[:, sel] == got_rec[k][:, sel]).all(), (j, k)
        assert torch.equal(tj.state[:, dev(sel)], rec_env.state[:, dev(sel)])


def test_mixed_map_gridworld(B, golden_gw):
    """Grid world: against the C oracle driven by the stacked actions, and against each table alone."""
    from oracle import oracle as O
    n, P, eps = 10007, 3, EPS
    rng = np.random.default_rng(4)
    grid_random = np.array([4, 9, 14, 19, 20, 21, 22, 23], np.int32)
    policies = np.stack([_gw_policy(golden_gw)] + [grid_random[rng.integers(0, 8, 400)] for _ in range(P - 1)])
    m = thread_mixed_map(n, P, 3)
    kw = dict(kind="gridworld", num_envs=n, env_seed=9, dispersal_prob=0.05, max_episode_steps=7, env_id_offset=BIG)
    okw = dict(kind="gridworld", n_envs=n, seed=9, dispersal_prob=0.05, max_episode_steps=7, env_id_offset=BIG)
    env, ora = B.CellularVectorEnv(**kw), O.OracleEnv(**okw)
    got = run_modes(env, dev(policies), eps, {}, dev(m))
    ret = np.zeros(n)
    for _ in range(K):
        ora.step(oracle_stack_actions(ora, policies, m, 0.0))
        ret += ora.reward
    np.testing.assert_allclose(got["ret"].view(np.float32), ret, rtol=1e-6)
    assert (got["after_rollout"]["state"] == ora.state).all()
    obs, act, rew, flags = oracle_collect(ora, K, policies, m, eps)
    rec = got["record"]
    assert (rec["obs"] == obs).all() and (rec["action"] == act).all() and (rec["flags"] == flags).all()
    assert (rec["reward"] == rew).all() and (got["after_collect"]["state"] == ora.state).all()
    oc = oracle_collect(ora, K, policies, m, eps)
    want = hist(dict(obs=oc[0], action=oc[1], reward=oc[2].astype(np.float32), flags=oc[3],
                     next_obs=np.zeros_like(oc[0])), 400, 25, transitions=False)
    for f in ("visits", "reward_q24", "unsafe"):
        assert (got["counts"][f] == want[f]).all(), f
    assert (got["after_counts"]["state"] == ora.state).all() and (got["after_counts"]["t"] == ora.t).all()
    env.check_actions()
    for j in range(P):
        one = run_modes(B.CellularVectorEnv(**kw), dev(policies[j]), eps, {})
        sel = m == j
        for k, v in one["record"].items():
            assert (v[:, sel] == rec[k][:, sel]).all(), (j, k)
        assert (one["after_counts"]["state"][:, sel] == got["after_counts"]["state"][:, sel]).all()


# ---------------------------------------------------------------------------------------------
# 3. counts = histogram of the stacked record; packed = int8

@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_stacked_counts_equal_histogram_of_stacked_record(B, golden_gw, kind):
    n, P = 10007, 4
    kw = dict(stochastic=True, rng_episodic=False) if kind == "cellular" else dict(dispersal_prob=0.05)
    A_, Bc = (B.CellularVectorEnv(kind=kind, num_envs=n, env_seed=23, max_episode_steps=5, **kw) for _ in range(2))
    nS, nA = A_._joint_sizes()
    rng = np.random.default_rng(8)
    policies = rng.integers(0, nA, (P, nS)).astype(np.int32)
    if kind == "gridworld":
        policies[0] = _gw_policy(golden_gw)
    m = dev(thread_mixed_map(n, P, 9))
    for _ in range(2):
        tr = A_.collect(7, dev(policies), 0.3, next_obs=True, policy_of_env=m)
        counts = Bc.collect_counts(7, dev(policies), 0.3, policy_of_env=m)
        assert_counts(counts, hist(record(tr), nS, nA, (3, 3, 3) if kind == "cellular" else None))
        assert torch.equal(A_.state, Bc.state) and A_.stats() == Bc.stats() and A_.launch_count == Bc.launch_count


@pytest.mark.parametrize("shape", [(3, 3), (8, 4)])
def test_packed_equals_int8(B, shape):
    Cn, S = shape
    kw = dict(num_envs=10007, n_cells=Cn, n_states=S, stochastic=True, env_seed=6, max_episode_steps=5)
    a, p = B.CellularVectorEnv(**kw), B.PackedCellularVectorEnv(**kw)
    P = 5
    policies = dev(np.random.default_rng(3).integers(0, S ** Cn, (P, S ** Cn)).astype(np.int32))
    m = dev(thread_mixed_map(a.num_envs, P, 1))
    joint = Cn == 3
    ra, rp = a.rollout(K, policies, policy_of_env=m), p.rollout(K, policies, policy_of_env=m)
    assert torch.equal(ra[0], rp[0]) and torch.equal(ra[1], rp[1])
    ta, tp = a.collect(K, policies, EPS, next_obs=True, policy_of_env=m), p.collect(K, policies, EPS, next_obs=True,
                                                                                   policy_of_env=m)
    for f in ta._fields:
        assert torch.equal(getattr(ta, f), getattr(tp, f)), f
    ca, cp = (e.collect_counts(K, policies, EPS, e.zero_counts(joint=joint), policy_of_env=m) for e in (a, p))
    for f in ca._fields:
        assert (getattr(ca, f) is None) == (getattr(cp, f) is None)
        if getattr(ca, f) is not None:
            assert torch.equal(getattr(ca, f), getattr(cp, f)), f
    assert torch.equal(p.unpack(p._state)[:, :a.num_envs], a.state)
    assert torch.equal(p.tabular_state(torch.int32), a.tabular_state(torch.int32))
    assert torch.equal(p.time_step, a.time_step) and p.stats() == a.stats()


# ---------------------------------------------------------------------------------------------
# 4. errors

def _unchanged(env):
    return env.state.clone(), env.time_step.clone(), env.stats(), env.launch_count


def _assert_unchanged(env, before):
    state, t, stats, launches_ = before
    assert torch.equal(env.state, state) and torch.equal(env.time_step, t)
    assert env.stats() == stats and env.launch_count == launches_


def test_errors(B):
    lib = _lib()
    env = B.CellularVectorEnv(num_envs=100, stochastic=True, env_seed=1)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())          # noqa: E731
    stack = torch.zeros(3, 27, dtype=torch.int32, device=env.device)
    ret = torch.zeros(env.ld, dtype=torch.float32, device=env.device)
    uns = torch.zeros(env.ld, dtype=torch.int32, device=env.device)
    counts = env.zero_counts()
    rec_buf = torch.zeros(4, env.ld, dtype=torch.int32, device=env.device)
    rec = lib.GcRecord(C.sizeof(lib.GcRecord), rec_buf.data_ptr(), None, None, None, None)
    cs = lib.GcCounts(C.sizeof(lib.GcCounts), *(None if t is None else t.data_ptr() for t in counts))

    def raw(entry, kind=lib.POLICY_TABLE_STACK, policy=stack):
        h, s, t, i, st, strm = env._h, p(env._state), p(env._t), p(env._index), p(env._stats), env._stream()
        if entry == "rollout":
            return env._lib.gc_rollout(h, 4, kind, p(policy), s, t, i, p(ret), p(uns), st, strm)
        if entry == "collect":
            return env._lib.gc_collect(h, 4, kind, p(policy), 0.0, s, t, i, C.byref(rec), st, strm)
        return env._lib.gc_collect_counts(h, 4, kind, p(policy), 0.0, s, t, i, C.byref(cs), st, strm)

    def refused(call, code, text):
        before = _unchanged(env)
        assert call() == code and text in env._lib.gc_last_error().decode(), env._lib.gc_last_error()
        _assert_unchanged(env, before)

    for entry in ("rollout", "collect", "counts"):                  # kind 2 without a map
        refused(lambda: raw(entry), lib.ERR_STATE, "gc_set_policy_stack")
    amap = torch.zeros(env.ld, dtype=torch.int32, device=env.device)
    assert env._lib.gc_set_policy_stack(env._h, p(amap), 0) == lib.ERR_INVALID
    assert b"n_tables" in env._lib.gc_last_error()
    assert env._lib.gc_set_policy_stack(env._h, p(amap), -3) == lib.ERR_INVALID
    assert env._lib.gc_set_policy_stack(env._h, C.c_void_p(amap.data_ptr() + 4), 3) == lib.ERR_INVALID
    assert b"16-byte" in env._lib.gc_last_error()
    for entry in ("rollout", "collect", "counts"):                  # rejected calls did not set a map
        refused(lambda: raw(entry), lib.ERR_STATE, "gc_set_policy_stack")
    lib.check(env._lib.gc_set_policy_stack(env._h, p(amap), 3))
    for entry in ("rollout", "collect", "counts"):
        refused(lambda: raw(entry, kind=7), lib.ERR_INVALID, "policy kind")
        refused(lambda: raw(entry, policy=None), lib.ERR_INVALID, "GC_POLICY_TABLE_STACK")
        assert raw(entry) == lib.OK
    lib.check(env._lib.gc_set_policy_stack(env._h, None, 0))        # switched off again
    refused(lambda: raw("collect"), lib.ERR_STATE, "gc_set_policy_stack")

    m = torch.zeros(100, dtype=torch.int32, device=env.device)
    bad = [(dict(policy=stack[0]), r"\[n_tables, 27\]"), (dict(policy=stack[:, :26]), r"\[n_tables, 27\]"),
           (dict(policy=None), "random policy"), (dict(m=m[:99]), r"shape \(100,\)"), (dict(m=m.cpu()), "lives on cpu"),
           (dict(m=m.float()), "integer tensor"), (dict(m=m + 3), r"outside \[0, 3\)"), (dict(m=m - 1), r"outside \[0, 3\)")]
    for args, msg in bad:
        for call in ("rollout", "collect", "collect_counts"):
            before = _unchanged(env)
            with pytest.raises(ValueError, match=msg):
                fn = getattr(env, call)
                pol, mp = args.get("policy", stack), args.get("m", m)
                fn(2, pol, policy_of_env=mp) if call == "rollout" else fn(2, pol, 0.0, policy_of_env=mp)
            _assert_unchanged(env, before)

    # 5-8 levels: still refused by all three entries, with a stack too
    from test_gpu_tables import derive_path
    tabs = make_tables(99, 3, 5, 3, noise=True)
    assert derive_path(tabs) == "pair8"
    wide, _ = build(B, tabs, "dyadic")
    ws, wm = torch.zeros(2, 125, dtype=torch.int32, device=env.device), torch.ones(wide.num_envs, dtype=torch.int32,
                                                                                  device=env.device)
    for call in (lambda: wide.rollout(2, ws, policy_of_env=wm), lambda: wide.collect(2, ws, policy_of_env=wm),
                 lambda: wide.collect_counts(2, ws, policy_of_env=wm, counts=wide.zero_counts(transitions=False))):
        with pytest.raises(lib.GcError) as ei:
            call()
        assert ei.value.code == lib.ERR_INVALID and "n_states, n_actions <= 4" in ei.value.message


def test_map_checked_once_per_version(B):
    """A repeated call with the same, unchanged map adds no synchronisation; an in-place change is checked again."""
    env = B.CellularVectorEnv(num_envs=1000, stochastic=True, env_seed=2)
    stack = torch.zeros(2, 27, dtype=torch.int32, device=env.device)
    m = torch.ones(1000, dtype=torch.int32, device=env.device)
    counts = env.zero_counts()
    env.collect_counts(2, stack, 0.3, counts, policy_of_env=m)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            env.collect_counts(2, stack, 0.3, counts, policy_of_env=m)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    m[7] = 2
    with pytest.raises(ValueError, match=r"outside \[0, 2\)"):
        env.collect_counts(2, stack, 0.3, counts, policy_of_env=m)
    with pytest.raises(ValueError, match=r"outside \[0, 1\)"):        # the same map, fewer tables
        m[7] = 1
        env.collect_counts(2, stack[:1], 0.3, counts, policy_of_env=m)
    env.collect_counts(2, stack, 0.3, counts, policy_of_env=m)
    # the env does not keep the caller's map alive, and a new map tensor is checked again
    import gc
    import weakref
    gone = weakref.ref(m)
    del m
    gc.collect()
    assert gone() is None
    with pytest.raises(ValueError, match=r"outside \[0, 2\)"):
        env.collect_counts(2, stack, 0.3, counts, policy_of_env=torch.full((1000,), 5, dtype=torch.int32, device=env.device))


def test_out_of_range_ids_read_only_the_stack(B):
    """Through the C ABI a map may hold any int32: an id outside [0, n_tables) is clamped (negative ids, read as
    unsigned, to n_tables - 1), so the kernel reads only the rows of the stack."""
    lib, n, P = _lib(), 4099, 3
    kw = dict(num_envs=n, stochastic=True, env_seed=12, max_episode_steps=5)
    raw_env, py_env = B.CellularVectorEnv(**kw), B.CellularVectorEnv(**kw)
    stack = dev(np.random.default_rng(2).integers(0, 27, (P, 27)).astype(np.int32))
    wild = np.random.default_rng(3).choice(np.array([0, 1, 2, -1, 3, 7, -(2 ** 31), 2 ** 31 - 1], np.int32), n)
    clamped = np.minimum(wild.astype(np.int64) & 0xFFFFFFFF, P - 1).astype(np.int32)
    amap = torch.zeros(raw_env.ld, dtype=torch.int32, device=raw_env.device)
    amap[:n] = dev(wild)
    lib.check(raw_env._lib.gc_set_policy_stack(raw_env._h, C.c_void_p(amap.data_ptr()), P))
    ret = torch.zeros(raw_env.ld, dtype=torch.float32, device=raw_env.device)
    uns = torch.zeros(raw_env.ld, dtype=torch.int32, device=raw_env.device)
    p = lambda t: C.c_void_p(t.data_ptr())                           # noqa: E731
    lib.check(raw_env._lib.gc_rollout(raw_env._h, 9, lib.POLICY_TABLE_STACK, p(stack), p(raw_env._state), p(raw_env._t),
                                      p(raw_env._index), p(ret), p(uns), p(raw_env._stats), raw_env._stream()))
    g_ret, g_uns = py_env.rollout(9, stack, policy_of_env=dev(clamped))
    assert torch.equal(ret[:n], g_ret) and torch.equal(uns[:n], g_uns) and torch.equal(raw_env.state, py_env.state)


# ---------------------------------------------------------------------------------------------
# 5. the example

def test_posterior_sampling_example(B):
    import importlib.util
    import os
    from conftest import REPO
    spec = importlib.util.spec_from_file_location("posterior_sampling", os.path.join(REPO, "examples", "posterior_sampling.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.learn(envs=16384, models=8, rounds=4)
    assert out["count_launches"] == 4 and out["counted_transitions"] == 4 * 64 * 16384
    assert out["learned_return"] > out["random_return"], out
