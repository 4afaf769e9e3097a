"""Experience counts (gc_collect_counts / `collect_counts`): the fused K-step collection that adds per-(state, action)
visit, transition, reward and unsafe counts on the device.  Against the histogram of `collect`'s record (same handle
state, same draws), against the float64 table reference, against the exact model, across calls, shards and layouts,
and with one bin above 2^32."""
import ctypes as C

import numpy as np
import pytest
from scipy import stats as sps

import _table_reference as TR
from test_gpu_tables import BIG, G0, SEED, derive_path, f32_tables, make_tables, start

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

FIELDS = ("visits", "next", "reward_q24", "unsafe", "cell_next")


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def host(t):
    return t.cpu().numpy()


def hist(rec, nS, nA, shape=None, joint=True, transitions=True):
    """The five count tables of a record {obs, action, reward, flags, next_obs} ([K, n] numpy arrays); shape = (C, S, A)
    for the per-cell table of the cellular family."""
    s, a, nx = (rec[k].astype(np.int64).ravel() for k in ("obs", "action", "next_obs"))
    q = np.rint(np.asarray(rec["reward"], np.float32).astype(np.float64).ravel() * 2.0 ** 24).astype(np.int64)
    uns = (rec["flags"].ravel() & 1).astype(np.int64)
    sa = s * nA + a
    out = dict.fromkeys(FIELDS)
    if joint:
        out["visits"] = np.bincount(sa, minlength=nS * nA).reshape(nS, nA)
        out["reward_q24"] = np.bincount(sa, weights=q, minlength=nS * nA).astype(np.int64).reshape(nS, nA)
        out["unsafe"] = np.bincount(sa, weights=uns, minlength=nS * nA).astype(np.int64).reshape(nS, nA)
        if transitions:
            out["next"] = np.bincount(sa * nS + nx, minlength=nS * nA * nS).reshape(nS, nA, nS)
    if shape is not None:
        Cn, S, A = shape
        cell = np.zeros((Cn, S, A, S), np.int64)
        for c in range(Cn):
            sc, ac, nc = (s // S ** c) % S, (a // A ** c) % A, (nx // S ** c) % S
            cell[c] = np.bincount((sc * A + ac) * S + nc, minlength=S * A * S).reshape(S, A, S)
        out["cell_next"] = cell
    return out


def assert_counts(counts, want):
    for f in FIELDS:
        got = getattr(counts, f)
        assert (got is None) == (want[f] is None), f
        if got is not None:
            g = host(got)
            assert g.shape == want[f].shape, f
            assert (g == want[f]).all(), (f, np.argwhere(g != want[f])[:5])


def record(tr):
    return {k: host(getattr(tr, k)).view(np.uint32) if k in ("obs", "action", "next_obs") else host(getattr(tr, k))
            for k in ("obs", "action", "reward", "flags", "next_obs")}


def check_invariants(env, counts, before, K):
    """Sum visits = K n = delta env_steps; sum reward_q24 and unsafe = the statistics' deltas; next sums to visits;
    each cell_next[c] sums to K n."""
    d = host(env._stats) - before
    Kn = K * env.num_envs
    assert d[TR_STEPS] == Kn
    if counts.visits is not None:
        assert int(counts.visits.sum()) == Kn
        assert int(counts.reward_q24.sum()) == d[TR_REWARD]
        assert int(counts.unsafe.sum()) == d[TR_UNSAFE]
    if counts.next is not None:
        assert torch.equal(counts.next.sum(2), counts.visits)
    if counts.cell_next is not None:
        assert (host(counts.cell_next.sum((1, 2, 3))) == Kn).all()


TR_STEPS, TR_UNSAFE, TR_REWARD = 0, 1, 4


def _sizes(env):
    return env._joint_sizes()


def _shape(env):
    return (env.n_cells, env.n_states, env.n_actions) if env.kind == "cellular" else None


def _gw_policy(golden_gw):
    policy = np.zeros(400, np.int32)
    st, pol = golden_gw["gw_states"].astype(int), golden_gw["gw_initial_policy"].astype(int)
    policy[st[:, 0] + 20 * st[:, 1]] = pol[:, 0] + 5 * pol[:, 1]
    return policy


# ---------------------------------------------------------------------------------------------
# 1. equals collect, bit for bit

CASES = {      # name: (env kwargs, zero_counts kwargs, policies)
    "3x3x3_noise_episodic": (dict(stochastic=True, rng_episodic=True), {}, ("random", "table", "eps")),
    "8x4x2_offset": (dict(n_cells=8, n_states=4, n_actions=2, stochastic=True, rng_episodic=False, env_id_offset=BIG),
                     dict(transitions=False), ("random", "table", "eps")),
    "16x4_cells": (dict(n_cells=16, n_states=4, stochastic=True, difficulty="hard"), dict(joint=False), ("random",)),
    "debug": (dict(cell_tables="debug"), {}, ("random", "table", "eps")),
    "gridworld": (dict(kind="gridworld", dispersal_prob=0.05), {}, ("random", "table", "eps")),
}
PARAMS = [pytest.param(c, p, id=f"{c}-{p}") for c, (_, _, pols) in CASES.items() for p in pols]


def _make(B, ekw, **kw):
    ekw = dict(ekw)
    if ekw.get("cell_tables") == "debug":
        ekw["cell_tables"] = B.tables.debug_tables()
    return B.CellularVectorEnv(**ekw, **kw)


def _policy(env, pol, golden_gw):
    if pol == "random":
        return None, 0.0
    if env.kind == "gridworld":
        table = _gw_policy(golden_gw)
    else:
        rng = np.random.default_rng(env.n_cells)
        table = rng.integers(0, env.n_actions ** env.n_cells, env.n_states ** env.n_cells).astype(np.int32)
    return table, (0.3 if pol == "eps" else 0.0)


@pytest.mark.parametrize("case,pol", PARAMS)
def test_counts_equal_collect_histogram(B, golden_gw, case, pol):
    ekw, zkw, _ = CASES[case]
    n, K = 10007, 12
    A, Bc = (_make(B, ekw, num_envs=n, env_seed=21, max_episode_steps=5) for _ in range(2))
    policy, eps = _policy(A, pol, golden_gw)
    nS, nA = _sizes(A)
    counts = B_counts = Bc.zero_counts(**zkw)
    before = host(Bc._stats)
    for _ in range(2):                                      # the second call adds to the first
        tr = A.collect(K, policy, eps, next_obs=True)
        want = hist(record(tr), nS, nA, _shape(A), joint=zkw.get("joint", True), transitions=zkw.get("transitions", True))
        if _ == 1:
            want = {f: None if w is None else w + prev[f] for f, w in want.items()}
        got = Bc.collect_counts(K, policy, eps, counts)
        assert got is B_counts
        assert_counts(got, want)
        check_invariants(Bc, got, before, K * (_ + 1))
        prev = {f: None if getattr(got, f) is None else host(getattr(got, f)) for f in FIELDS}
        assert torch.equal(A.state, Bc.state) and torch.equal(A.time_step, Bc.time_step)
        assert torch.equal(A.tabular_state(torch.int32), Bc.tabular_state(torch.int32))
        assert A.stats() == Bc.stats() and A.launch_count == Bc.launch_count
        assert A.sync_step_counter() == Bc.sync_step_counter()
    assert int(host(tr.truncated).sum()) > 0                # K spans a time-limit truncation
    if case == "gridworld":
        A.check_actions()
        Bc.check_actions()


# ---------------------------------------------------------------------------------------------
# 2. against the float64 table reference

REF_ROWS = [dict(C=3, S=3, A=3, epi=True, policies=("random", "table", "eps")),
            dict(C=5, S=2, A=3, epi=False, policies=("random", "table", "eps")),
            dict(C=8, S=4, A=2, epi=False, off=BIG, policies=("random", "eps"))]
REF_PARAMS = [pytest.param(r, p, id=f"C{r['C']}-S{r['S']}A{r['A']}-{p}") for r in REF_ROWS for p in r["policies"]]


@pytest.mark.parametrize("r,pol", REF_PARAMS)
def test_counts_equal_table_reference(B, r, pol):
    tabs = make_tables(r["C"] * 13 + r["A"], r["C"], r["S"], r["A"], noise=True, fam="dyadic")
    assert derive_path(tabs) == "pair"
    n, K, off = 4099, 7, r.get("off", 0)
    env = B.CellularVectorEnv(num_envs=n, cell_tables=tabs, env_seed=SEED, env_id_offset=off, rng_episodic=r["epi"],
                              max_episode_steps=3)
    ref = TR.TableEnv(f32_tables(tabs), n, seed=SEED, env_id_offset=off, rng_episodic=r["epi"], max_episode_steps=3)
    start(env, ref, np.random.default_rng(3))
    policy, eps = None, 0.0
    if pol != "random":
        policy = np.random.default_rng(r["C"]).integers(0, r["A"] ** r["C"], r["S"] ** r["C"]).astype(np.int32)
        eps = 0.3 if pol == "eps" else 0.0
    nS, nA = r["S"] ** r["C"], r["A"] ** r["C"]
    transitions = nS * nA * nS <= 2 ** 31
    before = host(env._stats)
    rec = ref.collect(K, policy, eps)
    counts = env.collect_counts(K, policy, eps, env.zero_counts(transitions=transitions))
    want = hist(rec, nS, nA, (r["C"], r["S"], r["A"]), transitions=transitions)
    assert_counts(counts, want)
    check_invariants(env, counts, before, K)
    assert (host(env.state) == ref.state).all() and (host(env.time_step) == ref.t).all()
    assert int(host(env._stats)[TR_REWARD]) == int(ref.stats[4]) and env.sync_step_counter() == G0 + K
    assert want["unsafe"].sum() > 0 and (rec["flags"] & 2).any()     # 'unsafe' and truncations happened


# ---------------------------------------------------------------------------------------------
# 4. one bin above 2^32

@pytest.mark.parametrize("n,K", [(1 << 22, 1025), (256, (1 << 24) + 3)], ids=["wide", "one_block"])
def test_hot_bin_above_2_32(B, n, K):
    """Deterministic 3 x 3 polarisation from the all-zero state under action 0 (a fixed point): every env-step lands on
    visits[0, 0] and on cell_next[c, 0, 0, 0].  'wide' spreads the bin over every SM; 'one_block' puts all 2^32+ counts
    of each per-cell bin into ONE block's shared-memory histogram, through its flushes at 2^31."""
    env = B.CellularVectorEnv(num_envs=n, n_cells=3, n_states=3, env_seed=5, emit_side_effects=False)
    assert (host(env.tabular_state()) == 0).all()
    counts = env.collect_counts(K, np.zeros(27, np.int32))
    total = K * n
    assert total > 2 ** 32
    v, nx, cell = host(counts.visits), host(counts.next), host(counts.cell_next)
    assert v[0, 0] == total and v.sum() == total
    assert nx[0, 0, 0] == total
    assert (cell[:, 0, 0, 0] == total).all() and (cell.sum((1, 2, 3)) == total).all()


# ---------------------------------------------------------------------------------------------
# 5. accumulation, shards, packed layout

def test_two_calls_add_up_to_one(B):
    kw = dict(num_envs=10007, stochastic=True, rng_episodic=False, env_seed=13, max_episode_steps=6)
    a, b = B.CellularVectorEnv(**kw), B.CellularVectorEnv(**kw)
    policy = np.random.default_rng(4).integers(0, 27, 27).astype(np.int32)
    ca = a.collect_counts(9, policy, 0.3)
    a.collect_counts(9, policy, 0.3, ca)
    cb = b.collect_counts(18, policy, 0.3)
    for f in FIELDS:
        assert torch.equal(getattr(ca, f), getattr(cb, f)), f
    assert torch.equal(a.state, b.state) and a.stats() == b.stats()


@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_shards_sum_to_one_handle(B, golden_gw, kind):
    n, h = 20008, 10004
    kw = dict(stochastic=True, rng_episodic=False) if kind == "cellular" else dict(dispersal_prob=0.1)
    kw.update(kind=kind, env_seed=7, max_episode_steps=6)
    policy = np.random.default_rng(5).integers(0, 27, 27).astype(np.int32) if kind == "cellular" else _gw_policy(golden_gw)
    whole = B.CellularVectorEnv(num_envs=n, **kw).collect_counts(14, policy, 0.3)
    parts = [B.CellularVectorEnv(num_envs=h, env_id_offset=o, **kw).collect_counts(14, policy, 0.3) for o in (0, h)]
    for f in FIELDS:
        if getattr(whole, f) is not None:
            assert torch.equal(getattr(parts[0], f) + getattr(parts[1], f), getattr(whole, f)), f


@pytest.mark.parametrize("shape", [(3, 3), (16, 4)])
def test_packed_equals_int8(B, shape):
    Cn, S = shape
    kw = dict(num_envs=10007, n_cells=Cn, n_states=S, stochastic=True, env_seed=6, max_episode_steps=5,
              difficulty="hard" if Cn == 16 else "easy")
    a, p = B.CellularVectorEnv(**kw), B.PackedCellularVectorEnv(**kw)
    policy, eps, joint = (np.random.default_rng(3).integers(0, 27, 27).astype(np.int32), 0.3, True) if Cn == 3 else (None, 0.0, False)
    ca, cp = a.zero_counts(joint=joint), p.zero_counts(joint=joint)
    for _ in range(2):
        a.collect_counts(9, policy, eps, ca)
        p.collect_counts(9, policy, eps, cp)
    for f in FIELDS:
        assert (getattr(ca, f) is None) == (getattr(cp, f) is None)
        if getattr(ca, f) is not None:
            assert torch.equal(getattr(ca, f), getattr(cp, f)), f
    assert torch.equal(p.unpack(p._state)[:, :a.num_envs], a.state)
    assert torch.equal(p.tabular_state(torch.int32), a.tabular_state(torch.int32))
    assert torch.equal(p.time_step, a.time_step) and p.stats() == a.stats()


# ---------------------------------------------------------------------------------------------
# 6. agrees with the exact model

def test_counts_agree_with_exact_model(B):
    from gym_cellular_b200.model import exact_model
    kw = dict(stochastic=True, difficulty="hard", env_seed=17)
    P, R, _ = exact_model(**kw)
    env = B.CellularVectorEnv(num_envs=1 << 20, rng_episodic=False, max_episode_steps=50, **kw)
    counts = env.collect_counts(32)
    v, nx, rq = host(counts.visits), host(counts.next), host(counts.reward_q24)
    assert (P[nx > 0] > 0).all()
    tested = 0
    for s, a in zip(*np.nonzero(v >= 10 ** 4)):
        p = P[s, a]
        sup = p > 0
        obs = nx[s, a][sup]
        exp = p[sup] * v[s, a]
        if sup.sum() > 1:
            assert sps.chisquare(obs, exp * obs.sum() / exp.sum()).pvalue > 1e-6, (s, a)
        tested += 1
    assert tested > 20
    r32 = R.astype(np.float32)
    q = np.rint(r32.astype(np.float64) * 2.0 ** 24).astype(np.int64)
    assert (rq == v * q).all()


# ---------------------------------------------------------------------------------------------
# 7. errors: rejected before any launch, nothing changes

def test_errors(B):
    from gym_cellular_b200 import _lib
    env = B.CellularVectorEnv(num_envs=100, stochastic=True, env_seed=1)
    env.collect_counts(3)
    counts = env.zero_counts()
    ptab = torch.zeros(27, dtype=torch.int32, device=env.device)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())          # noqa: E731

    def raw(e, cs, kind=_lib.POLICY_TABLE, eps=0.0, n_steps=4):
        return e._lib.gc_collect_counts(e._h, n_steps, kind, p(ptab), eps, p(e._state), p(e._t), p(e._index),
                                        C.byref(cs), p(e._stats), e._stream())

    def cs_of(c, size=C.sizeof(_lib.GcCounts), shift=0):
        return _lib.GcCounts(size, *(None if t is None else t.data_ptr() + shift for t in c))

    def invalid(e, call, text):
        state, t, stats, launches = e.state.clone(), e.time_step.clone(), e.stats(), e.launch_count
        rc = call()
        assert rc == _lib.ERR_INVALID and text in e._lib.gc_last_error().decode(), e._lib.gc_last_error()
        assert torch.equal(e.state, state) and torch.equal(e.time_step, t)
        assert e.stats() == stats and e.launch_count == launches

    ok = cs_of(counts)
    invalid(env, lambda: raw(env, ok, n_steps=0), "n_steps")
    invalid(env, lambda: raw(env, ok, kind=7), "policy kind")
    for eps in (-0.1, 1.5, float("nan")):
        invalid(env, lambda: raw(env, ok, eps=eps), "epsilon")
    invalid(env, lambda: raw(env, ok, kind=_lib.POLICY_RANDOM, eps=0.1), "epsilon")
    invalid(env, lambda: raw(env, cs_of(counts, size=8)), "struct_size")
    invalid(env, lambda: raw(env, cs_of(counts, shift=4)), "8-byte aligned")
    invalid(env, lambda: raw(env, _lib.GcCounts(C.sizeof(_lib.GcCounts))), "NULL")
    assert raw(env, ok) == _lib.OK
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=100, env_seed=1)
    cell = torch.zeros(16, dtype=torch.int64, device=gw.device)
    invalid(gw, lambda: gw._lib.gc_collect_counts(gw._h, 4, _lib.POLICY_RANDOM, None, 0.0, p(gw._state), p(gw._t),
                                                  p(gw._index), C.byref(_lib.GcCounts(C.sizeof(_lib.GcCounts), None, None,
                                                                                      None, None, cell.data_ptr())),
                                                  p(gw._stats), gw._stream()), "cell_next")
    big = B.CellularVectorEnv(num_envs=100, n_cells=16, n_states=4, env_seed=1)
    v = torch.zeros(16, dtype=torch.int64, device=big.device)
    invalid(big, lambda: big._lib.gc_collect_counts(big._h, 4, _lib.POLICY_RANDOM, None, 0.0, p(big._state), p(big._t),
                                                    p(big._index), C.byref(_lib.GcCounts(C.sizeof(_lib.GcCounts), v.data_ptr())),
                                                    p(big._stats), big._stream()), "2^31")
    with pytest.raises(ValueError, match="joint=False"):
        big.zero_counts()
    mid = B.CellularVectorEnv(num_envs=100, n_cells=8, n_states=4, n_actions=2, env_seed=1)
    with pytest.raises(ValueError, match="joint=False"):
        mid.zero_counts()
    invalid(mid, lambda: mid._lib.gc_collect_counts(mid._h, 4, _lib.POLICY_RANDOM, None, 0.0, p(mid._state), p(mid._t),
                                                    p(mid._index), C.byref(_lib.GcCounts(C.sizeof(_lib.GcCounts), None,
                                                                                         v.data_ptr())),
                                                    p(mid._stats), mid._stream()), "'next'")
    wide = B.CellularVectorEnv(num_envs=100, n_cells=2, n_states=6, env_seed=1)
    with pytest.raises(_lib.GcError, match="n_states, n_actions <= 4"):
        wide.collect_counts(4)
    z = wide.zero_counts()
    assert z.visits.shape == (36, 36) and z.next.shape == (36, 36, 36) and z.cell_next.shape == (2, 6, 6, 6)
    zg = gw.zero_counts(transitions=False)
    assert zg.visits.shape == (400, 25) and zg.next is None and zg.cell_next is None
    with pytest.raises(ValueError, match="int64"):
        env.collect_counts(2, counts=counts._replace(visits=counts.visits.to(torch.int32)))


# ---------------------------------------------------------------------------------------------
# the example plans on the counts

def test_count_and_plan_example(B):
    import importlib.util
    import os
    from conftest import REPO
    spec = importlib.util.spec_from_file_location("count_and_plan", os.path.join(REPO, "examples", "count_and_plan.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = mod.learn(envs=16384, rounds=4)
    assert out["counted_transitions"] == 4 * 64 * 16384
    assert out["learned_return"] > out["random_return"], out


# ---------------------------------------------------------------------------------------------
# a tail warp with 125..127 envs left: every lane but the last is live, the last one partly

@pytest.mark.parametrize("n", [10109, 10110, 10111])            # n mod 128 = 125, 126, 127
@pytest.mark.parametrize("kind", ["cellular", "gridworld"])
def test_tail_warp_counts_equal_collect(B, golden_gw, kind, n):
    kw = dict(stochastic=True) if kind == "cellular" else dict(dispersal_prob=0.05)
    A, Bc = (B.CellularVectorEnv(kind=kind, num_envs=n, env_seed=23, max_episode_steps=5, **kw) for _ in range(2))
    policy = np.random.default_rng(6).integers(0, 27, 27).astype(np.int32) if kind == "cellular" else _gw_policy(golden_gw)
    tr = A.collect(7, policy, 0.3, next_obs=True)
    counts = Bc.collect_counts(7, policy, 0.3)
    nS, nA = _sizes(A)
    assert_counts(counts, hist(record(tr), nS, nA, _shape(A)))
    assert torch.equal(A.state, Bc.state) and A.stats() == Bc.stats()


# ---------------------------------------------------------------------------------------------
# count tables of another shape are refused before the launch: the kernel would add past their end

def test_counts_of_another_env_are_rejected(B):
    three = B.CellularVectorEnv(num_envs=1000, n_cells=3, env_seed=2)
    four = B.CellularVectorEnv(num_envs=1000, n_cells=4, env_seed=2)
    gw = B.CellularVectorEnv(kind="gridworld", num_envs=1000, env_seed=2)
    wrong = [(four, three.zero_counts()), (four, three.zero_counts(joint=False)),
             (four, four.zero_counts()._replace(next=three.zero_counts().next)),
             (gw, gw.zero_counts()._replace(cell_next=three.zero_counts().cell_next)),
             (three, three.zero_counts()._replace(visits=three.zero_counts().visits[:, :26])),
             (three, B.Counts(None, None, None, None, None))]
    for env, counts in wrong:
        state, launches, stats = env.state.clone(), env.launch_count, env.stats()
        with pytest.raises(ValueError):
            env.collect_counts(2, counts=counts)
        assert env.launch_count == launches and torch.equal(env.state, state) and env.stats() == stats
    four.collect_counts(2, counts=four.zero_counts())
