"""Every `__global__` instantiation the library ships, launched and checked against a reference.

The library is mostly templates: the cell count, the noise mode, the side-effect row, the rollout mode and the block
size are template parameters, so every combination is separate machine code with its own unrolling, odd-cell tail,
SWAR folds and register allocation.  Here

  * `inventory()` lists the instantiations of the built library (`cuobjdump -sass`, names demangled by `cu++filt`) as
    (kernel, template values), e.g. ("cell_rollout_kernel", (13, 0, 2)), `true` read as 1;
  * every row declares the instantiations it is written to reach, runs under `torch.profiler` and asserts that the
    kernels it launched include them, so a dispatch rule (path, 64/256-thread blocks, fusion) that picks another
    kernel fails the row;
  * `test_every_instantiation_has_a_row` asserts that the declared sets plus `EXCLUDED` equal the inventory.

Cellular rows compare with the float64 table reference (tests/_table_reference.py), grid-world rows with the C
oracle.  Batches of hundreds of thousands of envs (256-thread blocks, grid-stride loops that wrap) are checked on
slices: envs are independent and every draw is keyed by the global env id, so a reference of m envs at env id offset
`off + start`, started from the slice's state and episode step, reproduces envs [start, start + m)."""
import contextlib
import functools
import json
import os
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import _collect_oracle as CO
import _table_reference as TR
from test_gpu_counts import assert_counts, hist, record
from test_gpu_tables import BIG, G0, SEED, build, check_reward, check_stats, check_step, derive_path, dev, f32_tables, \
    gpu_out, host, make_tables, start

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N = 4099                     # small batches: 64-thread blocks for the many-step and rollout kernels
K = 5                        # rollout / collect steps (the time limit is 3: every env truncates)
EPS = 0.3


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@pytest.fixture(scope="module")
def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------
# kernel names

_CALL = re.compile(r"(\w+)(?:<([^<>]*)>)?\(")


def _cuda_tool(name):
    from gym_cellular_b200 import build as _build
    path = os.path.join(os.path.dirname(_build._nvcc()), name)
    return path if os.path.exists(path) else shutil.which(name)


def _demangle(names):
    out = subprocess.run([_cuda_tool("cu++filt")], input="\n".join(names), capture_output=True, text=True, check=True)
    return out.stdout.splitlines()


def _value(v):
    v = re.sub(r"^\((?:unsigned |signed )?\w+\)", "", v.strip())
    if v in ("true", "false"):
        return int(v == "true")
    try:
        return int(v.rstrip("uUlL"), 0)
    except ValueError:
        return v


def normalise(name):
    """A demangled kernel name as (kernel, template values); (name, ()) for a name this does not parse."""
    m = _CALL.search(name)
    if m is None:
        return name, ()
    args = m.group(2)
    return m.group(1), tuple(_value(a) for a in args.split(",")) if args else ()


@functools.lru_cache(maxsize=None)
def inventory():
    """Every __global__ function of libgymcellular_b200.so, normalised."""
    from gym_cellular_b200 import build as _build
    sass = subprocess.run([_cuda_tool("cuobjdump"), "-sass", _build.LIB_PATH], capture_output=True, text=True, check=True)
    mangled = [line.split("Function :", 1)[1].strip() for line in sass.stdout.splitlines() if "Function :" in line]
    return frozenset(normalise(n) for n in _demangle(mangled))


class Launches:
    """The kernels launched inside `launches()`: `events` = [(normalised name, grid, block)]."""
    events = ()

    def names(self):
        return {e[0] for e in self.events}

    def of(self, key):
        return [e for e in self.events if e[0] == key]


@contextlib.contextmanager
def launches():
    from torch.profiler import ProfilerActivity, profile
    out = Launches()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        yield out
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            trace = json.load(f)
    events = trace["traceEvents"] if isinstance(trace, dict) else trace
    kern = [e for e in events if e.get("cat") == "kernel"]
    names = [e["name"] for e in kern]
    mangled = [n for n in names if n.startswith("_Z")]
    plain = dict(zip(mangled, _demangle(mangled))) if mangled else {}
    out.events = [(normalise(plain.get(e["name"], e["name"])), tuple(e.get("args", {}).get("grid", ())),
                   tuple(e.get("args", {}).get("block", ()))) for e in kern]


def assert_launched(L, want):
    missing = set(want) - L.names()
    assert not missing, dict(missing=sorted(missing), launched=sorted(L.names(), key=str))


def assert_wraps(L, keys, n, threads):
    """Every launch of `keys` ran `threads`-thread blocks and a grid whose stride (4 envs a thread) is below n, so
    the grid-stride loop took a second pass."""
    ev = [e for k in keys for e in L.of(k)]
    assert ev
    for _, grid, block in ev:
        assert block[0] == threads and grid[0] * block[0] * 4 < n, (grid, block, n)


# ---------------------------------------------------------------------------------------------
# helpers

def sl(got, s, e):
    return {k: v[..., s:e] for k, v in got.items()}


def slice_ref(tabs, ref, s, e, *, epi, off):
    """The reference of envs [s, e) of a batch whose full reference is `ref` (its start state)."""
    r = TR.TableEnv(f32_tables(tabs), e - s, seed=SEED, env_id_offset=off + s, rng_episodic=epi, max_episode_steps=3)
    r.set_state(ref.state[:, s:e], ref.t[s:e])
    r.global_step = G0
    return r


def slices(n, stride, m=1031):
    """A head slice, one past the first grid-stride wrap and a ragged tail (starts are multiples of 4)."""
    tail = (n - m) // 4 * 4
    return [(0, m), (stride + 4 * 97, stride + 4 * 97 + m), (tail, n)]


def power(refs):
    """A row's envs must have truncated (back to the non-zero initial state of the tables)."""
    tr = sum(int(r.stats[3]) for r in refs)
    assert tr > 0


def _table_policy(C, S, A, seed):
    return np.random.default_rng(seed).integers(0, A ** C, S ** C).astype(np.int32)


# ---------------------------------------------------------------------------------------------
# 1. step kernels: cell_pair_kernel<C, RNG, SE> for every C, RNG in {none, philox, replay}, SE; cell_packed_kernel
#    <C, RNG, EXTRA> for RNG in {none, philox}, bit-identical to the int8 layout

STEP_SA = {C: [(2, 4), (3, 3), (4, 2), (3, 4)][C % 4] for C in range(1, 17)}


def step_declared(C):
    return {("cell_pair_kernel", (C, r, se)) for r in (0, 1, 2) for se in (0, 1)} | \
           {("cell_packed_kernel", (C, r, x)) for r in (0, 1) for x in (0, 1)}


def _step_run(B, tabs, *, epi, off, se, replay, packed, seed, steps=3):
    """int8 (and a packed twin) against the reference for `steps` steps; returns the reference."""
    from gym_cellular_b200.packed_env import pack_host
    kw = dict(epi=epi, off=off, emit_side_effects=se)
    env, ref = build(B, tabs, "dyadic", replay=replay, **kw)
    pk = build(B, tabs, "dyadic", packed=True, **kw)[0] if packed else None
    rng = np.random.default_rng(seed)
    start(env, ref, rng)
    if pk is not None:
        pk.set_state(dev(ref.state), t=dev(ref.t))
        from gym_cellular_b200 import _lib
        _lib.check(pk._lib.gc_set_global_step(pk._h, G0))
    q = 0
    for _ in range(steps):
        a = (rng.random((ref.C, ref.n)) * ref.A).astype(np.int8)
        ru = rng.random((ref.n, ref.C)) if replay else None
        ref.step(a, ru)
        env.step_device(dev(a), replay_u=ru) if replay else env.step_device(dev(a))
        got = gpu_out(env)
        check_step(got, ref, "dyadic")
        q += TR.q24(got["reward"])
        if pk is not None:
            pk.step_device(dev(a))
            gp = gpu_out(pk)
            check_step(gp, ref, "dyadic")
            assert (gp["flags"] == (got["unsafe"] | (got["truncated"] << 1) | (got["count"] << 2))).all()
            assert (gp["reward"].view(np.uint32) == got["reward"].view(np.uint32)).all()
            if se:
                assert (gp["se_words"] == pack_host(got["se_row"])).all()
    check_stats(env, ref, q, "dyadic")
    if pk is not None:
        assert (host(pk._stats) == host(env._stats)).all()
    return ref


@pytest.mark.parametrize("C", range(1, 17))
def test_step_kernels_every_c(B, C):
    """Per (noise, side-effect row): pair tables with S = 4 when there is no side-effect row (the packed EXTRA = 0
    kernel needs the index to be the state word), the replay kernel with the noisy tables."""
    S, A = STEP_SA[C]
    refs, fired = [], 0
    with launches() as L:
        for noise in (False, True):
            for se in (0, 1):
                s = 4 if not se else S
                tabs = make_tables(7001 * C + 11 * noise + se, C, s, A, noise=noise)
                assert derive_path(tabs) == "pair"
                epi, off = (C + se) % 2 == 0, BIG if (C + noise) % 2 else 4 * C
                refs.append(_step_run(B, tabs, epi=epi, off=off, se=bool(se), replay=False, packed=True, seed=C))
                fired += int(refs[-1].last_fire.sum())
                if noise:
                    refs.append(_step_run(B, tabs, epi=epi, off=off, se=bool(se), replay=True, packed=False, seed=C + 1))
                    fired += int(refs[-1].last_fire.sum())
    assert_launched(L, step_declared(C))
    power(refs)
    assert fired > 0


# pair8 (S, A <= 8) and the generic kernel (forced): the existing rows of test_gpu_tables cover their table shapes;
# this row reaches every instantiation of both in one test
PAIR8_DECLARED = {("cell_pair8_kernel", (r, se)) for r in (0, 1) for se in (0, 1)}
GENERIC_DECLARED = {("cell_step_kernel", (r,)) for r in (0, 1, 2)}


def test_pair8_and_generic_kernels(B):
    refs = []
    with launches() as L:
        for noise in (False, True):
            for se in (False, True):
                tabs = make_tables(811 + 2 * noise + se, 6, 6, 5, noise=noise)
                assert derive_path(tabs) == "pair8"
                refs.append(_run_plain(B, tabs, se=se, force=False, replay=False, seed=noise + 2 * se))
        for noise, replay in ((False, False), (True, False), (True, True)):
            tabs = make_tables(911 + noise + replay, 7, 4, 4, noise=noise)
            assert derive_path(tabs, force=True) == "generic"
            refs.append(_run_plain(B, tabs, se=True, force=True, replay=replay, seed=5 + noise + replay))
    assert_launched(L, PAIR8_DECLARED | GENERIC_DECLARED)
    power(refs)


def _run_plain(B, tabs, *, se, force, replay, seed, steps=3):
    env, ref = build(B, tabs, "dyadic", epi=seed % 2 == 0, off=BIG if seed % 3 == 0 else 0, replay=replay,
                     emit_side_effects=se or force, force_generic_kernel=force)
    rng = np.random.default_rng(seed)
    start(env, ref, rng)
    q = 0
    for _ in range(steps):
        a = (rng.random((ref.C, ref.n)) * ref.A).astype(np.int8)
        ru = rng.random((ref.n, ref.C)) if replay else None
        ref.step(a, ru)
        env.step_device(dev(a), replay_u=ru) if replay else env.step_device(dev(a))
        got = gpu_out(env)
        check_step(got, ref, "dyadic")
        q += TR.q24(got["reward"])
    check_stats(env, ref, q, "dyadic")
    return ref


# ---------------------------------------------------------------------------------------------
# 2. step_many, fused: cell_pair_many_kernel<C, RNG, SE, THREADS> and cell_packed_many_kernel<C, RNG, EXTRA, THREADS>,
#    C = 1..8, at 64-thread blocks (a batch that does not fill the SMs) and at 256-thread blocks with a wrapping
#    grid-stride loop; against the reference and bit for bit against the separate launches

MANY_STEPS = 7
N_MANY_BIG = (1 << 20) + 3                  # fusion applies up to 2^21 envs


def many_declared(C, threads):
    return {(k, (C, r, x, threads)) for k in ("cell_pair_many_kernel", "cell_packed_many_kernel")
            for r in (0, 1) for x in (0, 1)}


def _many_run(B, monkeypatch, tabs, *, n, packed, se, epi, off, fused, seed):
    from gym_cellular_b200.packed_env import pack_host
    monkeypatch.setenv("GC_B200_STEP_MANY_FUSED", "1" if fused else "0")
    env, ref = build(B, tabs, "dyadic", n=n, epi=epi, off=off, packed=packed, emit_side_effects=se)
    rng = np.random.default_rng(seed)
    start(env, ref, rng)
    tape = [(rng.random((ref.C, n)) * ref.A).astype(np.int8) for _ in range(3)]
    ring = []
    for a in tape:
        if packed:
            t = torch.zeros(env.ld, dtype=torch.int32, device="cuda")
            t[:n] = dev(pack_host(a).view(np.int32))
        else:
            t = torch.zeros(ref.C, env.ld, dtype=torch.int8, device="cuda")
            t[:, :n] = dev(a)
        ring.append(t)
    before = env.launch_count
    env.step_many([env._bind(t) for t in ring], MANY_STEPS)
    if fused:
        assert env.launch_count - before == 1
    return env, ref, tape


@pytest.mark.parametrize("big", [False, True], ids=["threads64", "threads256"])
@pytest.mark.parametrize("C", range(1, 9))
def test_step_many_every_kernel(B, monkeypatch, n_sm, C, big):
    n = N_MANY_BIG if big else N
    threads = 256 if big else 64
    assert ((n + 1023) // 1024 >= n_sm) == big                  # the launchers' 64/256-thread rule
    S, A = STEP_SA[C]
    for noise in (False, True):
        for se in (False, True):
            tabs = make_tables(313 * C + 2 * noise + se, C, S if se else 4, A, noise=noise)
            assert derive_path(tabs) == "pair"
            epi, off = (C + noise) % 2 == 0, BIG if (C + se) % 2 else 0
            for packed in (False, True):
                outs = []
                for fused in (True, False):
                    if fused:
                        with launches() as L:
                            env, ref, tape = _many_run(B, monkeypatch, tabs, n=n, packed=packed, se=se, epi=epi, off=off,
                                                       fused=True, seed=C)
                        key = ("cell_packed_many_kernel" if packed else "cell_pair_many_kernel",
                               (C, int(noise), int(se or (packed and tabs["n_states"] != 4)), threads))
                        assert_launched(L, {key})
                        if big:
                            assert_wraps(L, [key], n, threads)
                    else:
                        env, ref, tape = _many_run(B, monkeypatch, tabs, n=n, packed=packed, se=se, epi=epi, off=off,
                                                   fused=False, seed=C)
                    got = gpu_out(env)
                    outs.append((got, host(env._stats)))
                if big:
                    stride = L.of(key)[0][1][0] * threads * 4
                    for s, e in slices(n, stride):
                        r = slice_ref(tabs, ref, s, e, epi=epi, off=off)
                        for k in range(MANY_STEPS):
                            r.step(tape[k % 3][:, s:e])
                        check_step(sl(outs[0][0], s, e), r, "dyadic")
                else:
                    for k in range(MANY_STEPS):
                        ref.step(tape[k % 3])
                    check_step(outs[0][0], ref, "dyadic")
                    check_stats(env, ref, ref.stats[4], "dyadic")
                    assert ref.stats[3] > 0
                for k in outs[0][0]:
                    a, b = (np.ascontiguousarray(o[0][k]).view(np.uint8) for o in outs)
                    assert (a == b).all(), (k, packed, noise, se)
                assert (outs[0][1] == outs[1][1]).all()


# ---------------------------------------------------------------------------------------------
# 3. rollout / record / count: cell_rollout_kernel<C, NOISE, MODE> for every C, with and without noise

ROLL_SA = {1: (4, 4), 2: (4, 3), 3: (3, 4), 4: (4, 2), 5: (2, 4), 6: (3, 3), 7: (3, 2), 8: (2, 3), 9: (3, 3),
           10: (4, 2), 11: (2, 4), 12: (4, 3), 13: (2, 2), 14: (3, 2), 15: (2, 3), 16: (2, 3)}
JOINT_MAX = 1 << 26


def roll_declared(C, noise):
    return {("cell_rollout_kernel", (C, int(noise), m)) for m in (0, 1, 2)}


def _count_tables(S, A, C):
    nS, nA = S ** C, A ** C
    joint = nS * nA <= JOINT_MAX
    return nS, nA, joint, joint and nS * nA * nS <= JOINT_MAX


def _check_record(tr, rec):
    for k in rec:
        want, got = rec[k], host(getattr(tr, k))
        if k == "reward":
            assert (got.astype(np.float64) == want).all()
        else:
            assert (got.view(want.dtype) == want).all(), k


def _check_end(env, ref):
    assert (host(env.state) == ref.state).all() and (host(env.time_step) == ref.t).all()
    assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ref.index).all()
    check_stats(env, ref, ref.stats[4], "dyadic")


@pytest.mark.parametrize("noise", [False, True], ids=["det", "noise"])
@pytest.mark.parametrize("C", range(1, 17))
def test_rollout_modes_every_c(B, C, noise):
    S, A = ROLL_SA[C]
    assert S ** C <= 1 << 24 and A ** C < 1 << 31
    tabs = make_tables(9173 * C + noise, C, S, A, noise=noise)
    assert derive_path(tabs) == "pair"
    policy = _table_policy(C, S, A, C)
    epi, off = (C + noise) % 2 == 0, BIG if (C // 2 + noise) % 2 else 0
    nS, nA, joint, trans = _count_tables(S, A, C)
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", epi=epi, off=off)           # rollout: returns and unsafe counts
        start(env, ref, np.random.default_rng(C))
        pol = policy if C % 2 else None
        ret, uns = np.zeros(ref.n), np.zeros(ref.n, np.int64)
        for _ in range(K):
            ref.collect(1, pol)
            ret += ref.reward_out
            uns += ref.unsafe
        g_ret, g_uns = env.rollout(K, pol)
        assert (host(g_ret).astype(np.float64) == ret).all() and (host(g_uns) == uns).all()
        _check_end(env, ref)

        env, ref = build(B, tabs, "dyadic", epi=epi, off=off)           # record: every field
        start(env, ref, np.random.default_rng(C))
        rec = ref.collect(K, policy, EPS)
        _check_record(env.collect(K, policy, EPS, next_obs=True), rec)
        _check_end(env, ref)
        assert (rec["flags"] & 1).any() and (rec["flags"] & 2).any()

        env, ref = build(B, tabs, "dyadic", epi=not epi, off=BIG - off)  # count: the histogram of the reference
        start(env, ref, np.random.default_rng(C + 100))
        pol, eps = (policy, EPS) if (C + noise) % 2 else (None, 0.0)
        rec = ref.collect(K, pol, eps)
        counts = env.collect_counts(K, pol, eps, env.zero_counts(joint=joint, transitions=trans))
        assert_counts(counts, hist(rec, nS, nA, (C, S, A), joint=joint, transitions=trans))
        _check_end(env, ref)
    assert_launched(L, roll_declared(C, noise))


# 256-thread blocks, the grid-stride loop wrapping: rollout against reference slices, record on slices, counts against
# the histogram of a twin handle's record
ROLL_BIG = [dict(C=5, S=2, A=4, noise=True, epi=True, off=BIG), dict(C=13, S=2, A=2, noise=False, epi=False, off=0)]
N_ROLL_BIG = (1 << 19) + 5


@pytest.mark.parametrize("r", ROLL_BIG, ids=[f"C{r['C']}-{'noise' if r['noise'] else 'det'}" for r in ROLL_BIG])
def test_rollout_modes_256_threads(B, n_sm, r):
    C, S, A, n, epi, off = r["C"], r["S"], r["A"], N_ROLL_BIG, r["epi"], r["off"]
    assert (n + 3) // 4 >= n_sm * 512                                  # rollout_threads: 256-thread blocks
    tabs = make_tables(5077 * C, C, S, A, noise=r["noise"])
    policy = _table_policy(C, S, A, C)
    nS, nA, joint, trans = _count_tables(S, A, C)
    keys = [("cell_rollout_kernel", (C, int(r["noise"]), m)) for m in (0, 1, 2)]
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", n=n, epi=epi, off=off)
        start(env, ref, np.random.default_rng(1))
        g_ret, g_uns = (host(x) for x in env.rollout(K, policy))
        rec_env, ref2 = build(B, tabs, "dyadic", n=n, epi=epi, off=off)
        start(rec_env, ref2, np.random.default_rng(1))
        tr = rec_env.collect(K, policy, EPS, next_obs=True)
        cnt_env, ref3 = build(B, tabs, "dyadic", n=n, epi=epi, off=off)
        start(cnt_env, ref3, np.random.default_rng(1))
        counts = cnt_env.collect_counts(K, policy, EPS, cnt_env.zero_counts(joint=joint, transitions=trans))
    assert_launched(L, set(keys))
    assert_wraps(L, keys, n, 256)
    stride = L.of(keys[0])[0][1][0] * 256 * 4
    got_rec = record(tr)
    for s, e in slices(n, stride):
        rr = slice_ref(tabs, ref, s, e, epi=epi, off=off)
        ret, uns = np.zeros(e - s), np.zeros(e - s, np.int64)
        for _ in range(K):
            rr.collect(1, policy)
            ret += rr.reward_out
            uns += rr.unsafe
        assert (g_ret[s:e].astype(np.float64) == ret).all() and (g_uns[s:e] == uns).all()
        rr = slice_ref(tabs, ref2, s, e, epi=epi, off=off)
        want = rr.collect(K, policy, EPS)
        _check_record(type(tr)(**{k: getattr(tr, k)[:, s:e] if getattr(tr, k) is not None else None
                                   for k in tr._fields}), want)
    assert_counts(counts, hist(got_rec, nS, nA, (C, S, A), joint=joint, transitions=trans))
    assert torch.equal(cnt_env.state, rec_env.state) and cnt_env.stats() == rec_env.stats()


# ---------------------------------------------------------------------------------------------
# 4. grid world: grid_step_kernel<RNG, LUT_GLOBAL>, grid_many_kernel, grid_rollout_kernel<MODE> at both block sizes

GRID_STEP_DECLARED = {("grid_step_kernel", (r, g)) for r in (1, 2) for g in (0, 1)}
GRID_MANY_DECLARED = {("grid_many_kernel", ())}
GRID_ROLL_DECLARED = {("grid_rollout_kernel", (m,)) for m in (0, 1, 2)}


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


def _grid_actions(rng, n):
    g = np.full((2, n), 4, np.int8)
    g[rng.integers(0, 2, n), np.arange(n)] = rng.integers(0, 4, n)
    return g


def _grid_check(env, ora):
    assert (host(env.state) == ora.state).all() and (host(env.time_step) == ora.t).all()
    assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ora.index).all()
    n = env.num_envs
    assert (host(env._truncated[:n]) == ora.truncated).all() and (host(env._count[:n]) == ora.count).all()
    np.testing.assert_allclose(host(env._reward[:n]), ora.reward, rtol=1e-6, atol=1e-7)


def test_grid_step_kernels(B, O, n_sm):
    """Both LUT placements (the table read from global memory for batches of at most three waves, staged in shared
    memory above) x Philox / replay."""
    wave = n_sm * 2 * 512 * 4                # one wave of 512-thread blocks, 2 per SM, 4 envs a thread (gc_grid.cu)
    with launches() as L:
        for n in (10007, 3 * wave + 5):
            for replay in (False, True):
                env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=3, dispersal_prob=0.2, max_episode_steps=4,
                                          env_id_offset=BIG if replay else 0)
                ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=3, dispersal_prob=0.2, max_episode_steps=4,
                                  env_id_offset=BIG if replay else 0, replay=replay)
                rng = np.random.default_rng(n + replay)
                for _ in range(3):
                    a = _grid_actions(rng, n)
                    ru = rng.random((n, 6)) if replay else None
                    ora.step(a, ru)
                    env.step_device(dev(a), replay_u=ru) if replay else env.step_device(dev(a))
                    _grid_check(env, ora)
                assert ora.truncated.sum() > 0 or ora.t.max() > 0
    assert_launched(L, GRID_STEP_DECLARED)


def test_grid_many_kernel(B, O, monkeypatch):
    n = 10007
    outs = []
    for fused in ("1", "0"):
        monkeypatch.setenv("GC_B200_STEP_MANY_FUSED", fused)
        with launches() as L:
            env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=5, dispersal_prob=0.2, max_episode_steps=4)
            ora = O.OracleEnv(kind="gridworld", n_envs=n, seed=5, dispersal_prob=0.2, max_episode_steps=4)
            rng = np.random.default_rng(2)
            tape = [_grid_actions(rng, n) for _ in range(3)]
            ring = []
            for a in tape:
                t = torch.zeros(2, env.ld, dtype=torch.int8, device="cuda")
                t[:, :n] = dev(a)
                ring.append(t)
            before = env.launch_count
            env.step_many([env._bind(t) for t in ring], MANY_STEPS)
            launched = env.launch_count - before
            for k in range(MANY_STEPS):
                ora.step(tape[k % 3])
            _grid_check(env, ora)
        if fused == "1":
            assert launched == 1
            assert_launched(L, GRID_MANY_DECLARED)
        outs.append((host(env.state), host(env._reward[:n]).view(np.uint32), host(env._stats)))
    for a, b in zip(*outs):
        assert (a == b).all()


@pytest.mark.parametrize("big", [False, True], ids=["threads64", "threads256"])
def test_grid_rollout_modes(B, O, golden_gw, n_sm, big):
    from test_gpu_counts import _gw_policy
    n = (1 << 19) + 5 if big else 10007
    threads = 256 if big else 64
    assert ((n + 3) // 4 >= n_sm * 128) == big
    policy = _gw_policy(golden_gw)
    kw = dict(kind="gridworld", num_envs=n, env_seed=9, dispersal_prob=0.05, max_episode_steps=7, env_id_offset=BIG)
    okw = dict(kind="gridworld", n_envs=n, seed=9, dispersal_prob=0.05, max_episode_steps=7, env_id_offset=BIG)
    with launches() as L:
        env, ora = B.CellularVectorEnv(**kw), O.OracleEnv(**okw)
        g_ret, g_uns = env.rollout(6)
        ret, uns = ora.rollout(6)
        np.testing.assert_allclose(host(g_ret), ret, rtol=1e-6)
        assert (host(g_uns) == 0).all() and (host(env.state) == ora.state).all()
        rec_env, ora = B.CellularVectorEnv(**kw), O.OracleEnv(**okw)
        tr = rec_env.collect(6, policy, EPS, next_obs=True)
        obs, act, rew, flags = CO.collect(ora, 6, policy, EPS)
        assert (host(tr.obs).view(np.uint32) == obs).all() and (host(tr.action).view(np.uint32) == act).all()
        assert (host(tr.flags) == flags).all() and (host(tr.reward) == rew).all()
        assert (host(rec_env.state) == ora.state).all() and (host(rec_env.time_step) == ora.t).all()
        cnt_env = B.CellularVectorEnv(**kw)
        counts = cnt_env.collect_counts(6, policy, EPS)
    assert_launched(L, GRID_ROLL_DECLARED)
    for m in (0, 1, 2):
        assert all(e[2][0] == threads for e in L.of(("grid_rollout_kernel", (m,))))
    assert_counts(counts, hist(record(tr), 400, 25))
    assert torch.equal(cnt_env.state, rec_env.state) and cnt_env.stats() == rec_env.stats()


# ---------------------------------------------------------------------------------------------
# 5. the codec, reset, pack / unpack and step-counter kernels

AUX_DECLARED = {(k, ()) for k in ("encode_kernel", "decode_kernel", "encode_mixed_kernel", "decode_mixed_kernel",
                                  "reset_kernel", "reset_packed_kernel", "pack_kernel", "unpack_kernel", "tick_kernel")}


def test_codec_reset_pack_and_tick(B):
    from gym_cellular_b200.packed_env import pack_host
    radix = [2, 4, 3, 4, 2, 3]
    with launches() as L:
        tabs = make_tables(77, 6, 4, 4, noise=True, radix=radix)
        env, ref = build(B, tabs, "dyadic", radix=radix)                           # reset_kernel at construction
        rng = np.random.default_rng(6)
        start(env, ref, rng, radix)
        assert (host(env.tabularize(env.state)) == ref.index).all()                        # encode_mixed
        assert (host(env.detabularize(torch.from_numpy(ref.index.astype(np.int64)).cuda())) == ref.state).all()
        u, uref = build(B, make_tables(78, 5, 3, 3, noise=False), "dyadic")
        start(u, uref, rng)
        assert (host(u.tabularize(u.state)) == uref.index).all()                           # encode
        assert (host(u.detabularize(torch.from_numpy(uref.index.astype(np.int64)).cuda())) == uref.state).all()
        u.reset()
        uref.reset()
        assert (host(u.state) == uref.state).all() and (host(u.time_step) == 0).all()
        pk, pref = build(B, make_tables(79, 9, 4, 4, noise=False), "dyadic", packed=True)
        start(pk, pref, rng)                                                               # pack
        assert (host(pk.packed_state).view(np.uint32) == pack_host(pref.state)).all()
        assert (host(pk.state) == pref.state).all()                                        # unpack
        mask = rng.random(pref.n) < 0.5
        pk.reset_envs(torch.from_numpy(mask).cuda())                                       # reset_packed
        want = np.where(mask[None, :], pref.init[:, None], pref.state)
        assert (host(pk.state) == want).all() and (host(pk.time_step)[mask] == 0).all()
        h, href = build(B, make_tables(80, 4, 3, 3, noise=True), "dyadic", host_chunk_envs=1008)
        start(h, href, rng)
        a = (rng.random((4, href.n)) * 3).astype(np.int8)
        href.step(a)
        obs, rew, term, trunc, info = h.step(a)                                            # chunked: tick_kernel
        assert (np.stack(obs) == href.state).all()
        assert h.sync_step_counter() == G0 + 1
    assert_launched(L, AUX_DECLARED)


# ---------------------------------------------------------------------------------------------
# the guard

EXCLUDED = {}                   # (kernel, template values): reason


def declared():
    out = set(PAIR8_DECLARED | GENERIC_DECLARED | GRID_STEP_DECLARED | GRID_MANY_DECLARED |
              GRID_ROLL_DECLARED | AUX_DECLARED)
    for C in range(1, 17):
        out |= step_declared(C) | roll_declared(C, False) | roll_declared(C, True)
    for C in range(1, 9):
        out |= many_declared(C, 64) | many_declared(C, 256)
    return out


def test_every_instantiation_has_a_row():
    inv = inventory()
    rows = declared()
    assert not (rows & set(EXCLUDED)), sorted(rows & set(EXCLUDED))
    assert rows | set(EXCLUDED) == inv, dict(missing=sorted(inv - rows - set(EXCLUDED)), unknown=sorted(rows - inv))
    print(f"{len(inv)} instantiations, {len(rows)} reached by a row, {len(EXCLUDED)} excluded")
