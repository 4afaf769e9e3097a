"""Reward BITS of every cellular kernel: against the float32 restatement of its arithmetic (tests/_reward_f32.py), with
+0.0 for a zero sum, and with log2(1 + .) a function of the env's own sum alone.

Dyadic rewards (test_gpu_tables.py) add exactly in any order; the families here round: `uniform` (random float32) and
`cancel` (+-127/C-sized entries among entries near 2^-20, so that sums cancel and round hard) are compared with the
model bit for bit, `negzero` (tables holding -0.0, with (level, action) rows where every entry a cell can reach is
-0.0) checks the sign of zero sums.  Every row asserts that it ran the kernels it names (test_gpu_every_kernel)."""
import numpy as np
import pytest

import _reward_f32 as RF
from test_gpu_counts import assert_counts, hist
from test_gpu_every_kernel import launches
from test_gpu_tables import BIG, G0, build, derive_path, dev, gpu_out, host, make_tables, start

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N = 4099
K = 3
CHUNK = 1008                     # host paths: chunks that do not divide N


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def f32(x):
    return np.float32(x)


def nextafter(x, y):
    return np.nextafter(f32(x), f32(y))


# ---------------------------------------------------------------------------------------------
# tables

def fam_rewards(rng, fam, C, S, A):
    if fam == "uniform":
        return rng.uniform(-1.0, 1.0, (S, A)).astype(np.float32)
    if fam == "cancel":
        sign = rng.choice([-1.0, 1.0], (S, A))
        big = sign * np.floor(127.0 / C * rng.uniform(0.5, 1.0, (S, A)) * 2 ** 16) * 2.0 ** -16
        small = sign * rng.uniform(1.0, 2.0, (S, A)) * 2.0 ** -20
        return np.where(rng.random((S, A)) < 0.5, big, small).astype(np.float32)
    assert fam == "negzero"                     # level 0 and action 0: -0.0 for every cell; elsewhere -0.0 or +-k/4
    r = np.where(rng.random((S, A)) < 0.4, -0.0, rng.integers(-4, 5, (S, A)) / 4.0).astype(np.float32)
    r[0, :] = r[:, 0] = -0.0
    return r


def tables(seed, fam, C, S, A, noise):
    tabs = make_tables(seed, C, S, A, noise=noise)
    rng = np.random.default_rng(seed + 1)
    tabs["reward"] = fam_rewards(rng, fam, C, S, A)
    if noise:
        tabs["reward_noisy"] = fam_rewards(rng, fam, C, S, A)
        if fam == "negzero":
            tabs["reward_noisy"][tabs["reward"].view(np.uint32) == 0x80000000] = -0.0
    return tabs


def step_actions(rng, ref, zero_frac=0.0):
    """Random actions; a fraction of the envs takes action 0 in every cell (a -0.0 entry for each cell in negzero)."""
    a = (rng.random((ref.C, ref.n)) * ref.A).astype(np.int8)
    a[:, rng.random(ref.n) < zero_frac] = 0
    return a


def check_model(got, ref, family):
    want = RF.prelog(ref, family)
    bad = np.flatnonzero(RF.bits(got) != RF.bits(want))
    assert bad.size == 0, dict(family=family, envs=bad[:5].tolist(), got=got[bad[:5]].tolist(), want=want[bad[:5]].tolist())
    return int(RF.q24(want).sum())


def assert_ran(L, name, *prefix):
    """Some launch of kernel `name` whose template values start with `prefix` (the rest, such as whether the
    side-effect row is written, is not what the row is about)."""
    hits = [k for k in L.names() if k[0] == name and tuple(k[1][:len(prefix)]) == prefix]
    assert hits, dict(want=(name, prefix), launched=sorted(L.names(), key=str))


def check_stats(env, q):
    s = host(env._stats)
    assert s[4] == q, (int(s[4]), q)


# ---------------------------------------------------------------------------------------------
# 1. pre-log bits against the model: step kernels (int8 + packed twin), fused step_many, pair8, generic, host paths

STEP_C = [1, 2, 3, 4, 5, 7, 8, 9, 16]
STEP_PARAMS = [pytest.param(C, noise, fam, id=f"C{C}-{'noise' if noise else 'det'}-{fam}")
               for C in STEP_C for noise in (False, True) for fam in ("uniform", "cancel")]


@pytest.mark.parametrize("C,noise,fam", STEP_PARAMS)
def test_step_kernel_reward_bits(B, C, noise, fam):
    A = 3 if C % 2 else 4
    tabs = tables(1000 * C + 10 * noise + len(fam), fam, C, 4, A, noise)
    assert derive_path(tabs) == "pair"
    epi, off = C % 2 == 0, BIG if C % 3 == 0 else 4 * C
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", epi=epi, off=off)
        pk, _ = build(B, tabs, "dyadic", epi=epi, off=off, packed=True)
        rng = np.random.default_rng(C)
        start(env, ref, rng)
        pk.set_state(dev(ref.state), t=dev(ref.t))
        from gym_cellular_b200 import _lib
        _lib.check(pk._lib.gc_set_global_step(pk._h, G0))
        q, fired = 0, 0
        for _ in range(K):
            a = step_actions(rng, ref)
            ref.step(a)
            fired += int(ref.last_fire.sum())
            env.step_device(dev(a))
            pk.step_device(dev(a))
            g, gp = gpu_out(env), gpu_out(pk)
            assert (g["state"] == ref.state).all() and (gp["state"] == ref.state).all()
            q += check_model(g["reward"], ref, RF.PAIR)
            check_model(gp["reward"], ref, RF.PAIR)
        check_stats(env, q)
        check_stats(pk, q)
    assert_ran(L, "cell_pair_kernel", C, int(noise))
    assert_ran(L, "cell_packed_kernel", C, int(noise))
    assert fired > 0 or not noise


MANY_PARAMS = [pytest.param(C, packed, id=f"C{C}-{'packed' if packed else 'int8'}") for C in range(1, 9)
               for packed in (False, True)]


def many_run(B, monkeypatch, tabs, fam, *, packed, fused, seed, steps=7, cells=None, t0=None, tape=None, n=N,
             log2=False):
    """`steps` bound steps over a ring of three action tensors in one gc_step_many call; returns (env, ref, tape)."""
    from gym_cellular_b200 import _lib
    from gym_cellular_b200.packed_env import pack_host
    monkeypatch.setenv("GC_B200_STEP_MANY_FUSED", "1" if fused else "0")
    env, ref = build(B, tabs, "log2" if log2 else "dyadic", n=n, epi=seed % 2 == 0, off=BIG if seed % 3 else 0,
                     packed=packed, limit=0 if cells is not None else 3)
    rng = np.random.default_rng(seed)
    if cells is None:
        start(env, ref, rng)
    else:
        ref.set_state(cells, t0)
        ref.global_step = G0
        env.set_state(dev(cells), t=dev(t0))
        _lib.check(env._lib.gc_set_global_step(env._h, G0))
    if tape is None:
        tape = [step_actions(rng, ref) for _ in range(3)]
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
    env.step_many([env._bind(t) for t in ring], steps)
    if fused:
        assert env.launch_count - before == 1
    return env, ref, tape


@pytest.mark.parametrize("C,packed", MANY_PARAMS)
def test_step_many_reward_bits(B, monkeypatch, C, packed):
    """The fused kernel: its last step against the model, its reward statistic against the model's q24 of every step,
    and every output bit-identical with the separate launches."""
    noise, fam = C % 2 == 1, ("uniform", "cancel")[C % 2]
    tabs = tables(2000 + C, fam, C, 4, 4, noise)
    outs = []
    for fused in (True, False):
        with launches() as L:
            env, ref, tape = many_run(B, monkeypatch, tabs, fam, packed=packed, fused=fused, seed=C)
        if fused:
            kern = "cell_packed_many_kernel" if packed else "cell_pair_many_kernel"
            assert_ran(L, kern, C, int(noise))
        q = 0
        for k in range(7):
            ref.step(tape[k % 3])
            q += int(RF.q24(RF.prelog(ref, RF.PAIR)).sum())
        got = gpu_out(env)
        check_model(got["reward"], ref, RF.PAIR)
        check_stats(env, q)
        outs.append((got["reward"].view(np.uint32), host(env._stats)))
    assert (outs[0][0] == outs[1][0]).all() and (outs[0][1] == outs[1][1]).all()


PAIR8_PARAMS = [pytest.param(noise, fam, id=f"{'noise' if noise else 'det'}-{fam}")
                for noise in (False, True) for fam in ("uniform", "cancel")]


@pytest.mark.parametrize("noise,fam", PAIR8_PARAMS)
def test_pair8_reward_bits(B, noise, fam):
    """pair8: the pair entries without noise, single entries in cell order with it."""
    C = 7
    tabs = tables(3000 + noise, fam, C, 6, 5, noise)
    assert derive_path(tabs) == "pair8"
    family = RF.SINGLE if noise else RF.PAIR
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", epi=True, off=BIG)
        rng = np.random.default_rng(5)
        start(env, ref, rng)
        q = 0
        for _ in range(K):
            a = step_actions(rng, ref)
            ref.step(a)
            env.step_device(dev(a))
            q += check_model(host(env._reward[:ref.n]), ref, family)
        check_stats(env, q)
    assert_ran(L, "cell_pair8_kernel", int(noise))
    if noise:       # the two families differ on these tables: the row tells them apart
        assert (RF.bits(RF.prelog(ref, RF.PAIR)) != RF.bits(RF.prelog(ref, RF.SINGLE))).any()


@pytest.mark.parametrize("noise,fam", PAIR8_PARAMS)
def test_generic_kernel_reward_bits(B, noise, fam):
    C = 9
    tabs = tables(4000 + noise, fam, C, 4, 4, noise)
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", epi=False, off=0, force_generic_kernel=True, emit_side_effects=True)
        rng = np.random.default_rng(6)
        start(env, ref, rng)
        q = 0
        for _ in range(K):
            a = step_actions(rng, ref)
            ref.step(a)
            env.step_device(dev(a))
            q += check_model(host(env._reward[:ref.n]), ref, RF.SINGLE)
        check_stats(env, q)
    assert_ran(L, "cell_step_kernel", int(noise))


@pytest.mark.parametrize("packed", [False, True], ids=["int8", "packed"])
def test_host_path_reward_bits(B, packed):
    """gc_step_host / gc_step_host_packed in chunks of 1008 envs (which do not divide 4099)."""
    from gym_cellular_b200.packed_env import pack_host
    C = 9 if packed else 6
    tabs = tables(5000 + packed, "cancel" if packed else "uniform", C, 4, 4, True)
    with launches() as L:
        env, ref = build(B, tabs, "dyadic", epi=not packed, off=BIG, packed=packed, host_chunk_envs=CHUNK)
        rng = np.random.default_rng(8)
        start(env, ref, rng)
        q = 0
        for _ in range(K):
            a = step_actions(rng, ref)
            ref.step(a)
            obs, rew, term, trunc, info = env.step(pack_host(a) if packed else a)
            q += check_model(np.asarray(rew, np.float32), ref, RF.PAIR)
        check_stats(env, q)
    assert_ran(L, "cell_packed_kernel" if packed else "cell_pair_kernel", C, 1)


# ---------------------------------------------------------------------------------------------
# 2. rollout / collect / counts against the model

def _policy(C, S, A, seed):
    return np.random.default_rng(seed).integers(0, A ** C, S ** C).astype(np.int32)


@pytest.mark.parametrize("fam", ["uniform", "cancel"])
@pytest.mark.parametrize("C", [3, 6], ids=["C3", "C6"])
def test_rollout_collect_counts_reward_bits(B, C, fam):
    S, A = 3, 3
    tabs = tables(6000 + C + len(fam), fam, C, S, A, True)
    pol, eps = _policy(C, S, A, C), 0.3
    with launches() as L:
        # rollout: the float32 running sum, from 0, of the per-step model rewards
        env, ref = build(B, tabs, "dyadic", epi=True, off=BIG)
        start(env, ref, np.random.default_rng(1))
        ret, q = np.zeros(ref.n, np.float32), 0
        for _ in range(K):
            ref.collect(1, None)
            ret = ret + RF.prelog(ref, RF.PAIR)
            q += int(RF.q24(RF.prelog(ref, RF.PAIR)).sum())
        g_ret, _ = env.rollout(K)
        assert (RF.bits(host(g_ret)) == RF.bits(ret)).all()
        check_stats(env, q)
        # collect: the model, and the step kernel replaying the recorded actions from the same start
        env, ref = build(B, tabs, "dyadic", epi=True, off=BIG)
        twin, _ = build(B, tabs, "dyadic", epi=True, off=BIG)
        start(env, ref, np.random.default_rng(2))
        twin.set_state(dev(ref.state), t=dev(ref.t))
        from gym_cellular_b200 import _lib
        _lib.check(twin._lib.gc_set_global_step(twin._h, G0))
        model, q = [], 0
        for _ in range(K):
            ref.collect(1, pol, eps)
            model.append(RF.prelog(ref, RF.PAIR))
            q += int(RF.q24(model[-1]).sum())
        tr = env.collect(K, pol, eps, next_obs=True)
        rew, act = host(tr.reward), host(tr.action).view(np.uint32).astype(np.int64)
        check_stats(env, q)
        for k in range(K):
            assert (RF.bits(rew[k]) == RF.bits(model[k])).all(), k
            cells = np.stack([(act[k] // A ** c) % A for c in range(C)]).astype(np.int8)
            twin.step_device(dev(cells))
            assert (RF.bits(host(twin._reward[:ref.n])) == RF.bits(rew[k])).all(), k
        # counts: reward_q24 = the histogram of the model's per-step q24
        env, ref = build(B, tabs, "dyadic", epi=True, off=BIG)
        start(env, ref, np.random.default_rng(3))
        rec = {k: [] for k in ("obs", "action", "reward", "flags", "next_obs")}
        for _ in range(K):
            one = ref.collect(1, pol, eps)
            one["reward"] = RF.prelog(ref, RF.PAIR)[None, :]
            for k in rec:
                rec[k].append(one[k])
        rec = {k: np.concatenate(v) for k, v in rec.items()}
        trans = C == 3                                  # 3^18 transition bins of six cells: too large to hold
        counts = env.collect_counts(K, pol, eps, env.zero_counts(transitions=trans))
        assert_counts(counts, hist(rec, S ** C, A ** C, (C, S, A), transitions=trans))
    for m in (0, 1, 2):
        assert_ran(L, "cell_rollout_kernel", C, 1, m)
    assert_ran(L, "cell_pair_kernel", C, 1)


# ---------------------------------------------------------------------------------------------
# 3. signed zero: wherever the float64 reference reward is 0, every path returns +0.0 (bits 0x00000000)

def _zero_check(got, ref):
    zero = ref.reward_pre_log == 0
    assert zero.sum() > 10
    bad = np.flatnonzero(zero & (RF.bits(got) != 0))
    assert bad.size == 0, dict(envs=bad[:5].tolist(), bits=[hex(b) for b in RF.bits(got)[bad[:5]]])


ZERO_PATHS = ["int8", "packed", "many_int8", "many_packed", "pair8", "pair8_noise", "generic", "host_int8",
              "host_packed", "rollout", "collect"]


@pytest.mark.parametrize("log2", [False, True], ids=["plain", "log2"])
@pytest.mark.parametrize("path", ZERO_PATHS)
def test_zero_reward_is_positive_zero(B, monkeypatch, path, log2):
    from gym_cellular_b200.packed_env import pack_host
    C = 3
    S, A = (6, 5) if path.startswith("pair8") else (4, 4)
    noise = path in ("int8", "packed", "pair8_noise", "generic", "host_packed", "collect", "many_packed")
    tabs = tables(7000 + ZERO_PATHS.index(path), "negzero", C, S, A, noise)
    if log2:
        tabs["reward"] = np.where(tabs["reward"] < 0, np.float32(-0.25), tabs["reward"])    # sums above -1
        if noise:
            tabs["reward_noisy"] = np.where(tabs["reward_noisy"] < 0, np.float32(-0.25), tabs["reward_noisy"])
    fam = "log2" if log2 else "dyadic"
    packed = path in ("packed", "many_packed", "host_packed")
    z = int(noise)
    kern = {"int8": ("cell_pair_kernel", C, z), "packed": ("cell_packed_kernel", C, z),
            "many_int8": ("cell_pair_many_kernel", C, z), "many_packed": ("cell_packed_many_kernel", C, z),
            "pair8": ("cell_pair8_kernel", 0), "pair8_noise": ("cell_pair8_kernel", 1), "generic": ("cell_step_kernel", z),
            "host_int8": ("cell_pair_kernel", C, z), "host_packed": ("cell_packed_kernel", C, z),
            "rollout": ("cell_rollout_kernel", C, z, 0), "collect": ("cell_rollout_kernel", C, z, 1)}[path]
    with launches() as L:
        if path.startswith("many"):
            rng = np.random.default_rng(0)
            tape = [(rng.random((C, N)) * A).astype(np.int8) for _ in range(3)]
            for a in tape:
                a[:, rng.random(N) < 0.5] = 0
            env, ref, tape = many_run(B, monkeypatch, tabs, fam, packed=packed, fused=True, seed=4, steps=4, tape=tape,
                                      log2=log2)
            for k in range(4):
                ref.step(tape[k % 3])
            _zero_check(host(env._reward[:ref.n]), ref)
        elif path in ("rollout", "collect"):
            env, ref = build(B, tabs, fam, epi=True, off=BIG)
            start(env, ref, np.random.default_rng(1))
            pol = np.zeros(S ** C, np.int32) if path == "collect" else None     # action 0 everywhere: -0.0 entries
            if path == "rollout":
                for _ in range(2):
                    ref.collect(1, None)
                g_ret, _ = env.rollout(2)
                zero = ref.reward_pre_log == 0          # the last step; check the return where both steps were zero
                ret = host(g_ret)
                assert not (np.signbit(ret) & (ret == 0)).any()
                assert zero.any()
            else:
                ref.collect(1, pol, 0.0)
                tr = env.collect(1, pol, 0.0)
                _zero_check(host(tr.reward)[0], ref)
        else:
            kw = dict(force_generic_kernel=True) if path == "generic" else {}
            if path.startswith("host"):
                kw["host_chunk_envs"] = CHUNK
            env, ref = build(B, tabs, fam, epi=True, off=BIG, packed=packed, **kw)
            rng = np.random.default_rng(2)
            start(env, ref, rng)
            for _ in range(2):
                a = step_actions(rng, ref, zero_frac=0.5)
                ref.step(a)
                if path.startswith("host"):
                    _, rew, *_ = env.step(pack_host(a) if packed else a)
                    got = np.asarray(rew, np.float32)
                else:
                    env.step_device(dev(a))
                    got = host(env._reward[:ref.n])
                _zero_check(got, ref)
                if not log2:
                    check_model(got, ref, RF.SINGLE if path in ("generic", "pair8_noise") else RF.PAIR)
    assert_ran(L, *kern)


# ---------------------------------------------------------------------------------------------
# 4. log2: neighbour independence, one function of the entry in every kernel, accuracy at the edges

LO_MIN = f32(-1.0 + 2.0 ** -18 + 2.0 ** -24)      # the smallest entry gc_set_tables admits for one cell under log2
HI_MAX = nextafter(128.0, 0.0)                      # the largest |entry| it admits for one cell
TARGETS = [f32(-0.5), nextafter(-0.5, 1.0), nextafter(1.0, 0.0), f32(1.0), f32(2.0 ** -30), f32(0.3), f32(-0.2),
           f32(0.77), f32(2.0 ** -126), f32(2.0 ** -127)]             # in [-1/2, 1]
HIGHS = [nextafter(1.0, 2.0), f32(3.5), HI_MAX]
LOWS = [nextafter(-0.5, -1.0), f32(-0.75), LO_MIN]
ENTRIES = TARGETS + HIGHS + LOWS                                       # 16 = the 4 x 4 table of one cell
CONTEXTS = ("in_range", "high_mate", "low_mate")


def _log2_table(S, A, values):
    """One cell, deterministic; move[s][a] = s keeps every env at its level, so every step repeats its reward."""
    v = np.asarray(values, np.float32)
    tabs = make_tables(77, 1, S, A, noise=False)
    tabs["move"] = np.repeat(np.arange(S)[:, None], A, 1).astype(np.int8)
    tabs["reward"] = v.reshape(S, A) if v.size == S * A else np.repeat(v[:, None], A, 1)
    return tabs


def _words_of(target_ids, mates, highs, lows):
    """Env layout: for every target, context and lane, one 4-env word with the target in that lane.  Returns the entry
    id of every env and, per target, the env positions where it sits."""
    ids, where = [], {}
    for j, t in enumerate(target_ids):
        for ci, ctx in enumerate(CONTEXTS):
            for lane in range(4):
                word = [mates[(j + i) % len(mates)] for i in range(4)]
                if ctx == "high_mate":
                    word[(lane + 1) % 4] = highs[(j + lane) % len(highs)]
                elif ctx == "low_mate":
                    word[(lane + 3) % 4] = lows[(j + lane) % len(lows)]
                word[lane] = t
                where.setdefault(t, []).append(len(ids) + lane)
                ids += word
    return np.array(ids), where


def _step_kernel_log2(B, monkeypatch, kernel):
    """(entry value per env, reward bits per env) of one step of a C = 1 log2 table through `kernel`."""
    S, A = (4, 5) if kernel == "pair8" else (4, 4)
    vals = np.array(ENTRIES, np.float32).reshape(4, 4)
    table = np.concatenate([vals, vals[:, :A - 4]], 1) if A > 4 else vals
    tabs = _log2_table(S, A, table)
    t_ids = list(range(len(TARGETS)))
    ids, _ = _words_of(t_ids, t_ids, list(range(10, 13)), list(range(13, 16)))
    ids = np.concatenate([ids, np.repeat(np.arange(16), 4)])            # every entry also in a word of its own
    n = ids.size
    cells, acts = (ids // 4)[None, :].astype(np.int8), (ids % 4)[None, :].astype(np.int8)
    t0 = np.zeros(n, np.int32)
    if kernel in ("many_int8", "many_packed"):
        env, ref, _ = many_run(B, monkeypatch, tabs, "log2", packed=kernel == "many_packed", fused=True, seed=6, steps=3,
                               cells=cells, t0=t0, tape=[acts] * 3, n=n, log2=True)
    else:
        from gym_cellular_b200 import _lib
        env, ref = build(B, tabs, "log2", n=n, epi=True, limit=0, packed=kernel == "packed",
                         force_generic_kernel=kernel == "generic")
        env.set_state(dev(cells), t=dev(t0))
        _lib.check(env._lib.gc_set_global_step(env._h, G0))
        env.step_device(dev(acts))
    return vals.ravel()[ids], host(env._reward[:n])


def _fused_log2(B, kernel):
    """The same for rollout / collect / counts: C = 1 tables whose reward depends on the level only (so the random
    policy does not matter), one table per target: level 0 = the target, 1 a high entry, 2 a low one, 3 an in-range
    mate.  Returns (entry value per env and step, reward bits per env and step); counts return the q24 check."""
    vals, outs = [], []
    for j, t in enumerate(TARGETS):
        levels = [t, HIGHS[j % 3], LOWS[j % 3], TARGETS[(j + 1) % len(TARGETS)]]
        tabs = _log2_table(4, 4, levels)
        ids, _ = _words_of([0], [3], [1], [2])
        n = ids.size
        env, ref = build(B, tabs, "log2", n=n, epi=True, limit=0)
        env.set_state(dev(ids[None, :].astype(np.int8)), t=dev(np.zeros(n, np.int32)))
        lv = np.asarray(levels, np.float32)[ids]
        if kernel == "rollout":
            g_ret, _ = env.rollout(K)
            vals.append(lv)
            outs.append(host(g_ret))
        elif kernel == "collect":
            tr = env.collect(K, None)
            r = host(tr.reward)
            for k in range(K):
                vals.append(lv)
                outs.append(r[k])
        else:
            counts = env.collect_counts(K, None, 0.0, env.zero_counts())
            visits, rq = host(counts.visits), host(counts.reward_q24)
            outs.append((visits, rq))
            vals.append(lv)
    return vals, outs


def _assert_one_value_per_entry(vals, got, what):
    for v in np.unique(RF.bits(vals)):
        b = np.unique(RF.bits(got)[RF.bits(vals) == v])
        assert b.size == 1, dict(kernel=what, entry=float(np.uint32(v).view(np.float32)), bits=[hex(x) for x in b])


STEP_LOG2 = {"pair": ("cell_pair_kernel", 1, 0), "packed": ("cell_packed_kernel", 1, 0), "pair8": ("cell_pair8_kernel", 0),
             "many_int8": ("cell_pair_many_kernel", 1, 0), "many_packed": ("cell_packed_many_kernel", 1, 0),
             "generic": ("cell_step_kernel", 0)}
FUSED_LOG2 = {"rollout": 0, "collect": 1, "counts": 2}


@pytest.mark.parametrize("kernel", list(STEP_LOG2) + list(FUSED_LOG2))
def test_log2_independent_of_word_mates(B, monkeypatch, kernel):
    """An env whose pre-log sum lies in [-1/2, 1], in each lane of a 4-env word whose other envs are all in range, or
    hold one sum above 1, or one below -1/2: the same reward bits in every placement."""
    with launches() as L:
        if kernel in STEP_LOG2:
            vals, got = _step_kernel_log2(B, monkeypatch, kernel)
            _assert_one_value_per_entry(vals, got, kernel)
        elif kernel in ("rollout", "collect"):
            vals, got = _fused_log2(B, kernel)
            _assert_one_value_per_entry(np.concatenate(vals), np.concatenate(got), kernel)
        else:
            # every target env sits at level 0 at every step: reward_q24[0, a] = visits[0, a] x q24 of its one value
            vals, got = _fused_log2(B, "counts")
            _, ref_bits = _fused_log2(B, "collect")
            for j, (visits, rq) in enumerate(got):
                one = ref_bits[j * K][0]                      # the target's collect reward (env 0 of the layout)
                assert (rq[0] == visits[0] * RF.q24(np.array([one]))[0]).all(), TARGETS[j]
    assert_ran(L, *(STEP_LOG2.get(kernel) or ("cell_rollout_kernel", 1, 0, FUSED_LOG2[kernel])))


def test_log2_same_function_in_every_kernel_and_accurate(B, monkeypatch):
    """With one cell the pre-log sum is the table entry itself in every kernel: every kernel maps an entry to the same
    bits, within 6e-7 relative of float64 log2(1 + r).  Below 2^-125 the polynomial's quotient r / (2 + r) is below the
    smallest normal float and div.approx.ftz flushes it: the result is 0, within 2^-124 of log2(1 + r)."""
    per_entry = {}
    for kernel in STEP_LOG2:
        vals, got = _step_kernel_log2(B, monkeypatch, kernel)
        for v, b in zip(RF.bits(vals), RF.bits(got)):
            per_entry.setdefault(int(v), set()).add((kernel, int(b)))
    for kernel in ("collect",):
        vals, got = _fused_log2(B, kernel)
        for v, b in zip(RF.bits(np.concatenate(vals)), RF.bits(np.concatenate(got))):
            per_entry.setdefault(int(v), set()).add((kernel, int(b)))
    bad = {}
    for v, kb in per_entry.items():
        if len({b for _, b in kb}) != 1:
            bad[float(np.uint32(v).view(np.float32))] = sorted((k, hex(b)) for k, b in kb)
    assert not bad, bad
    for v, kb in per_entry.items():
        r = float(np.uint32(v).view(np.float32))
        got = float(np.uint32(next(iter(kb))[1]).view(np.float32))
        want = np.log1p(r) / np.log(2.0)
        if abs(r) >= 2.0 ** -125:
            assert abs(got - want) <= 6e-7 * abs(want), (r, got, want)
        else:
            assert abs(got - want) <= 2.0 ** -124, (r, got, want)


# ---------------------------------------------------------------------------------------------
# 5. permutation: the envs of a deterministic batch permuted (state, t and actions together) permute the rewards

PERM_PATHS = ["int8", "packed", "many_int8", "pair8", "generic", "host_int8", "rollout", "collect"]


@pytest.mark.parametrize("log2", [False, True], ids=["uniform", "log2"])
@pytest.mark.parametrize("path", PERM_PATHS)
def test_rewards_permute_with_the_envs(B, monkeypatch, path, log2):
    C = 5
    S, A = (6, 5) if path == "pair8" else (4, 4)
    tabs = make_tables(8000 + PERM_PATHS.index(path), C, S, A, noise=False)
    rng = np.random.default_rng(9)
    # log2: sums from -0.5 to 2, so that words mix in-range and out-of-range sums
    tabs["reward"] = (rng.uniform(-0.1, 0.4, (S, A)) if log2 else rng.uniform(-1, 1, (S, A))).astype(np.float32)
    fam = "log2" if log2 else "dyadic"
    n = N
    cells = (rng.random((C, n)) * S).astype(np.int8)
    t0 = rng.integers(0, 3, n).astype(np.int32)
    acts = (rng.random((C, n)) * A).astype(np.int8)
    perm = rng.permutation(n)
    pol = _policy(C, S, A, 3)
    kw = dict(force_generic_kernel=True) if path == "generic" else {}
    if path == "host_int8":
        kw["host_chunk_envs"] = CHUNK
    out = []
    with launches() as L:
        for order in (np.arange(n), perm):
            c, t, a = cells[:, order], t0[order], acts[:, order]
            if path == "many_int8":
                env, _, _ = many_run(B, monkeypatch, tabs, fam, packed=False, fused=True, seed=0, steps=2, cells=c, t0=t,
                                     tape=[a] * 3, log2=log2)
                out.append(host(env._reward[:n]))
                continue
            from gym_cellular_b200 import _lib
            env, _ = build(B, tabs, fam, epi=True, limit=0, packed=path == "packed", **kw)
            env.set_state(dev(c), t=dev(t))
            _lib.check(env._lib.gc_set_global_step(env._h, G0))
            if path == "rollout":
                out.append(host(env.rollout(K, pol)[0]))
            elif path == "collect":
                out.append(host(env.collect(K, pol).reward))
            elif path == "host_int8":
                out.append(np.asarray(env.step(a)[1], np.float32))
            else:
                env.step_device(dev(a))
                out.append(host(env._reward[:n]))
    base, permuted = (RF.bits(o) for o in out)
    assert (base[..., perm] == permuted).all()
    kern = {"int8": ("cell_pair_kernel", C, 0), "packed": ("cell_packed_kernel", C, 0),
            "many_int8": ("cell_pair_many_kernel", C, 0), "pair8": ("cell_pair8_kernel", 0), "generic": ("cell_step_kernel", 0),
            "host_int8": ("cell_pair_kernel", C, 0), "rollout": ("cell_rollout_kernel", C, 0, 0),
            "collect": ("cell_rollout_kernel", C, 0, 1)}[path]
    assert_ran(L, *kern)
