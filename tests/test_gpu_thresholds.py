"""Every Philox threshold compare at its exact boundary, in every kernel that draws.

Everything random reduces to a compare of a 32-bit value v with ceil(p * 2^32): the narrow cellular compare
`word <= thr - 1`, the SWAR compare of the wide envs (`fire_bits_wide`, with its k16 >= 0x8000 branch) and its tie
path (`noise_fire_with_ties`), the grid-world dispersal trigger and the explore test of `collect`.  A random test
cannot see an off-by-one there (it moves P by 2^-32 per draw), so each boundary case picks ONE draw v of a target env
g, cell c and counter T from the numpy restatement of DESIGN §4 (`_noise_draws`) and runs two handles of the same
ragged batch: A at p = v * 2^-32 (the target must not fire) and B at p = (v + 1) * 2^-32 (it must fire).  The oracle
runs of A and B must differ in env g only -- that proves the numpy derivation and the oracle agree on which draw
decides -- and the GPU must equal the oracle bit for bit in both.  For a wide env the target is a tie with the
threshold's top half by construction, so the low-half compare sits exactly at its boundary.

The sweep runs whole batches (2^16 envs x 16 cells: every 16-bit half value occurs many times per step) at the edge
probabilities of the three compare forms, against the oracle."""
import ctypes as C
import math

import numpy as np
import pytest

import _collect_oracle as CO
import _noise_draws as ND

REWARD_RTOL = 1e-6
REWARD_ATOL = 1e-7
N = 4099                         # ragged: the last 4-env group of a thread holds 3 envs
SEED = 0x0123456789ABCDEF        # both key words non-zero
T0 = 5                           # episode step the episodic cases start from
G0 = 7                           # global step the non-episodic cases start from
SEARCH_FROM = 8192               # env ids >= every local index, so that env_id_offset = g - local >= 0


@pytest.fixture(scope="module")
def B():
    torch = pytest.importorskip("torch")
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    return oracle


@pytest.fixture(scope="module")
def torch():
    return pytest.importorskip("torch")


def host(t):
    return t.cpu().numpy()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _lib():
    from gym_cellular_b200 import _lib as lib
    return lib


def set_global_step(env, step):
    _lib().check(env._lib.gc_set_global_step(env._h, step))


def prob(v):
    return v * 2.0 ** -32          # exact in double for every 32-bit v (and v = 2^32 gives 1.0)


# ---------------------------------------------------------------------------------------------
# targets

WIDE_KINDS = {                   # name: (top half, low half) constraint; None = any
    "tie_mid": (None, "mid"),    # the tie path, both outcomes
    "low_0000": (None, 0x0000),  # A has r16 = 0: a tie can never fire
    "low_ffff": (None, 0xFFFF),  # B carries into k16 and takes no tie
    "top_0000": (0x0000, None),  # k16 = 0: only the tie path can fire
    "top_7fff": (0x7FFF, None),
    "top_8000": (0x8000, None),  # the noise_kmask branch of the SWAR compare
    "top_ffff": (0xFFFF, None),
}
NARROW_KINDS = {"mid": lambda d: (d >> 28 >= 4) & (d >> 28 < 8), "top_bit": lambda d: d >= 0xC0000000}
# A wide draw of value 2^32 - 1 (both halves 0xFFFF, 2^-32 per draw: found by a search over the env ids of this seed,
# re-derived by every case that uses it): p = 1 - 2^-32 must not fire it, p = 1 must -- the clamp of a threshold of
# 2^32 to k16 = 0xFFFF, r16 = 2^16.  (n_cells, T, g, c)
MAX_DRAW = (16, T0, 100456401, 11)

_cache = {}


def cell_targets(n_cells, T, kind):
    """Candidates (g, c, v): draws of cell c of env g at counter T of the wanted kind."""
    key = (n_cells, T, kind)
    if key not in _cache:
        if kind == "max_draw":
            assert (n_cells, T) == MAX_DRAW[:2]
            g, c = MAX_DRAW[2:]
            hits = [(g, c, int(ND.cell_draws(SEED, n_cells, g, 1, T)[c, 0]))]
        elif n_cells <= ND.NARROW_CELLS:
            hits = ND.search(lambda f, m: ND.cell_draws(SEED, n_cells, f, m, T), NARROW_KINDS[kind], SEARCH_FROM)
        elif WIDE_KINDS[kind][1] == "mid":
            hits = ND.search(lambda f, m: ND.cell_draws(SEED, n_cells, f, m, T),
                             lambda d: ((d & 0xFFFF) >= 0x1000) & ((d & 0xFFFF) < 0xF000), SEARCH_FROM, n=1 << 12)
        else:
            top_is, low_is = WIDE_KINDS[kind]
            hits = ND.search_wide(SEED, n_cells, T, top_is, low_is, SEARCH_FROM)
        _cache[key] = hits
    return _cache[key]


def word_targets(words, T, kind):
    key = (words.__name__, T, kind)
    if key not in _cache:
        _cache[key] = ND.search(lambda f, m: words(SEED, f, m, T), NARROW_KINDS[kind], SEARCH_FROM)
    return _cache[key]


def place(g, where):
    """Local index of env g (mid-batch, or in the last, partial 4-env group) and the env_id_offset that puts it
    there; None if g cannot sit there."""
    local = (2048 if where == "mid" else 4096) + g % 4
    return None if local >= N else (local, g - local)


def placed(cands, where):
    for g, c, v in cands:
        p = place(g, where)
        if p is not None:
            yield (g, c, v) + p


# ---------------------------------------------------------------------------------------------
# comparisons

def gpu_outputs(env, outputs=True):
    import torch
    n = env.num_envs
    out = dict(state=host(env.state), index=host(env.tabular_state(torch.int32)).view(np.uint32), t=host(env.time_step))
    if outputs:
        if hasattr(env, "_flags"):
            f = host(env._flags[:n])
            out.update(unsafe=f & 1, truncated=(f >> 1) & 1, count=f >> 2)
        else:
            out.update(unsafe=host(env._unsafe[:n]), truncated=host(env._truncated[:n]), count=host(env._count[:n]))
        out["reward"] = host(env._reward[:n])
        if getattr(env, "_se_row", None) is not None and env._se_row.dim() == 2:
            out["se_row"] = host(env._se_row[:, :n])
    return out


def ora_outputs(ora, outputs=True):
    out = dict(state=ora.state.copy(), index=ora.index.copy(), t=ora.t.copy())
    if outputs:
        out.update(unsafe=ora.unsafe.copy(), truncated=ora.truncated.copy(), count=ora.count.copy(),
                   reward=ora.reward.copy(), se_row=ora.se_row.copy())
    return out


def assert_gpu_equals_oracle(env, ora, outputs=True):
    got, want = gpu_outputs(env, outputs), ora_outputs(ora, outputs)
    for k, v in got.items():
        if k == "reward":
            np.testing.assert_allclose(v, want[k], rtol=REWARD_RTOL, atol=REWARD_ATOL)
        else:
            assert (v == want[k]).all(), k
    s = env.stats()
    assert (s["env_steps"], s["unsafe_steps"], s["count_sum"], s["episodes_truncated"]) == tuple(ora.stats[:4])


def columns_except(a, local):
    return np.delete(a, local, axis=a.ndim - 1)


def assert_only_env_differs(a, b, local):
    """Oracle A and oracle B agree on every env but `local` (dicts of [.., n] arrays)."""
    for k in a:
        assert (columns_except(a[k], local) == columns_except(b[k], local)).all(), k


def assert_only_cell_fired(a_state, b_state, c, local):
    """After the target step the oracle runs differ in cell c of env `local` only, and B's level is the lower one."""
    diff = np.argwhere(a_state != b_state)
    assert diff.tolist() == [[c, local]], diff.tolist()
    assert b_state[c, local] == a_state[c, local] - 1


def assert_record_equal(tr, rec):
    obs, act, rew, flags = rec
    assert (host(tr.obs).view(np.uint32) == obs).all()
    assert (host(tr.action).view(np.uint32) == act).all()
    assert (host(tr.flags) == flags).all()
    np.testing.assert_allclose(host(tr.reward), rew, rtol=REWARD_RTOL, atol=REWARD_ATOL)


# ---------------------------------------------------------------------------------------------
# (a) cellular noise at its boundary

CELL_ROWS = {                    # name: (env class, n_states, env kwargs)
    "pair": ("CellularVectorEnv", 4, {}),
    "pair_nose": ("CellularVectorEnv", 4, dict(emit_side_effects=False)),
    "generic": ("CellularVectorEnv", 3, dict(force_generic_kernel=True)),
    "pair8": ("CellularVectorEnv", 5, {}),
    "packed": ("PackedCellularVectorEnv", 4, {}),
}
CELL_CASES = (                   # (row, drive, n_cells, rng_episodic)
    [("pair", "step", C, C % 2 == 1) for C in (3, 4, 5, 9, 16)]
    + [("pair_nose", "step", C, C % 2 == 0) for C in (3, 5, 16)]
    + [("generic", "step", C, True) for C in (3, 9)]
    + [("pair8", "step", C, False) for C in (3, 10)]
    + [("packed", "step", C, C == 3) for C in (3, 16)]
    + [("pair", "many", C, C == 3) for C in (3, 7)]
    + [("packed", "many", C, C == 7) for C in (3, 7)]
    + [("pair", drive, C, C == 16) for drive in ("rollout", "collect") for C in (3, 16)]
)
MAX_DRAW_CASES = [(row, "step", 16, True) for row in ("pair", "pair_nose", "generic", "packed")] + \
                 [("pair", drive, 16, True) for drive in ("rollout", "collect")]


def _kinds(C):
    return sorted(NARROW_KINDS) if C <= ND.NARROW_CELLS else sorted(WIDE_KINDS)


CELL_PARAMS = [pytest.param(row, drive, C, epi, kind, id=f"{row}-{drive}-C{C}-{'epi' if epi else 'glob'}-{kind}")
               for row, drive, C, epi in CELL_CASES for kind in _kinds(C)] + \
              [pytest.param(row, drive, C, epi, "max_draw", id=f"{row}-{drive}-C{C}-epi-max_draw") for row, drive, C, epi in MAX_DRAW_CASES]


def _drive_plan(drive, C, S):
    """(steps, target step, start level, policy) of a drive.  From a level >= 1 a cell whose action moves it up
    consumes a draw at every step, and a fired draw drops it one level: every target is visible."""
    if drive == "step":
        return 1, 0, 1, None
    if drive == "many":
        return 3, 2, 1, None                                   # the target at step k = 2 of the fused launch
    if C <= 3:                                                 # a table policy that moves every cell up
        return 3, 1, 1, np.full(S ** C, S ** C - 1, np.int32)
    return 3, 0, 2, None                                       # random actions: from level 2 of 4 every move draws


@pytest.mark.gpu
@pytest.mark.parametrize("row,drive,C,episodic,kind", CELL_PARAMS)
def test_noise_boundary(B, O, torch, row, drive, C, episodic, kind):
    cls, S, ekw = CELL_ROWS[row]
    if drive in ("rollout", "collect") and C <= 3:
        S = 3
    K, k_t, level, policy = _drive_plan(drive, C, S)
    T = (T0 if episodic else G0) + k_t
    where = "mid" if kind == "max_draw" or sorted(_kinds(C)).index(kind) % 2 == 0 else "last"
    g, c, v, local, off = next(placed(cell_targets(C, T, kind), where))
    if C > ND.NARROW_CELLS:                     # the numpy draws: at p = v * 2^-32 the target ties with k16
        assert int(ND.wide_tops(SEED, C, g, 1, T)[c, 0]) == ND.top(v) == v >> 16
        assert int(ND.wide_lows(SEED, [c], g, 1, T)[0, 0]) == ND.low(v)
        assert kind != "max_draw" or (v == 0xFFFFFFFF and prob(v + 1) == 1.0)
    else:
        assert int(ND.cell_draws(SEED, C, g, 1, T)[c, 0]) == v

    envs, oras = [], []
    for p in (prob(v), prob(v + 1)):
        env = getattr(B, cls)(num_envs=N, n_cells=C, n_states=S, stochastic=True, rng_episodic=episodic, noise_prob=p,
                              env_seed=SEED, env_id_offset=off, **ekw)
        ora = O.OracleEnv(n_envs=N, n_cells=C, n_states=S, noise=True, rng_episodic=episodic, noise_prob=p, seed=SEED,
                          env_id_offset=off, reward="nonlinear_rp")
        cells = np.full((C, N), level, np.int8)
        env.set_state(dev(cells), t=torch.full((N,), T0, dtype=torch.int32) if episodic else None)
        ora.state[:] = cells
        ora.index[:] = O.encode(cells, S)
        if episodic:
            ora.t[:] = T0
        else:
            set_global_step(env, G0)
            ora.global_step = G0
        envs.append(env)
        oras.append(ora)

    # the oracle runs
    up = np.full((C, N), S - 1, np.int8)
    recs = [[], []]
    for k in range(K):
        for i, ora in enumerate(oras):
            if drive == "collect":
                recs[i].append(CO.collect(ora, 1, policy))
            elif drive == "rollout":
                ora.step(ora.policy_actions(policy))
            else:
                ora.step(up)
        if k == k_t:
            assert_only_cell_fired(oras[0].state, oras[1].state, c, local)
    outputs = drive in ("step", "many")
    assert_only_env_differs(ora_outputs(oras[0], outputs), ora_outputs(oras[1], outputs), local)

    # the GPU runs
    for i, (env, ora) in enumerate(zip(envs, oras)):
        if drive == "step":
            env.step_device(dev(up))
        elif drive == "many":
            if cls == "CellularVectorEnv":
                ring = [torch.full((C, env.ld), S - 1, dtype=torch.int8, device="cuda") for _ in range(2)]
            else:
                word = sum((S - 1) << (2 * j) for j in range(C))
                ring = [torch.full((env.ld,), word, dtype=torch.int32, device="cuda") for _ in range(2)]
            env.step_many([env._bind(a) for a in ring], K)
        elif drive == "rollout":
            env.rollout(K, policy)
        else:
            tr = env.collect(K, policy)
            assert_record_equal(tr, [np.concatenate(f) for f in zip(*recs[i])])
        assert_gpu_equals_oracle(env, ora, outputs)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(NARROW_KINDS))
def test_noise_boundary_deadlock(B, O, torch, kind):
    """With `deadlock` a polarised cell stays polarised: the target cell starts below the top level."""
    C, S = 3, 4
    g, c, v, local, off = next(placed(cell_targets(C, T0, kind), "mid"))
    envs, oras = [], []
    for p in (prob(v), prob(v + 1)):
        env = B.CellularVectorEnv(num_envs=N, n_cells=C, n_states=S, stochastic=True, deadlock=True, rng_episodic=True,
                                  noise_prob=p, env_seed=SEED, env_id_offset=off)
        ora = O.OracleEnv(n_envs=N, n_cells=C, n_states=S, noise=True, deadlock=True, rng_episodic=True, noise_prob=p,
                          seed=SEED, env_id_offset=off, reward="nonlinear_rp")
        cells = np.full((C, N), 1, np.int8)
        env.set_state(dev(cells), t=torch.full((N,), T0, dtype=torch.int32))
        ora.state[:], ora.t[:], ora.index[:] = cells, T0, O.encode(cells, S)
        a = np.full((C, N), 2, np.int8)                        # 1 -> 2, below the top level 3
        ora.step(a)
        env.step_device(dev(a))
        envs.append(env)
        oras.append(ora)
    assert_only_cell_fired(oras[0].state, oras[1].state, c, local)
    assert_only_env_differs(ora_outputs(oras[0]), ora_outputs(oras[1]), local)
    for env, ora in zip(envs, oras):
        assert_gpu_equals_oracle(env, ora)


# ---------------------------------------------------------------------------------------------
# (a) grid-world dispersal and the explore test of collect at their boundaries

GRID_DRIVES = {"step": (1, 0), "many": (3, 2), "rollout": (3, 1), "collect": (3, 1)}


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(NARROW_KINDS))
@pytest.mark.parametrize("drive", sorted(GRID_DRIVES))
def test_dispersal_boundary(B, O, torch, drive, kind):
    K, k_t = GRID_DRIVES[drive]
    T = G0 + k_t
    a = np.full((2, N), 4, np.int8)
    a[0] = 3                                                    # the agent stays at (1, 1) of jurisdiction 0
    tried = 0
    for g, _, v, local, off in placed(word_targets(ND.grid_triggers, T, kind), "last" if drive == "step" else "mid"):
        tried += 1
        assert tried <= 12, "no candidate whose dispersal changes the state"
        oras = []
        for p in (prob(v), prob(v + 1)):
            ora = O.OracleEnv(kind="gridworld", n_envs=N, seed=SEED, dispersal_prob=p, env_id_offset=off)
            ora.global_step = G0
            oras.append(ora)
        recs = [[], []]
        for k in range(K):
            for i, ora in enumerate(oras):
                if drive == "collect":
                    recs[i].append(CO.collect(ora, 1))
                elif drive == "rollout":
                    ora.step(ora.policy_actions(None))
                else:
                    ora.step(a)
            if k == k_t:
                diff = np.argwhere(oras[0].state != oras[1].state)
        if len(diff) == 0:
            continue                                            # dispersal re-seeded what was there: next candidate
        assert set(diff[:, 1].tolist()) == {local}
        outputs = drive in ("step", "many")
        assert_only_env_differs(ora_outputs(oras[0], outputs), ora_outputs(oras[1], outputs), local)
        for i, (p, ora) in enumerate(zip((prob(v), prob(v + 1)), oras)):
            env = B.CellularVectorEnv(kind="gridworld", num_envs=N, env_seed=SEED, dispersal_prob=p, env_id_offset=off)
            set_global_step(env, G0)
            if drive == "step":
                env.step_device(dev(a))
            elif drive == "many":
                ring = []
                for _ in range(2):
                    t = torch.zeros(2, env.ld, dtype=torch.int8, device="cuda")
                    t[:, :N] = dev(a)
                    ring.append(t)
                env.step_many([env._bind(x) for x in ring], K)
            elif drive == "rollout":
                env.rollout(K)
            else:
                assert_record_equal(env.collect(K), [np.concatenate(f) for f in zip(*recs[i])])
            assert_gpu_equals_oracle(env, ora, outputs)
        return


def _gw_policy(golden_gw):
    policy = np.zeros(400, np.int32)
    st, pol = golden_gw["gw_states"].astype(int), golden_gw["gw_initial_policy"].astype(int)
    policy[st[:, 0] + 20 * st[:, 1]] = pol[:, 0] + 5 * pol[:, 1]
    return policy


@pytest.mark.gpu
@pytest.mark.parametrize("kind", sorted(NARROW_KINDS))
@pytest.mark.parametrize("family", ["cellular", "gridworld"])
def test_explore_boundary(B, O, golden_gw, family, kind):
    """epsilon = v * 2^-32 against (v + 1) * 2^-32 on the explore word of the target env at global step G0 + 1: the
    recorded actions differ at that env and step only."""
    K, k_t = 3, 1
    if family == "cellular":
        policy = np.random.default_rng(3).integers(0, 27, 27).astype(np.int32)
        ekw, okw = dict(stochastic=True, rng_episodic=True), dict(noise=True, rng_episodic=True, reward="nonlinear_rp")
    else:
        policy = _gw_policy(golden_gw)
        ekw, okw = {}, {}
    tried = 0
    for g, _, v, local, off in placed(word_targets(ND.explore_words, G0 + k_t, kind), "mid" if kind == "mid" else "last"):
        tried += 1
        assert tried <= 12, "no candidate whose explored action differs from the table's"
        eps = (prob(v), prob(v + 1))
        oras = [O.OracleEnv(kind=family, n_envs=N, seed=SEED, env_id_offset=off, **okw) for _ in eps]
        for ora in oras:
            ora.global_step = G0
        recs = [CO.collect(ora, K, policy, e) for ora, e in zip(oras, eps)]
        act_diff = np.argwhere(recs[0][1] != recs[1][1])
        if len(act_diff) == 0:
            continue                                            # the explored action happened to be the table's
        # first at the target step, and at the target env only (later table actions follow its diverged state)
        assert act_diff[0].tolist() == [k_t, local] and set(act_diff[:, 1].tolist()) == {local}
        for f in range(4):                                      # obs, action, reward, flags
            assert (recs[0][f][:k_t] == recs[1][f][:k_t]).all()
            assert (columns_except(recs[0][f], local) == columns_except(recs[1][f], local)).all()
        assert (recs[0][0][k_t] == recs[1][0][k_t]).all()
        assert_only_env_differs(ora_outputs(oras[0], False), ora_outputs(oras[1], False), local)
        for e, ora, rec in zip(eps, oras, recs):
            env = B.CellularVectorEnv(kind=family, num_envs=N, env_seed=SEED, env_id_offset=off, **ekw)
            set_global_step(env, G0)
            assert_record_equal(env.collect(K, policy, e), rec)
            assert_gpu_equals_oracle(env, ora, outputs=False)
        return


# ---------------------------------------------------------------------------------------------
# (b) threshold sweep: whole batches at the edge probabilities

SWEEP_P = [2.0 ** -32, 1e-6, 2.0 ** -16, (2 ** 31 - 1) * 2.0 ** -32, 0.5, (2 ** 31 + 1) * 2.0 ** -32, 0.75,
           1 - 2.0 ** -32, 1 - 2.0 ** -16, 1.0]
SWEEP_ROWS = {                   # name: (env class, n_cells, n_states, env kwargs, drive)
    "pair16": ("CellularVectorEnv", 16, 4, {}, "step"),
    "packed16": ("PackedCellularVectorEnv", 16, 4, {}, "step"),
    "generic16": ("CellularVectorEnv", 16, 4, dict(force_generic_kernel=True), "step"),
    "rollout16": ("CellularVectorEnv", 16, 4, {}, "rollout"),
    "pair8_10": ("CellularVectorEnv", 10, 5, {}, "step"),
    "pair4": ("CellularVectorEnv", 4, 4, {}, "step"),
}
SWEEP_N = 1 << 16


def k16_of(p):
    thr = math.ceil(p * 2.0 ** 32)
    return min(thr >> 16, 0xFFFF)


@pytest.mark.gpu
@pytest.mark.parametrize("p", SWEEP_P, ids=[f"p{p!r}" for p in SWEEP_P])
@pytest.mark.parametrize("row", sorted(SWEEP_ROWS))
def test_threshold_sweep(B, O, torch, row, p):
    cls, C, S, ekw, drive = SWEEP_ROWS[row]
    n, steps = SWEEP_N, 3
    env = getattr(B, cls)(num_envs=n, n_cells=C, n_states=S, stochastic=True, rng_episodic=True, noise_prob=p,
                          env_seed=SEED, env_id_offset=4 * 77777, **ekw)
    ora = O.OracleEnv(n_envs=n, n_cells=C, n_states=S, noise=True, rng_episodic=True, noise_prob=p, seed=SEED,
                      env_id_offset=4 * 77777, reward="nonlinear_rp")
    level = 2 if drive == "rollout" else 1           # every cell draws at every step (rollout: at its first step)
    cells = np.full((C, n), level, np.int8)
    env.set_state(dev(cells))
    ora.state[:], ora.index[:] = cells, O.encode(cells, S)
    if C > ND.NARROW_CELLS:                          # the batch ties with the threshold's top half: not vacuous
        tops = ND.wide_tops(SEED, C, 4 * 77777, n, 0)
        assert (tops == k16_of(p)).sum() >= 1
    from gym_cellular_b200 import tables
    move, noisy, draws = tables.noise_tables(S, S)
    up = np.full((C, n), S - 1, np.int8)
    for k in range(steps):
        before = ora.state.copy()
        a = ora.policy_actions(None) if drive == "rollout" else up
        ora.step(a)
        if p == 1.0:                                  # every draw-consuming cell fired
            d = draws[before, a].astype(bool)
            assert d.any() and (ora.state == np.where(d, noisy[before, a], move[before, a])).all()
        if drive == "step":
            env.step_device(dev(a))
            assert_gpu_equals_oracle(env, ora)
    if drive == "rollout":
        env.rollout(steps)
        assert_gpu_equals_oracle(env, ora, outputs=False)


# ---------------------------------------------------------------------------------------------
# probabilities outside [0, 1] are rejected

def _cfg(_lib, **kw):
    cfg = _lib.GcConfig()
    cfg.struct_size = C.sizeof(cfg)
    cfg.n_envs, cfg.ld, cfg.n_cells, cfg.n_states, cfg.n_actions = 16, 16, 3, 3, 3
    cfg.noise_prob, cfg.dispersal_prob = 0.1, 0.01
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def test_create_rejects_probabilities_outside_the_unit_interval():
    """Validated before any CUDA call: NaN, negative and > 1 values of noise_prob and dispersal_prob are errors, not
    'never' or 'always'."""
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    L = _lib.load()
    h = C.c_void_p()
    for field in ("noise_prob", "dispersal_prob"):
        for bad in (float("nan"), -0.1, -5e-324, 1.5, 1.0 + 2.0 ** -52, float("inf")):
            for kind in (_lib.KIND_CELLULAR, _lib.KIND_GRIDWORLD):
                kw = dict(kind=kind) if kind == _lib.KIND_CELLULAR else dict(kind=kind, n_cells=2, n_states=20, n_actions=5)
                assert L.gc_create(C.byref(_cfg(_lib, **{field: bad}, **kw)), C.byref(h)) == _lib.ERR_INVALID
                assert field.encode() in L.gc_last_error(), (field, bad)
    for ok in (0.0, 1.0, 2.0 ** -32):                 # accepted: whatever fails next is not about the probabilities
        for field in ("noise_prob", "dispersal_prob"):
            rc = L.gc_create(C.byref(_cfg(_lib, **{field: ok})), C.byref(h))
            if rc == _lib.OK:
                L.gc_destroy(h)
            else:
                assert b"_prob" not in L.gc_last_error()


@pytest.mark.gpu
def test_env_rejects_probabilities_outside_the_unit_interval(B):
    from gym_cellular_b200 import tables
    for bad in (float("nan"), -0.1, 1.5):
        with pytest.raises(_lib().GcError) as ei:
            B.CellularVectorEnv(num_envs=16, stochastic=True, noise_prob=bad)
        assert ei.value.code == _lib().ERR_INVALID and "noise_prob" in ei.value.message
        with pytest.raises(_lib().GcError) as ei:
            B.CellularVectorEnv(num_envs=16, cell_tables=dict(tables.deep_exploration_tables(), noise_prob=bad))
        assert ei.value.code == _lib().ERR_INVALID and "noise_prob" in ei.value.message
    with pytest.raises(_lib().GcError) as ei:
        B.CellularVectorEnv(kind="gridworld", num_envs=16, dispersal_prob=1.5)
    assert ei.value.code == _lib().ERR_INVALID and "dispersal_prob" in ei.value.message
    for ok in (0.0, 1.0):
        B.CellularVectorEnv(num_envs=16, stochastic=True, noise_prob=ok)
        B.CellularVectorEnv(kind="gridworld", num_envs=16, dispersal_prob=ok)
        B.CellularVectorEnv(num_envs=16, cell_tables=dict(tables.deep_exploration_tables(), noise_prob=ok))
