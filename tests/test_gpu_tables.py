"""Random cell tables through every cellular kernel, against the float64 table reference (tests/_table_reference.py).

The oracle hard-codes the reference's rules, so every other GPU test runs tables of one structure: one step towards the
action, counted = {S - 1}, an all-zero initial state, A = S, side effects from 3 x 3 role tables with entry 0 never
'unsafe' and one table for every cell j >= 2.  Here a seeded generator draws tables the header admits and nothing
else: any move / noisy table, draws on about half the (level, action) pairs, a random counted subset, a non-zero
initial state, side-effect codes with about 1/6 'unsafe' (entry 0 included), A != S and rewards of either sign.

Rewards are dyadic (multiples of 2^-8 in [-8, 8]; for the large family up to the bound gc_set_tables enforces,
n_cells x max|reward| < 128) unless a row says otherwise: float32 sums of them are exact in any order, so they are
compared bit for bit.  The non-dyadic families are
compared against a rounding bound.  The reward statistic is checked exactly against the GPU's own float outputs.

Each row names the path `gc_set_tables` takes for its tables (`derive_path` restates the rule of gc_api.cu), and each
case checks its own power: draws fire at a fraction near p, `unsafe` takes both values, some env truncates back to the
non-zero initial state and `count` takes at least two values."""
import ctypes as C
import math
import zlib

import numpy as np
import pytest

import _table_reference as TR

pytestmark = pytest.mark.gpu

SEED = 0x243F6A8885A308D3
P = 0.3
G0 = 5
BIG = (1 << 32) + 4 * 12345
N = 4099
K = 6


@pytest.fixture(scope="module")
def B():
    torch = pytest.importorskip("torch")
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def host(t):
    return t.cpu().numpy()


def dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _lib():
    from gym_cellular_b200 import _lib as lib
    return lib


# ---------------------------------------------------------------------------------------------
# tables

def _rewards(rng, fam, C, S, A):
    if fam == "dyadic":
        return rng.integers(-8 * 256, 8 * 256 + 1, (S, A)) / 256.0
    if fam == "large":                                      # up to the bound: C * max|r| = 127 at most
        m = int(127 / C * 256)
        r = rng.integers(-m, m + 1, (S, A)) / 256.0
        r.flat[rng.choice(S * A, 2, replace=False)] = (m / 256.0, -m / 256.0)
        return r
    if fam == "uniform":
        return rng.uniform(-1.0, 1.0, (S, A))
    assert fam == "log2"                                    # every sum stays >= -1/2
    return rng.uniform(-0.5 / C, 1.0, (S, A))


def make_tables(seed, C, S, A, *, noise, fam="dyadic", se_mode="pair", radix=None):
    """A random table set; se_mode 'pair' copies SE[2] to every cell j >= 3, 'generic' makes them differ."""
    rng = np.random.default_rng(seed)
    if radix is None:
        move, noisy = rng.integers(0, S, (S, A)), rng.integers(0, S, (S, A))
    else:                                                   # next(s, a) <= max(s, a): cell c stays below radix[c]
        hi = np.maximum.outer(np.arange(S), np.arange(A)) + 1
        move, noisy = (rng.random((S, A)) * hi).astype(int), (rng.random((S, A)) * hi).astype(int)
    draws = rng.random((S, A)) < 0.5
    counted = np.zeros(S, np.uint8)
    counted[rng.choice(S, rng.integers(1, S), replace=False)] = 1
    levels = np.array(radix if radix is not None else [S] * C)
    init = rng.integers(0, levels)
    if not init.any():
        init[int(np.argmax(levels))] = 1
    se = rng.choice(3, size=(C, S, S), p=[5 / 12, 5 / 12, 1 / 6])
    if not (se[0] == 2).any():
        se[0, rng.integers(S), rng.integers(S)] = 2
    if C == 1:                                              # entry 0 pairs cell 0 with itself: the diagonal
        k = rng.integers(S)
        se[0, k, k], se[0, (k + 1) % S, (k + 1) % S] = 2, 1
    if se_mode == "pair":
        se[3:] = se[2:3]
    else:
        assert C >= 4
        while (se[3] == se[2]).all():
            se[3] = rng.choice(3, size=(S, S), p=[5 / 12, 5 / 12, 1 / 6])
    tabs = dict(n_cells=C, n_states=S, n_actions=A, move=move.astype(np.int8), reward=_rewards(rng, fam, C, S, A),
                side_effects=se.astype(np.int8), counted=counted, initial_state=init.astype(np.int8),
                reset_row=[1] + [0] * (C - 1), noise_prob=P)
    if noise:
        tabs.update(noisy=noisy.astype(np.int8), draws=draws.astype(np.uint8), reward_noisy=_rewards(rng, fam, C, S, A))
    return tabs


def derive_path(tabs, radix=None, force=False):
    """The kernel family `gc_set_tables` selects (gc_api.cu): the pair table for S, A <= 4, the 3-bit pair table for
    S, A <= 8, else the generic kernel -- the first two only for a uniform radix, without GC_F_GENERIC_KERNEL and when
    every cell j >= 3 has the side-effect table of cell 2."""
    C, S, A, se = tabs["n_cells"], tabs["n_states"], tabs["n_actions"], tabs["side_effects"]
    ragged = radix is not None and any(r != S for r in radix)
    shared = all((se[j] == se[2]).all() for j in range(3, C))
    if not ragged and not force and shared:
        if S <= 4 and A <= 4:
            return "pair"
        if S <= 8 and A <= 8:
            return "pair8"
    return "generic"


def _log_reward(tab):
    """A per-cell table reward under log2(1 + sum), lowered as `CellularVectorEnv` lowers a CellReward."""
    from gym_cellular_b200 import tables

    class _T(tables.CellReward):
        def __init__(self):
            self.__name__, self.log2, self.spec = "table_log2", True, None
            self.n_states, self.n_actions = tab.shape

        def table(self, n_states, n_actions):
            return tab
    return _T()


def f32_tables(tabs):
    """The reward tables as the device receives them."""
    out = dict(tabs, reward=np.asarray(tabs["reward"], np.float32))
    if "reward_noisy" in tabs:
        out["reward_noisy"] = np.asarray(tabs["reward_noisy"], np.float32)
    return out


def build(B, tabs, fam, *, n=N, epi=True, limit=3, off=0, packed=False, radix=None, replay=False, **kw):
    cls = B.PackedCellularVectorEnv if packed else B.CellularVectorEnv
    rf = _log_reward(tabs["reward"]) if fam == "log2" else None
    env = cls(num_envs=n, cell_tables=tabs, reward_func=rf, env_seed=SEED, env_id_offset=off, rng_episodic=epi,
              max_episode_steps=limit, cell_radix=radix, **kw)
    ref = TR.TableEnv(f32_tables(tabs), n, seed=SEED, env_id_offset=off, rng_episodic=epi, max_episode_steps=limit,
                      reward_log2=fam == "log2", radix=radix, replay=replay)
    return env, ref


def start_ref(ref, rng, radix=None):
    """Puts the reference at random states (below each cell's radix), random episode steps and global step G0."""
    levels = np.array(radix if radix is not None else [ref.S] * ref.C)[:, None]
    cells = (rng.random((ref.C, ref.n)) * levels).astype(np.int8)
    t0 = rng.integers(0, max(ref.limit, 1), ref.n).astype(np.int32)
    ref.set_state(cells, t0)
    ref.global_step = G0
    return cells, t0


def start(env, ref, rng, radix=None):
    """Checks the reset state (the non-zero initial state and its index), then puts both at the states of
    `start_ref`."""
    import torch
    got = gpu_out(env)
    assert (got["state"] == ref.state).all() and (got["index"] == ref.index).all() and (got["t"] == 0).all()
    cells, t0 = start_ref(ref, rng, radix)
    env.set_state(dev(cells), t=torch.from_numpy(t0).cuda())
    _lib().check(env._lib.gc_set_global_step(env._h, G0))


def actions(rng, ref, radix=None):
    levels = np.minimum(np.array(radix if radix is not None else [ref.A] * ref.C), ref.A)[:, None]
    return (rng.random((ref.C, ref.n)) * levels).astype(np.int8)


# ---------------------------------------------------------------------------------------------
# comparisons

def _unpack(words, C):
    from gym_cellular_b200.packed_env import unpack_host
    return unpack_host(words.view(np.uint32), C)


def gpu_out(env):
    import torch
    n, Cn = env.num_envs, env.n_cells
    o = dict(state=host(env.state), index=host(env.tabular_state(torch.int32)).view(np.uint32), t=host(env.time_step),
             reward=host(env._reward[:n]))
    if hasattr(env, "_flags"):
        f = host(env._flags[:n])
        o.update(flags=f, unsafe=f & 1, truncated=(f >> 1) & 1, count=f >> 2)
        if env._se_row is not None:
            o["se_words"] = host(env._se_row[:n]).view(np.uint32)
            o["se_row"] = _unpack(o["se_words"], Cn)
        if env._final is not None:
            o["final_words"] = host(env._final[:n]).view(np.uint32)
            o["final"] = _unpack(o["final_words"], Cn)
    else:
        o.update(unsafe=host(env._unsafe[:n]), truncated=host(env._truncated[:n]), count=host(env._count[:n]))
        if env._se_row is not None:
            o["se_row"] = host(env._se_row[:, :n])
        if env._final is not None:
            o["final"] = host(env._final[:, :n])
    return o


def check_reward(got, ref, fam):
    want = ref.reward_out
    if fam in ("dyadic", "large"):
        assert (got.astype(np.float64) == want).all(), np.argwhere(got.astype(np.float64) != want)[:5]
        return
    bound = (ref.C + 2) * 2.0 ** -24 * ref.reward_abs
    if fam == "log2":
        x = ref.reward_pre_log
        bound = (bound + 2.0 ** -24 * (1 + x)) / ((1 + x) * math.log(2)) + 4e-7 * np.abs(want) + 2.0 ** -24
    err = np.abs(got.astype(np.float64) - want)
    assert (err <= bound).all(), (err - bound).max()


def check_step(got, ref, fam):
    for k in ("state", "index", "t", "unsafe", "truncated", "count"):
        assert (got[k] == getattr(ref, k)).all(), k
    if "se_row" in got:
        assert (got["se_row"] == ref.se_row).all(), "se_row"
    if "final" in got:
        assert (got["final"] == ref.final_state).all(), "final_state"
    check_reward(got["reward"], ref, fam)


def check_stats(env, ref, q24, fam):
    s = host(env._stats)
    assert (s[:4] == ref.stats[:4]).all(), (s[:4], ref.stats[:4])
    assert s[4] == q24, (int(s[4]), q24)
    if fam in ("dyadic", "large"):
        assert s[4] == ref.stats[4]


class Power:
    """What a batch must exercise for its comparisons to mean something."""

    def __init__(self, ref):
        self.ref, self.fired, self.drawn, self.unsafe, self.counts, self.trunc = ref, 0, 0, set(), set(), 0
        self.big = 0.0

    def add(self, ref):
        self.fired += int(ref.last_fire.sum())
        self.drawn += int(ref.last_draws.sum())
        self.unsafe |= set(np.unique(ref.unsafe).tolist())
        self.counts |= set(np.unique(ref.count).tolist())
        self.trunc += int(ref.truncated.sum())
        self.big = max(self.big, float(np.abs(ref.reward_out).max()))

    def check(self, fam=None):
        ref = self.ref
        if ref.noise and not ref.replay:
            p = ref.noise_prob
            assert self.drawn > 100
            assert abs(self.fired / self.drawn - p) < 6 * math.sqrt(p * (1 - p) / self.drawn)
        elif ref.noise:
            assert 0 < self.fired < self.drawn
        assert self.unsafe == {0, 1}
        assert self.trunc > 0 and ref.init.any()
        assert len(self.counts) >= 2
        if fam == "large":
            assert self.big >= 32


def drive_steps(env, ref, fam, rng, radix=None, replay=False, steps=K):
    power, q = Power(ref), 0
    for _ in range(steps):
        a = actions(rng, ref, radix)
        ru = rng.random((ref.n, ref.C)) if replay else None
        ref.step(a, ru)
        power.add(ref)
        if replay:
            env.step_device(dev(a), replay_u=ru)
        else:
            env.step_device(dev(a))
        got = gpu_out(env)
        check_step(got, ref, fam)
        q += TR.q24(got["reward"])
    check_stats(env, ref, q, fam)
    power.check(fam)
    return got


# ---------------------------------------------------------------------------------------------
# the step kernels

SA4 = [(2, 4), (4, 2), (3, 3), (4, 4)]
PAIR_FAM = {5: "uniform", 9: "log2", 16: "large"}
PAIR_ROWS = [dict(path="pair", C=C, S=SA4[i % 4][0], A=SA4[i % 4][1], noise=i % 2 == 1, epi=i % 3 != 0,
                  fam=PAIR_FAM.get(C, "dyadic"), extras=i % 2 == 0, n=20011 if C == 12 else N,
                  off=BIG if i % 3 == 2 else 4 * i) for i, C in enumerate([1, 2, 3, 4, 5, 7, 8, 9, 12, 16])]
PAIR_ROWS.append(dict(path="pair", C=16, S=4, A=4, noise=True, epi=True, fam="dyadic", extras=True, n=N, off=BIG))
PAIR8_SA = {1: (8, 8), 2: (6, 2), 3: (5, 3), 6: (6, 2), 10: (8, 8), 13: (5, 3), 16: (3, 7)}
PAIR8_FAM = {6: "uniform", 13: "log2", 16: "large"}
PAIR8_ROWS = [dict(path="pair8", C=C, S=PAIR8_SA[C][0], A=PAIR8_SA[C][1], noise=i % 2 == 0, epi=i % 3 != 1,
                   fam=PAIR8_FAM.get(C, "dyadic"), extras=i % 2 == 1, n=N, off=BIG if i % 3 == 0 else 0)
              for i, C in enumerate([1, 2, 3, 6, 10, 13, 16])]
GENERIC_ROWS = [
    dict(path="generic", C=4, S=4, A=4, noise=True, epi=True, fam="dyadic", se_mode="generic"),
    dict(path="generic", C=9, S=3, A=3, noise=False, epi=False, fam="uniform", se_mode="generic", off=BIG),
    dict(path="generic", C=16, S=4, A=4, noise=True, epi=False, fam="large", se_mode="generic"),
    dict(path="generic", C=16, S=3, A=2, noise=True, epi=True, fam="log2", se_mode="generic", n=20011),
    dict(path="generic", C=5, S=8, A=8, noise=True, epi=True, fam="dyadic", se_mode="generic"),
    dict(path="generic", C=10, S=8, A=5, noise=False, epi=True, fam="large", se_mode="generic", off=BIG),
    dict(path="generic", C=6, S=4, A=4, noise=True, epi=True, fam="dyadic", radix=[2, 4, 3, 4, 2, 3]),
    dict(path="generic", C=11, S=5, A=5, noise=True, epi=False, fam="large", radix=[5, 2, 3, 5, 4, 2, 5, 3, 2, 4, 5]),
    dict(path="generic", C=7, S=4, A=4, noise=True, epi=False, fam="dyadic", force=True),
    dict(path="generic", C=16, S=4, A=4, noise=False, epi=True, fam="large", force=True),
    dict(path="generic", C=5, S=3, A=3, noise=True, epi=True, fam="dyadic", se_mode="generic", replay=True),
    dict(path="pair", C=3, S=4, A=4, noise=True, epi=True, fam="uniform", replay=True),
    dict(path="pair", C=12, S=4, A=2, noise=True, epi=False, fam="dyadic", replay=True),
]


def _row_id(r):
    bits = [r["path"], f"C{r['C']}", f"S{r['S']}A{r['A']}", f"p{P}" if r["noise"] else "det",
            "epi" if r["epi"] else "glob", r["fam"]]
    for k in ("se_mode", "radix", "force", "replay", "extras"):
        if r.get(k):
            bits.append({"se_mode": "se_differs", "radix": "ragged", "force": "forced", "replay": "replay",
                         "extras": "se_final"}[k])
    if r.get("n", N) != N:
        bits.append(f"n{r['n']}")
    if r.get("off", 0) >= 1 << 32:
        bits.append("off2^32")
    return "-".join(bits)


def _row_seed(r):
    return zlib.crc32(_row_id(r).encode())


def _row_tables(r):
    return make_tables(_row_seed(r), r["C"], r["S"], r["A"], noise=r["noise"], fam=r["fam"], se_mode=r.get("se_mode", "pair"),
                       radix=r.get("radix"))


STEP_ROWS = PAIR_ROWS + PAIR8_ROWS + GENERIC_ROWS


@pytest.mark.parametrize("r", STEP_ROWS, ids=[_row_id(r) for r in STEP_ROWS])
def test_step_kernels(B, r):
    tabs = _row_tables(r)
    assert derive_path(tabs, r.get("radix"), r.get("force", False)) == r["path"]
    ex = r.get("extras", False)
    env, ref = build(B, tabs, r["fam"], n=r.get("n", N), epi=r["epi"], off=r.get("off", 0), radix=r.get("radix"),
                     replay=r.get("replay", False), emit_side_effects=ex or r["path"] == "generic",
                     emit_final_obs=ex, force_generic_kernel=r.get("force", False))
    rng = np.random.default_rng(_row_seed(r))
    start(env, ref, rng, r.get("radix"))
    drive_steps(env, ref, r["fam"], rng, r.get("radix"), r.get("replay", False))


PACKED_ROWS = [r for r in PAIR_ROWS if r["C"] in (1, 3, 5, 8, 12, 16)]


@pytest.mark.parametrize("r", PACKED_ROWS, ids=[_row_id(r).replace("pair", "packed", 1) for r in PACKED_ROWS])
def test_packed_layout(B, r):
    """The pair tables in the packed layout: equal to the reference, and to the int8 layout bit for bit."""
    tabs = _row_tables(r)
    kw = dict(n=r["n"], epi=r["epi"], off=r["off"], emit_side_effects=True, emit_final_obs=True)
    pk, ref = build(B, tabs, r["fam"], packed=True, **kw)
    i8, _ = build(B, tabs, r["fam"], **kw)
    rng = np.random.default_rng(r["C"])
    start(pk, ref, rng)
    i8.set_state(dev(ref.state), t=dev(ref.t))
    _lib().check(i8._lib.gc_set_global_step(i8._h, G0))
    from gym_cellular_b200.packed_env import pack_host
    power, q = Power(ref), 0
    for _ in range(K):
        a = actions(rng, ref)
        ref.step(a)
        power.add(ref)
        pk.step_device(dev(a))
        i8.step_device(dev(a))
        got, g8 = gpu_out(pk), gpu_out(i8)
        check_step(got, ref, r["fam"])
        q += TR.q24(got["reward"])
        assert (got["flags"] == (g8["unsafe"] | (g8["truncated"] << 1) | (g8["count"] << 2))).all()
        assert (got["se_words"] == pack_host(g8["se_row"])).all()
        assert (got["final_words"] == pack_host(g8["final"])).all()
        assert (got["reward"].view(np.uint32) == g8["reward"].view(np.uint32)).all()
        assert (got["index"] == g8["index"]).all() and (got["t"] == g8["t"]).all()
        if r["S"] == 4:
            assert (got["index"] == pack_host(got["state"])).all()
    check_stats(pk, ref, q, r["fam"])
    assert (host(pk._stats) == host(i8._stats)).all()
    power.check(r["fam"])


# ---------------------------------------------------------------------------------------------
# step_many: the fused many-step kernels

MANY_ROWS = [dict(C=3, S=3, A=3, noise=True, epi=True, fam="dyadic"),
             dict(C=8, S=4, A=4, noise=True, epi=False, fam="large", off=BIG),
             dict(C=5, S=2, A=4, noise=False, epi=True, fam="dyadic")]


@pytest.mark.parametrize("packed", [False, True], ids=["int8", "packed"])
@pytest.mark.parametrize("r", MANY_ROWS, ids=[f"C{r['C']}-S{r['S']}A{r['A']}-{r['fam']}" for r in MANY_ROWS])
def test_step_many_fused(B, monkeypatch, r, packed):
    """Seven steps over a ring of three action bindings in one launch: the last step and the statistics against the
    reference, and every output bit-identical with the separate launches (GC_B200_STEP_MANY_FUSED=0)."""
    import torch
    from gym_cellular_b200.packed_env import pack_host
    tabs = make_tables(r["C"] * 7 + r["S"], r["C"], r["S"], r["A"], noise=r["noise"], fam=r["fam"])
    assert derive_path(tabs) == "pair"
    steps, outs, stats = 7, [], []
    for fused in ("1", "0"):
        monkeypatch.setenv("GC_B200_STEP_MANY_FUSED", fused)
        env, ref = build(B, tabs, r["fam"], epi=r["epi"], off=r.get("off", 0), packed=packed, emit_side_effects=True)
        rng = np.random.default_rng(11)
        start(env, ref, rng)
        tape = [actions(rng, ref) for _ in range(3)]
        ring = []
        for a in tape:
            if packed:
                t = torch.zeros(env.ld, dtype=torch.int32, device="cuda")
                t[:ref.n] = dev(pack_host(a).view(np.int32))
            else:
                t = torch.zeros(ref.C, env.ld, dtype=torch.int8, device="cuda")
                t[:, :ref.n] = dev(a)
            ring.append(t)
        power = Power(ref)
        for k in range(steps):
            ref.step(tape[k % 3])
            power.add(ref)
        before = env.launch_count
        env.step_many([env._bind(t) for t in ring], steps)
        if fused == "1":
            assert env.launch_count - before == 1                 # the fused kernel ran
        got = gpu_out(env)
        check_step(got, ref, r["fam"])
        check_stats(env, ref, ref.stats[4], r["fam"])
        power.check(r["fam"])
        outs.append(got)
        stats.append(host(env._stats))
    for k in outs[0]:
        assert (np.ascontiguousarray(outs[0][k]).view(np.uint8) == np.ascontiguousarray(outs[1][k]).view(np.uint8)).all(), k
    assert (stats[0] == stats[1]).all()


# ---------------------------------------------------------------------------------------------
# rollout and collect

ROLL_ROWS = [dict(C=3, S=3, A=3, noise=True, epi=True, fam="dyadic", policies=("random", "table", "eps")),
             dict(C=8, S=4, A=2, noise=True, epi=False, fam="large", off=BIG, policies=("random", "table", "eps")),
             dict(C=16, S=4, A=4, noise=False, epi=True, fam="large", policies=("random",)),
             dict(C=5, S=2, A=3, noise=True, epi=False, fam="dyadic", policies=("random", "table", "eps"))]
ROLL_PARAMS = [pytest.param(r, pol, id=f"C{r['C']}-S{r['S']}A{r['A']}-{r['fam']}-{pol}")
               for r in ROLL_ROWS for pol in r["policies"]]


def _policy(pol, r):
    if pol == "random":
        return None, 0.0
    rng = np.random.default_rng(r["C"])
    table = rng.integers(0, r["A"] ** r["C"], r["S"] ** r["C"]).astype(np.int32)
    return table, (0.3 if pol == "eps" else 0.0)


@pytest.mark.parametrize("r,pol", ROLL_PARAMS)
def test_rollout_and_collect(B, r, pol):
    tabs = make_tables(r["C"] * 13 + r["A"], r["C"], r["S"], r["A"], noise=r["noise"], fam=r["fam"])
    assert derive_path(tabs) == "pair"
    policy, eps = _policy(pol, r)
    for drive in ("rollout", "collect"):
        if drive == "rollout" and eps:
            continue
        env, ref = build(B, tabs, r["fam"], epi=r["epi"], off=r.get("off", 0))
        rng = np.random.default_rng(3)
        start(env, ref, rng)
        power = Power(ref)
        rec = {k: [] for k in ("obs", "action", "reward", "flags", "next_obs")}
        ret, uns = np.zeros(ref.n), np.zeros(ref.n, np.int64)
        for _ in range(K):
            one = ref.collect(1, policy, eps)
            power.add(ref)
            for k in rec:
                rec[k].append(one[k])
            ret += ref.reward_out
            uns += ref.unsafe
        if drive == "rollout":
            g_ret, g_uns = env.rollout(K, policy)
            assert (host(g_ret).astype(np.float64) == ret).all()
            assert (host(g_uns) == uns).all()
        else:
            tr = env.collect(K, policy, eps, next_obs=True)
            for k in rec:
                want, got = np.concatenate(rec[k]), host(getattr(tr, k))
                if k == "reward":
                    assert (got.astype(np.float64) == want).all()
                else:
                    assert (got.view(want.dtype) == want).all(), k
        import torch
        assert (host(env.state) == ref.state).all() and (host(env.time_step) == ref.t).all()
        assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ref.index).all()
        check_stats(env, ref, ref.stats[4], r["fam"])
        power.check(r["fam"])


@pytest.mark.parametrize("kind", ["pair8", "generic"])
def test_rollout_and_collect_reject_other_tables(B, kind):
    C, S, A, mode = (3, 5, 3, "pair") if kind == "pair8" else (4, 4, 4, "generic")
    tabs = make_tables(99, C, S, A, noise=True, se_mode=mode)
    assert derive_path(tabs) == kind
    env, _ = build(B, tabs, "dyadic")
    for call in (lambda: env.rollout(2), lambda: env.collect(2)):
        with pytest.raises(_lib().GcError) as ei:
            call()
        assert ei.value.code == _lib().ERR_INVALID


# ---------------------------------------------------------------------------------------------
# host path

@pytest.mark.parametrize("packed", [False, True], ids=["int8", "packed"])
def test_host_path(B, packed):
    """step() with numpy arrays, in chunks of 1008 envs (which do not divide 4099)."""
    from gym_cellular_b200.packed_env import pack_host
    C, S, A, fam = (9, 4, 3, "dyadic") if not packed else (16, 4, 4, "large")
    tabs = make_tables(1234 + C, C, S, A, noise=True, fam=fam)
    env, ref = build(B, tabs, fam, epi=not packed, off=BIG if packed else 0, packed=packed, host_chunk_envs=1008)
    rng = np.random.default_rng(8)
    start(env, ref, rng)
    power, q = Power(ref), 0
    for _ in range(K):
        a = actions(rng, ref)
        ref.step(a)
        power.add(ref)
        if packed:
            obs, rew, term, trunc, info = env.step(pack_host(a))
            assert (obs == pack_host(ref.state)).all()
            f = info["flags"]
            got = dict(unsafe=f & 1, truncated=(f >> 1) & 1, count=f >> 2)
        else:
            obs, rew, term, trunc, info = env.step(a)
            assert (np.stack(obs) == ref.state).all()
            got = dict(unsafe=info["unsafe"].view(np.uint8), count=info["count"], truncated=trunc.view(np.uint8))
            assert (info["side_effects"] == ref.se_row).all()
        for k, v in got.items():
            assert (v == getattr(ref, k)).all(), k
        assert (info["tabular_state"] == ref.index).all() and (trunc == ref.truncated.astype(bool)).all()
        check_reward(np.array(rew), ref, fam)
        q += TR.q24(rew)
    check_stats(env, ref, q, fam)
    power.check(fam)


# ---------------------------------------------------------------------------------------------
# ragged index through set_state / state_dict, non-finite rewards

def test_ragged_index_through_set_state_and_state_dict(B):
    import torch
    radix = [2, 4, 3, 4, 2, 3]
    tabs = make_tables(77, 6, 4, 4, noise=True, radix=radix)
    env, ref = build(B, tabs, "dyadic", radix=radix)
    rng = np.random.default_rng(6)
    start(env, ref, rng, radix)                              # set_state: the ragged index at once
    assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ref.index).all()
    assert (host(env.tabularize(env.state)) == ref.index).all()
    assert (host(env.detabularize(torch.from_numpy(ref.index.astype(np.int64)).cuda())) == ref.state).all()
    sd = env.state_dict()
    saved = (ref.state.copy(), ref.t.copy())
    for _ in range(2):
        a = actions(rng, ref, radix)
        ref.step(a)
        env.step_device(dev(a))
    assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ref.index).all()
    env.load_state_dict(sd)
    ref.set_state(*saved)
    assert (host(env.tabular_state(torch.int32)).view(np.uint32) == ref.index).all()
    bad = ref.state.copy()
    bad[0, 5] = radix[0]                                     # below n_states, outside cell 0's levels
    with pytest.raises(ValueError):
        env.set_state(dev(bad))


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf"), 32.0, -32.0],
                         ids=["nan", "inf", "-inf", "at_bound", "at_-bound"])
@pytest.mark.parametrize("which", ["reward", "reward_noisy"])
def test_set_tables_rejects_bad_rewards(B, which, bad):
    """Non-finite rewards, and rewards whose step sum can reach 128 in magnitude (4 cells x 32: the reward statistic
    rounds each step to a 32-bit integer of 2^-24 units), are GC_ERR_INVALID; the previous tables stay in force."""
    tabs = make_tables(5, 4, 4, 4, noise=True)
    env, ref = build(B, tabs, "dyadic")
    L = _lib()
    arr = {k: np.ascontiguousarray(tabs[k], dt) for k, dt in (
        ("move", np.int8), ("noisy", np.int8), ("draws", np.uint8), ("reward", np.float32), ("side_effects", np.int8),
        ("counted", np.uint8), ("initial_state", np.int8), ("reward_noisy", np.float32))}
    arr[which] = arr[which].copy()
    arr[which][1, 2] = bad
    t = L.GcCellTables(*[arr[k].ctypes.data for k in ("move", "noisy", "draws", "reward", "side_effects", "counted",
                                                        "initial_state", "reward_noisy")], None)
    assert env._lib.gc_set_tables(env._h, C.byref(t)) == L.ERR_INVALID
    assert (b"finite" if math.isnan(bad) or math.isinf(bad) else b"128") in env._lib.gc_last_error()
    rng = np.random.default_rng(1)
    start(env, ref, rng)
    drive_steps(env, ref, "dyadic", rng)


def test_reward_bound_through_the_env(B):
    """The bound as a user meets it: n_cells x max|reward| must stay below 128, and under log2(1 + .) the smallest sum
    must stay above -1."""
    with pytest.raises(_lib().GcError) as ei:
        B.CellularVectorEnv(num_envs=16, n_cells=16, n_states=4, reward_func=np.full((4, 4), 10.0))
    assert ei.value.code == _lib().ERR_INVALID and "128" in ei.value.message
    B.CellularVectorEnv(num_envs=16, n_cells=16, n_states=4, reward_func=np.full((4, 4), 127 / 16))
    for lo, ok in ((-0.25, False), (-0.2, True)):           # 4 cells: 1 + 4 lo = 0 (log2 = -inf) or 0.2
        tabs = make_tables(9, 4, 4, 4, noise=False)
        tabs["reward"] = np.full((4, 4), lo)
        if ok:
            build(B, tabs, "log2")
        else:
            with pytest.raises(_lib().GcError) as ei:
                build(B, tabs, "log2")
            assert ei.value.code == _lib().ERR_INVALID
