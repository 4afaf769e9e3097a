"""Sequence tests: seeded random programs of calls on ONE handle, against a reference model stepped alongside.

Every other GPU test builds a fresh handle and calls one entry point.  Real callers interleave them: collect, step,
checkpoint, reset some envs, step from the host, run `step_many` on a ring of bindings.  All of these share handle state
that no single-entry test reaches:
  * the device global step (RNG counter of non-episodic envs, exploration key of collect), advanced by whole-shard
    kernels, ticked after the last chunk of a chunked or host pass, advanced by n inside fused launches and by graph
    replays, overwritten by `gc_set_global_step`, and its host mirror; programs cross its 32-bit wrap inside one launch
    and between launches;
  * bindings and cached `gc_step_many` graphs across `gc_set_tables` and `gc_set_final_obs`;
  * a fused `step_many` longer than one launch (4096 steps), whose later launches start the ring mid-way;
  * refused calls, which must leave state, t, statistics, the global step and the launch count untouched.

The model is `tests/_table_reference.TableEnv` (cellular, dyadic rewards: compared bit for bit) or the C oracle plus
`tests/_collect_oracle.collect` (grid world).  Operations are enqueued without a host synchronisation between them,
except where one synchronises by contract (host path, `state_dict`, table swap, global-step writes, graph capture);
each clones its outputs on the stream, and everything is compared after one synchronisation at the end.  The host
mirror of the global step and the launch count are checked after every operation against what the dispatch rules
predict.  After a torch graph capture the mirror is compared modulo 2^32: replays advance only the device word, and
`gc_sync_global_step` keeps the mirror's high word."""
import ctypes as C
import zlib

import numpy as np
import pytest

import _collect_oracle as CO
import _table_reference as TR
from test_gpu_counts import assert_counts, hist
from test_gpu_tables import SEED, Power, check_stats, check_step, f32_tables, gpu_out, make_tables

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

WRAP = 1 << 32
FUSED_MAX = 4096                 # kManyFusedMaxSteps: steps per fused launch
GRAPH_MAX_ENVS = 1 << 21         # kManyGraphMaxEnvs: larger shards take plain launches
MANY_MAX_CELLS = 8               # GC_MANY_MAX_CELLS
GRID_SEED = 0x5EED

ROWS = {
    # the counter protocol on every path, the wrap, final-obs toggling, pair <-> pair table swaps
    "a": dict(C=3, S=3, A=3, p=0.3, epi=False, limit=5, n=4099, final=True, swap="pair"),
    # p >= 1/2 on more than 4 cells: the wide draws' 16-bit-half compare; swaps to differing side-effect tables and back
    "b": dict(C=5, S=4, A=2, p=0.6, epi=False, limit=6, n=4099, swap="generic"),
    # packed bindings across a swap to tables the packed layout does not admit, and back
    "c": dict(C=6, S=4, A=4, p=0.3, epi=False, limit=7, n=4099, final=True, swap="generic", packed=True),
    # fused and graph step_many over more than 4096 steps; epsilon-collect across the wrap (exploration keys on G)
    "d": dict(C=8, S=4, A=4, p=None, epi=True, limit=9, n=517, swap="pair", long=True),
    # grid world against the C oracle
    "e": dict(grid=True, p=0.1, epi=False, limit=7, n=20011),
    # above kManyGraphMaxEnvs: plain step_many launches, the host path over several streams
    "g": dict(C=3, S=3, A=3, p=0.3, epi=False, limit=5, n=(1 << 21) + 19, big=True),
}


def _lib():
    from gym_cellular_b200 import _lib as lib
    return lib


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class _Ref(TR.TableEnv):
    """The table reference, feeding each step to the program's `Power`."""
    power = None

    def step(self, actions, replay_u=None):
        super().step(actions, replay_u)
        if self.power is not None:
            self.power.add(self)
        return self


def _grid_oracle():
    from oracle import oracle as O

    class Grid(O.OracleEnv):
        """The oracle, recording what its steps exercised: truncations and counts."""
        seen = None

        def step(self, actions, replay_u=None, lo=0, hi=None):
            out = super().step(actions, replay_u, lo, hi)
            self.seen["count"] |= set(np.unique(self.count).tolist())
            self.seen["trunc"] += int(self.truncated.sum())
            return out
    return Grid


class _Snap:
    """Clones, queued on the current stream, of every buffer `gpu_out` reads from an env."""

    def __init__(self, env):
        self.num_envs, self.n_cells = env.num_envs, env.n_cells
        self.state = env.state.clone()
        self._index = env.tabular_state(torch.int32).clone()
        self.time_step = env.time_step.clone()
        for k in ("_reward", "_flags", "_unsafe", "_truncated", "_count", "_se_row", "_final", "_stats"):
            if hasattr(env, k):
                v = getattr(env, k)
                setattr(self, k, None if v is None else v.clone())

    def tabular_state(self, dtype):
        return self._index


class Refused(Exception):
    pass


class Program:
    """One handle, its reference model and a log of (operation, device clones, expected values)."""

    def __init__(self, B, row, seed, monkeypatch):
        self.B, self.row, self.seed, self.mp = B, row, seed, monkeypatch
        self.grid, self.packed = row.get("grid", False), row.get("packed", False)
        self.n, self.limit = row["n"], row["limit"]
        self.rng = np.random.default_rng(seed)
        self.log, self.snapshots = [], []
        self.final_on = row.get("final", False)
        self.loose = False                         # mirror compared modulo 2^32 (after a graph capture)
        n = self.n
        if self.grid:
            self.C, self.S, self.A = 2, 20, 5
            self.env = B.CellularVectorEnv(kind="gridworld", num_envs=n, env_seed=GRID_SEED, max_episode_steps=self.limit,
                                           dispersal_prob=row["p"], rng_episodic=False)
            self.m = _grid_oracle()(kind="gridworld", n_envs=n, seed=GRID_SEED, max_episode_steps=self.limit,
                                    dispersal_prob=row["p"])
            self.m.seen = dict(count=set(), trunc=0)
            self.fast = True
        else:
            self.C, self.S, self.A = row["C"], row["S"], row["A"]
            base = zlib.crc32(repr(sorted(row.items())).encode()) ^ seed
            self.tabs = self._tables(base, "pair")
            self.alt = self._tables(base + 1, row.get("swap", "pair"))
            cls = B.PackedCellularVectorEnv if self.packed else B.CellularVectorEnv
            kw = dict(emit_side_effects=True) if self.packed else {}
            self.env = cls(num_envs=n, cell_tables=self.tabs, env_seed=SEED, rng_episodic=row["epi"],
                           max_episode_steps=self.limit, emit_final_obs=self.final_on, **kw)
            self.m = self._ref(self.tabs)
            self.power = Power(self.m)
            self.m.power = self.power
            self.fast = True
        self.toggle_final = self.final_on and not self.packed     # gc_set_final_obs is an int8-layout output
        self.graphs = []
        self.last = self._reset_outputs()
        # the binding ring first (up to 5 of the 16 slots), then two action tensors step_device binds on first use
        self.ring_actions = [self.actions() for _ in range(int(self.rng.choice([3, 5]) if row.get("long") else
                                                               self.rng.integers(2, 6)))]
        self.ring = [self.env._bind(self.action_tensor(a)) for a in self.ring_actions]
        self.orders = [list(range(len(self.ring))), list(self.rng.permutation(len(self.ring)))]
        self.cached = [(a, self.action_tensor(a)) for a in (self.actions(), self.actions())]

    # ---- reference -------------------------------------------------------------------------------
    def _tables(self, seed, mode):
        t = make_tables(seed, self.C, self.S, self.A, noise=self.row["p"] is not None, se_mode=mode)
        t["noise_prob"] = self.row["p"] if self.row["p"] is not None else 0.3
        return t

    def _ref(self, tabs):
        return _Ref(f32_tables(tabs), self.n, seed=SEED, rng_episodic=self.row["epi"], max_episode_steps=self.limit)

    def actions(self):
        n = self.n
        if self.grid:
            g = np.full((2, n), 4, np.int8)
            g[self.rng.integers(0, 2, n), np.arange(n)] = self.rng.integers(0, 4, n)
            return g
        return self.rng.integers(0, self.A, (self.C, n)).astype(np.int8)

    def action_tensor(self, a):
        """The [C, ld] int8 (or [ld] packed word) tensor a binding takes."""
        from gym_cellular_b200.packed_env import pack_host
        if self.packed:
            t = torch.zeros(self.env.ld, dtype=torch.int32, device="cuda")
            t[:self.n] = dev(pack_host(a).view(np.int32))
        else:
            t = torch.zeros(self.C, self.env.ld, dtype=torch.int8, device="cuda")
            t[:, :self.n] = dev(a)
        return t

    def policy(self, kind):
        if kind == "random":
            return None, 0.0
        hi = 24 if self.grid else self.A ** self.C            # grid world: never the invalid joint action (4, 4)
        table = self.rng.integers(0, hi, self.S ** self.C).astype(np.int32)
        return table, {"table": 0.0, "eps0.3": 0.3, "eps1": 1.0}[kind]

    def _reset_outputs(self):
        m, n = self.m, self.n
        if self.grid:
            se = np.full((self.C, n), 1, np.int8)                # the grid world's reset info: every entry 'safe'
        else:
            se = np.repeat(np.asarray(self.tabs["reset_row"], np.int8)[:, None], n, 1)
        z = np.zeros(n, np.uint8)
        return dict(unsafe=z, truncated=z, count=z, reward=np.zeros(n), se_row=se, final=m.state.copy())

    def _step_outputs(self):
        m = self.m
        out = dict(unsafe=m.unsafe.copy(), truncated=m.truncated.copy(), count=m.count.copy(), se_row=m.se_row.copy(),
                   reward=(m.reward if self.grid else m.reward_out).copy(), final=self.last["final"])
        if self.final_on:
            out["final"] = m.final_state.copy()
        return out

    def ref_step(self, a):
        self.m.step(a)
        self.last = self._step_outputs()

    def encode(self, cells):
        if self.grid:
            return (cells[0].astype(np.uint32) + 20 * cells[1].astype(np.uint32)).astype(np.uint32)
        return self.m.encode(cells)

    @property
    def G(self):
        return self.m.global_step

    @G.setter
    def G(self, v):
        self.m.global_step = v

    def fused(self, n_steps, fused_env):
        """Whether gc_step_many runs the whole call in fused launches (many_fusable)."""
        if not fused_env or n_steps < 2 or self.n > GRAPH_MAX_ENVS:
            return False
        if self.grid:
            return True
        if not self.fast or self.C > MANY_MAX_CELLS:
            return False
        return not self.final_on        # packed: the final-word buffer is part of every packed binding

    # ---- the operations --------------------------------------------------------------------------
    def op_step(self, cached=False):
        a, t = self.cached[int(self.rng.integers(2))] if cached else (self.actions(), None)
        if self.packed and not self.fast:
            raise Refused(lambda: self.env.step_device(t if cached else dev(a)))
        self.env.step_device(t if cached else dev(a))
        self.ref_step(a)
        return dict(launches=1, steps=1)

    def op_chunked(self):
        from gym_cellular_b200.packed_env import pack_host
        env, n = self.env, self.n
        cuts = np.sort(self.rng.choice(np.arange(1, (n - 1) // 16 + 1), int(self.rng.integers(1, 4)), replace=False)) * 16
        bounds = [0, *cuts.tolist(), n]
        a = self.actions()
        if self.packed:
            env._actions[:n].copy_(dev(pack_host(a).view(np.int32)))
        else:
            env._actions[:, :n].copy_(dev(a))
        L = _lib()

        def run():
            for b, e in zip(bounds[:-1], bounds[1:]):
                if self.packed:
                    L.check(env._lib.gc_step_packed(env._h, b, e - b, _ptr(env._actions), _ptr(env._state), _ptr(env._t),
                                                    _ptr(env._reward), env._index_ptr(), _ptr(env._flags), _ptr(env._final),
                                                    _ptr(env._se_row), _ptr(env._stats), env._stream()))
                else:
                    L.check(env._lib.gc_step(env._h, b, e - b, _ptr(env._actions), _ptr(env._state), _ptr(env._t),
                                             _ptr(env._reward), _ptr(env._index), _ptr(env._terminated),
                                             _ptr(env._truncated), _ptr(env._unsafe), _ptr(env._count), _ptr(env._se_row),
                                             None, _ptr(env._stats), env._stream()))
        if self.packed and not self.fast:
            raise Refused(run)
        run()
        self.ref_step(a)
        return dict(launches=len(bounds) - 1, steps=1, note=f"bounds {bounds}")

    def _bound_call(self, slot):
        L = _lib()
        return lambda: L.check(self.env._lib.gc_step_bound(self.env._h, self.ring[slot], self.env._stream()))

    def op_bound(self):
        i = int(self.rng.integers(len(self.ring)))
        if self.packed and not self.fast:
            raise Refused(self._bound_call(i))
        self._bound_call(i)()
        self.ref_step(self.ring_actions[i])
        return dict(launches=1, steps=1, note=f"slot {i}")

    def op_many(self, n_steps, fused_env, order):
        order = self.orders[order]
        self.mp.setenv("GC_B200_STEP_MANY_FUSED", "1" if fused_env else "0")
        call = lambda: self.env.step_many([self.ring[i] for i in order], n_steps)    # noqa: E731
        if self.packed and not self.fast:
            raise Refused(call)
        fused = self.fused(n_steps, fused_env)
        call()
        for k in range(n_steps):
            self.ref_step(self.ring_actions[order[k % len(order)]])
        launches = -(-n_steps // FUSED_MAX) if fused else n_steps
        return dict(launches=launches, steps=n_steps, note=f"order {order} fused={fused}")

    def op_many_restore(self, n_steps):
        """A long step_many and, right behind it while its kernels still run, `load_state_dict` of an earlier
        snapshot; the model steps only after both are enqueued."""
        self.mp.setenv("GC_B200_STEP_MANY_FUSED", "1")
        fused = self.fused(n_steps, True)
        sd, mine = self.snapshots[-1]
        self.env.step_many([self.ring[i] for i in self.orders[0]], n_steps)
        self.env.load_state_dict(sd)
        for k in range(n_steps):
            self.ref_step(self.ring_actions[k % len(self.ring)])
        self._restore_model(mine)
        return dict(launches=-(-n_steps // FUSED_MAX) if fused else n_steps, note=f"fused={fused}")

    def op_host(self):
        from gym_cellular_b200.packed_env import pack_host
        env, n = self.env, self.n
        a = self.actions()
        if self.packed:                  # final / side-effect words: the device path, copied out
            if not self.fast:
                raise Refused(lambda: env.step(pack_host(a)))
            obs, rew, _, trunc, info = env.step(pack_host(a))
            self.ref_step(a)
            assert (obs == pack_host(self.m.state)).all() and (info["flags"] == (
                self.m.unsafe | (self.m.truncated << 1) | (self.m.count << 2))).all()
            assert (rew.astype(np.float64) == self.m.reward_out).all()
            return dict(launches=1, steps=1)
        chunk = int(self.rng.integers(n // 6, n // 4)) | 1                 # odd: never a multiple of 16
        env.host_chunk_envs = chunk
        obs, rew, _, trunc, info = env.step(a)
        self.ref_step(a)
        m = self.m
        assert (np.stack(obs) == m.state).all() and (info["tabular_state"] == m.index).all()
        assert (info["unsafe"].view(np.uint8) == m.unsafe).all() and (info["count"] == m.count).all()
        assert (trunc.view(np.uint8) == m.truncated).all() and (info["side_effects"] == m.se_row).all()
        if self.grid:
            np.testing.assert_allclose(rew, m.reward, rtol=1e-6, atol=1e-7)
        else:
            assert (rew.astype(np.float64) == m.reward_out).all()
        per = (chunk + 15) // 16 * 16
        return dict(launches=-(-n // per), steps=1, note=f"chunk {chunk}")

    def _check_fast_call(self, call):
        if not self.fast:
            raise Refused(call)
        return call()

    def op_rollout(self, K, pol):
        policy, _ = self.policy(pol)
        got = self._check_fast_call(lambda: self.env.rollout(K, policy))
        got = tuple(g.clone() for g in got)
        if self.grid:
            ret, uns = self.m.rollout(K, policy)
        else:
            rec = self.m.collect(K, policy)
            ret, uns = rec["reward"].sum(0), (rec["flags"] & 1).astype(np.int64).sum(0)
        return dict(launches=1, steps=K, rollout=(got, ret, uns))

    def _record(self, K, policy, eps):
        if self.grid:
            obs, act, rew, flags = CO.collect(self.m, K, policy, eps)
            return dict(obs=obs, action=act, reward=rew, flags=flags, next_obs=obs)
        return self.m.collect(K, policy, eps)

    def op_collect(self, K, pol):
        policy, eps = self.policy(pol)
        tr = self._check_fast_call(lambda: self.env.collect(K, policy, eps, next_obs=not self.grid))
        got = {k: getattr(tr, k).clone() for k in ("obs", "action", "reward", "flags") + (() if self.grid else ("next_obs",))}
        return dict(launches=1, steps=K, collect=(got, self._record(K, policy, eps)))

    def op_counts(self, K, pol):
        policy, eps = self.policy(pol)
        nS, nA = self.env._joint_sizes()
        joint, transitions = nS * nA <= 1 << 22, nS * nA * nS <= 1 << 22 and not self.grid
        counts = self.env.zero_counts(joint=joint, transitions=transitions)
        self._check_fast_call(lambda: self.env.collect_counts(K, policy, eps, counts))
        rec = self._record(K, policy, eps)
        want = hist(rec, nS, nA, None if self.grid else (self.C, self.S, self.A), joint, transitions)
        return dict(launches=1, steps=K, counts=(counts, want))

    def op_reset(self):
        if self.packed and not self.fast:
            raise Refused(self.env.reset)
        self.env.reset()
        self.m.reset()
        self.last = self._reset_outputs()
        return dict(launches=1)

    def op_reset_envs(self):
        mask = self.rng.random(self.n) < 0.3
        if self.packed and not self.fast:
            raise Refused(lambda: self.env.reset_envs(dev(mask)))
        self.env.reset_envs(dev(mask))
        m = self.m
        if self.grid:
            m.reset(mask.astype(np.uint8))
        else:                            # the masked reset, done by hand: initial state, t = 0, the index re-encoded
            m.state[:, mask] = m.init[:, None]
            m.t[mask] = 0
            m.index = m.encode(m.state)
        return dict(launches=1)

    def op_set_state(self):
        m, n = self.m, self.n
        t = self.rng.integers(0, self.limit, n).astype(np.int32)
        if self.grid:                    # valid grid states only: the current ones, shuffled over the envs
            cells = m.state[:, self.rng.permutation(n)].copy()
        else:
            cells = self.rng.integers(0, self.S, (self.C, n)).astype(np.int8)
        self.env.set_state(dev(cells), t=dev(t), validate=False)
        if self.grid:
            m.state[:], m.t[:], m.index[:] = cells, t, self.encode(cells)
        else:
            m.set_state(cells, t)
        return dict(launches=0)

    def op_snapshot(self):
        sd = self.env.state_dict()
        m = self.m
        self.snapshots.append((sd, dict(state=m.state.copy(), t=m.t.copy(), stats=m.stats.copy(), G=self.G,
                                        loose=self.loose)))
        return dict(launches=0)

    def op_restore(self):
        if not self.snapshots:
            return self.op_snapshot()
        sd, mine = self.snapshots[int(self.rng.integers(len(self.snapshots)))]
        self.env.load_state_dict(sd)
        self._restore_model(mine)
        return dict(launches=0)

    def _restore_model(self, mine):
        m = self.m
        m.state[:], m.t[:], m.stats[:] = mine["state"], mine["t"], mine["stats"]
        m.index[:] = self.encode(m.state)
        self.G, self.loose = mine["G"], mine["loose"]

    def op_set_gstep(self, value):
        torch.cuda.current_stream().synchronize()          # ordered only after blocking streams (header)
        _lib().check(self.env._lib.gc_set_global_step(self.env._h, value))
        self.G, self.loose = value, False
        return dict(launches=0, note=f"G = {value:#x}")

    def op_final(self):
        self.final_on = not self.final_on
        ptr = _ptr(self.env._final) if self.final_on else None
        _lib().check(self.env._lib.gc_set_final_obs(self.env._h, ptr))
        return dict(launches=0, note=f"final {'on' if self.final_on else 'off'}")

    def op_swap(self, which):
        tabs = self.alt if which == "alt" else self.tabs
        arr = {k: None if tabs.get(k) is None else np.ascontiguousarray(tabs[k], dt) for k, dt in (
            ("move", np.int8), ("noisy", np.int8), ("draws", np.uint8), ("reward", np.float32), ("side_effects", np.int8),
            ("counted", np.uint8), ("initial_state", np.int8), ("reward_noisy", np.float32))}
        t = _lib().GcCellTables(*[None if arr[k] is None else arr[k].ctypes.data for k in (
            "move", "noisy", "draws", "reward", "side_effects", "counted", "initial_state", "reward_noisy")], None)
        torch.cuda.current_stream().synchronize()          # the header: steps in flight must be waited for
        _lib().check(self.env._lib.gc_set_tables(self.env._h, C.byref(t)))
        old, new = self.m, self._ref(tabs)
        new.state, new.t, new.index = old.state.copy(), old.t.copy(), old.index.copy()
        new.global_step, new.stats, new.power = old.global_step, old.stats.copy(), old.power
        self.m = new
        se = tabs["side_effects"]
        self.fast = all((se[j] == se[2]).all() for j in range(3, self.C))
        return dict(launches=0, note=f"tables {which} fast={self.fast}")

    def op_capture(self):
        if self.packed and not self.fast:                  # the capture would bind: refused as a bound step is
            return self.op_bound()
        acts = [self.actions() for _ in range(2)]
        ring = [self.action_tensor(a) for a in acts]
        reps = int(self.rng.integers(1, 4))
        graph = self.env.capture_steps(ring)
        for _ in range(reps):
            graph.replay()
            for a in acts:
                self.ref_step(a)
        self.env.sync_step_counter()
        self.graphs.append((graph, ring))              # the graph's kernels hold the ring's pointers
        self.loose = True
        return dict(launches=len(ring), note=f"{reps} replays")

    # ---- running -----------------------------------------------------------------------------------
    def run(self, ops):
        env = self.env
        L = _lib()
        for i, (name, kw) in enumerate(ops):
            where = f"seed {self.seed}, operation {i}: {name} {kw}"
            before = env.launch_count
            G0 = self.G
            try:
                info = getattr(self, "op_" + name)(**kw)
            except Refused as r:
                try:
                    r.args[0]()
                except L.GcError as e:
                    assert e.code == L.ERR_INVALID, f"{where}: {e}"
                else:
                    raise AssertionError(f"{where}: not refused under tables the call does not admit")
                info = dict(launches=0, note="refused")
            except AssertionError as e:
                raise AssertionError(f"{where}: {e}") from e
            got_l = env.launch_count - before
            assert got_l == info["launches"], f"{where}: {got_l} launches, expected {info['launches']} ({info.get('note')})"
            mirror = int(env._lib.gc_get_global_step(env._h))
            want = self.G
            if self.loose:
                assert (mirror - want) % WRAP == 0, f"{where}: mirror {mirror:#x}, model {want:#x} (mod 2^32)"
            else:
                assert mirror == want, f"{where}: mirror {mirror:#x}, model {want:#x} ({info.get('note')})"
            if not info.get("launches") and name not in ("restore", "set_gstep"):
                assert self.G == G0, where
            self.log.append((where, _Snap(env), self._expected(), info))
        synced = env.sync_step_counter()
        assert (synced - self.G) % WRAP == 0 and (self.loose or synced == self.G), (synced, self.G)
        torch.cuda.synchronize()
        for where, snap, want, info in self.log:
            try:
                self._compare(snap, want, info)
            except AssertionError as e:
                raise AssertionError(f"{where} ({info.get('note')}): {e}") from e
        self._check_power()

    def _expected(self):
        m = self.m
        return dict(state=m.state.copy(), index=m.index.copy(), t=m.t.copy(), stats=m.stats.copy(), C=self.C,
                    **self.last)

    def _compare(self, snap, want, info):
        from types import SimpleNamespace
        got = gpu_out(snap)
        ns = SimpleNamespace(**want)
        ns.reward_out, ns.final_state = want["reward"], want["final"]
        if self.grid:
            np.testing.assert_allclose(got["reward"], want["reward"], rtol=1e-6, atol=1e-7)
            ns.reward_out = got["reward"].astype(np.float64)
            s = snap._stats.cpu().numpy()
            assert (s[:4] == want["stats"][:4]).all(), (s[:4], want["stats"][:4])
            assert abs(int(s[4]) - int(want["stats"][4])) <= s[0]
        else:
            check_stats(snap, ns, want["stats"][4], "dyadic")
        check_step(got, ns, "dyadic")
        if "rollout" in info:
            (g_ret, g_uns), ret, uns = info["rollout"]
            g_ret, g_uns = g_ret.cpu().numpy(), g_uns.cpu().numpy()
            if self.grid:
                np.testing.assert_allclose(g_ret, ret, rtol=1e-5, atol=1e-5 * info["steps"])
            else:
                assert (g_ret.astype(np.float64) == ret).all(), "rollout return"
            assert (g_uns == uns).all(), "rollout unsafe steps"
        if "collect" in info:
            got_rec, rec = info["collect"]
            for k, v in got_rec.items():
                v = v[:, :self.n].cpu().numpy()
                if k == "reward":
                    if self.grid:
                        np.testing.assert_allclose(v, rec[k], rtol=1e-6, atol=1e-7)
                    else:
                        assert (v.astype(np.float64) == rec[k]).all(), "record reward"
                else:
                    assert (v.view(rec[k].dtype) == rec[k]).all(), f"record {k}"
        if "counts" in info:
            counts, want_c = info["counts"]
            if self.grid:                  # q24 of a float32 grid reward against the oracle's float64: within 1 a step
                g = counts.reward_q24.cpu().numpy()
                assert (np.abs(g - want_c["reward_q24"]) <= want_c["visits"]).all()
                counts = counts._replace(reward_q24=None)
                want_c = dict(want_c, reward_q24=None)
            assert_counts(counts, want_c)

    def _check_power(self):
        if self.grid:                    # grid world: 'unsafe' is overwritten by 'safe' (grid_world.py:174-175)
            s = self.m.seen
            assert s["trunc"] > 0 and len(s["count"]) >= 2, s
        else:
            self.power.check()


# ---------------------------------------------------------------------------------------------
# programs

def _n_steps_choices(prog):
    k = len(prog.ring)
    return [1, 2, 2 * k - 1, 37]


def _random_op(prog, rng, allow):
    names = [x for x in ("step", "step_cached", "chunked", "bound", "many", "host", "rollout", "collect", "counts",
                         "reset", "reset_envs", "set_state", "snapshot", "restore", "set_gstep", "final", "capture")
             if x in allow]
    name = names[int(rng.integers(len(names)))]
    pols = ["random", "table"] + ([] if name == "rollout" else ["eps0.3", "eps1"])
    if name in ("step", "step_cached"):
        return ("step", dict(cached=name == "step_cached"))
    if name == "many":
        return ("many", dict(n_steps=int(rng.choice(_n_steps_choices(prog))), fused_env=bool(rng.integers(2)),
                             order=int(rng.integers(2))))
    if name in ("rollout", "collect", "counts"):
        return (name, dict(K=int(rng.choice([1, 3, 7, 64])), pol=str(rng.choice(pols))))
    if name == "set_gstep":
        v = WRAP - int(rng.integers(1, 6)) if rng.random() < 0.5 else int(rng.integers(0, 1 << 34))
        return ("set_gstep", dict(value=v))
    if name == "swap":
        return ("swap", dict(which="alt"))
    return (name, {})


def build_program(prog, rng, n_ops=40, side_stream=False):
    """A backbone that places the operations every row must exercise, in order, with random operations between its
    units."""
    row = prog.row
    k = len(prog.ring)
    crossing = [("set_gstep", dict(value=WRAP - 2)), ("rollout", dict(K=7, pol="random"))]
    units = [
        [("many", dict(n_steps=37, fused_env=False, order=0))],                     # builds the cached graph
        crossing,                                                                   # the wrap inside one rollout
        [("set_gstep", dict(value=WRAP - 3)), ("collect", dict(K=7, pol="eps0.3"))],
        [("set_gstep", dict(value=WRAP - 1)), ("step", dict(cached=False)), ("bound", {}), ("chunked", {})],
        [("set_gstep", dict(value=WRAP - 4)), ("counts", dict(K=64, pol="eps1"))],
        [("set_gstep", dict(value=WRAP - 5)), ("many", dict(n_steps=37, fused_env=True, order=1))],
        [("snapshot", {})],
    ]
    if side_stream:                      # a restore right behind a step_many that is still running
        units.append([("many_restore", dict(n_steps=600 if not prog.packed else 300))])
    if row.get("long"):
        long = FUSED_MAX + k + 1
        units.append([("many", dict(n_steps=long, fused_env=True, order=1))])
        units.append([("many", dict(n_steps=long, fused_env=False, order=0))])
    if prog.toggle_final:
        units.append([("final", {}), ("bound", {}), ("many", dict(n_steps=2 * k - 1, fused_env=True, order=0)),
                      ("step", dict(cached=True))])
        units.append([("final", {}), ("bound", {}), ("step", dict(cached=True)), ("host", {})])
    if "swap" in row:
        units.append([("swap", dict(which="alt")), ("many", dict(n_steps=37, fused_env=False, order=0)), ("bound", {}),
                      ("step", dict(cached=True)), ("many", dict(n_steps=2 * k - 1, fused_env=True, order=1)),
                      ("rollout", dict(K=3, pol="table")), ("collect", dict(K=3, pol="random")), ("host", {}),
                      ("reset_envs", {}), ("chunked", {})])
        units.append([("swap", dict(which="orig")), ("bound", {}), ("many", dict(n_steps=37, fused_env=False, order=0))])
    units.append([("capture", {}), ("restore", {})])
    allow = {"step", "step_cached", "chunked", "bound", "many", "host", "rollout", "collect", "counts", "reset",
             "reset_envs", "set_state", "snapshot", "restore", "set_gstep", "capture"}
    if prog.toggle_final:
        allow.add("final")
    filler = max(0, n_ops - sum(len(u) for u in units))
    for _ in range(filler):
        op = _random_op(prog, rng, allow)
        if op[0] == "capture" and sum(1 for u in units for o in u if o[0] == "capture") >= 2:
            op = ("step", dict(cached=True))
        units.insert(int(rng.integers(1, len(units) + 1)), [op])
    return [op for u in units for op in u]


BIG_PROGRAM = [("step", dict(cached=False)), ("host", {}), ("many", dict(n_steps=3, fused_env=True, order=0)),
               ("chunked", {}), ("bound", {}), ("set_gstep", dict(value=WRAP - 2)),
               ("many", dict(n_steps=3, fused_env=False, order=1)), ("reset_envs", {}), ("snapshot", {}), ("host", {}),
               ("restore", {}), ("step", dict(cached=True))]


@pytest.fixture(scope="module")
def B():
    import gym_cellular_b200 as pkg
    assert torch.cuda.is_available()
    return pkg


def _run(B, monkeypatch, name, seed, side_stream=False):
    row = ROWS[name]
    prog = Program(B, row, seed, monkeypatch)
    if row.get("big"):
        ops = BIG_PROGRAM
    else:
        ops = build_program(prog, np.random.default_rng(seed + 1000), side_stream=side_stream)
    prog.run(ops)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("name", ["a", "b", "c", "d", "e"])
def test_sequence(B, monkeypatch, name, seed):
    _run(B, monkeypatch, name, seed)


@pytest.mark.parametrize("seed", [1, 2, 3])
@pytest.mark.parametrize("name", ["a", "c"])
def test_sequence_on_a_side_stream(B, monkeypatch, name, seed):
    """Rows a and c on a non-blocking stream: a `load_state_dict` right behind a long `step_many` must not lose the
    restored global step to the kernel still running."""
    with torch.cuda.stream(torch.cuda.Stream()):
        _run(B, monkeypatch, name, seed, side_stream=True)


def test_sequence_above_graph_limit(B, monkeypatch):
    _run(B, monkeypatch, "g", 1)
