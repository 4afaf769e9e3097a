"""ctypes/numpy front end of the C oracle (oracle/gc_oracle.c).  TEST INFRASTRUCTURE ONLY.

`OracleEnv` mirrors the device-side batch layout (cell-major structure of arrays) so that the
parity tests can hand the very same numpy arrays to the oracle and, as device copies, to the
CUDA path.  Nothing in gym_cellular_b200/ imports this module.
"""
import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libgc_oracle.so")

KIND_POLARISATION, KIND_GRIDWORLD = 0, 1
REWARD_IDS = {"right_polarizing": 0, "multiple_optima": 1, "nonlinear_mo": 2, "nonlinear_rp": 3,
              "table": 4, "table_log2": 5}
DIFFICULTIES = {"easy": 0, "hard": 1, "impossible": 2}
F_NOISE, F_DEADLOCK, F_RNG_EPISODIC, F_REPLAY = 1, 2, 4, 8
N_STATS = 8
STAT_STEPS, STAT_UNSAFE, STAT_COUNT, STAT_TRUNCATED, STAT_REWARD_Q24 = range(5)


class _Config(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_cells", C.c_int32), ("n_states", C.c_int32),
                ("n_actions", C.c_int32), ("reward_id", C.c_int32), ("difficulty", C.c_int32),
                ("flags", C.c_uint32), ("max_episode_steps", C.c_int32),
                ("noise_prob", C.c_double), ("dispersal_prob", C.c_double),
                ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
                ("reward_table", C.POINTER(C.c_double))]


# Where lib() compiles the oracle when the library in this directory is missing or older than its source;
# None = this directory.  bench.py points it at a temporary directory: it must run from a read-only tree.
build_dir = None


def _stale(path):
    return not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(os.path.join(_HERE, "gc_oracle.c"))


def build(force=False, out_dir=None):
    """Compile oracle/gc_oracle.c with gcc (Makefile in this directory) into `out_dir` (default: this
    directory); returns the library's path."""
    path = _LIB_PATH if out_dir is None else os.path.join(out_dir, "libgc_oracle.so")
    if force or _stale(path):
        subprocess.check_call(["make", "-s", "-C", _HERE, "OUT=" + path])
    return path


_lib = None


def lib():
    global _lib
    if _lib is None:
        path = build(out_dir=build_dir if _stale(_LIB_PATH) else None)
        L = C.CDLL(path)
        vp = C.c_void_p
        L.gco_step.restype = C.c_int64
        L.gco_step.argtypes = [C.POINTER(_Config), C.c_int64, C.c_int64] + [vp] * 11 + [C.c_int64, vp]
        L.gco_reset.restype = C.c_int
        L.gco_reset.argtypes = [C.POINTER(_Config), C.c_int64, C.c_int64, vp, vp, vp, vp]
        L.gco_initial_state.argtypes = [C.POINTER(_Config), vp]
        L.gco_n_slots.argtypes = [C.POINTER(_Config)]
        L.gco_policy_actions.argtypes = [C.POINTER(_Config), C.c_int64, C.c_int64, C.c_int, vp, vp, vp, C.c_int64, vp]
        L.gco_encode.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_int, vp, vp]
        L.gco_decode.argtypes = [C.c_int64, C.c_int64, C.c_int, C.c_int, vp, vp]
        L.gco_encode_one.restype = C.c_uint64
        L.gco_encode_one.argtypes = [vp, vp, vp, C.c_int]
        L.gco_decode_one.argtypes = [C.c_uint64, vp, vp, C.c_int, vp]
        L.gco_philox4x32_10.argtypes = [vp, vp, vp]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def philox4x32_10(ctr, key):
    c = np.asarray(ctr, np.uint32)
    k = np.asarray(key, np.uint32)
    out = np.zeros(4, np.uint32)
    lib().gco_philox4x32_10(_p(c), _p(k), _p(out))
    return out


def encode_mixed_radix(cells, mins, lens):
    cells, mins, lens = (np.ascontiguousarray(x, np.int64) for x in (cells, mins, lens))
    return int(lib().gco_encode_one(_p(cells), _p(mins), _p(lens), len(lens)))


def decode_mixed_radix(idx, mins, lens):
    mins, lens = (np.ascontiguousarray(x, np.int64) for x in (mins, lens))
    out = np.zeros(len(lens), np.int64)
    lib().gco_decode_one(int(idx), _p(mins), _p(lens), len(lens), _p(out))
    return out


def encode(cells, radix):
    cells = np.ascontiguousarray(cells, np.int8)
    n_cells, n = cells.shape
    out = np.zeros(n, np.uint32)
    lib().gco_encode(n, n, n_cells, radix, _p(cells), _p(out))
    return out


def decode(index, n_cells, radix):
    index = np.ascontiguousarray(index, np.uint32)
    out = np.zeros((n_cells, index.shape[0]), np.int8)
    lib().gco_decode(index.shape[0], index.shape[0], n_cells, radix, _p(index), _p(out))
    return out


class OracleEnv:
    """Batch of independent envs stepped by the C oracle.  Arrays are [C][n] (cell-major)."""

    def __init__(self, kind="polarisation", n_envs=1, n_cells=3, n_states=3, n_actions=None,
                 reward="right_polarizing", difficulty="easy", noise=False, deadlock=False,
                 rng_episodic=False, replay=False, max_episode_steps=0, noise_prob=0.1,
                 dispersal_prob=0.01, seed=0, env_id_offset=0, reward_table=None):
        self.cfg = _Config()
        if kind in ("gridworld", KIND_GRIDWORLD):
            self.cfg.kind, n_cells, n_states, n_actions = KIND_GRIDWORLD, 2, 20, 5
        else:
            self.cfg.kind = KIND_POLARISATION
        self.cfg.n_cells, self.cfg.n_states = n_cells, n_states
        self.cfg.n_actions = n_actions if n_actions is not None else n_states
        self._table = None
        if reward_table is not None:
            self._table = np.ascontiguousarray(reward_table, np.float64)
            assert self._table.shape == (n_states, self.cfg.n_actions)
            self.cfg.reward_table = self._table.ctypes.data_as(C.POINTER(C.c_double))
            if reward not in ("table", "table_log2"):
                reward = "table"
        self.cfg.reward_id = REWARD_IDS[reward]
        self.cfg.difficulty = DIFFICULTIES[difficulty]
        self.cfg.flags = ((F_NOISE if noise else 0) | (F_DEADLOCK if deadlock else 0) |
                          (F_RNG_EPISODIC if rng_episodic else 0) | (F_REPLAY if replay else 0))
        self.cfg.max_episode_steps = max_episode_steps
        self.cfg.noise_prob, self.cfg.dispersal_prob = noise_prob, dispersal_prob
        self.cfg.seed, self.cfg.env_id_offset = seed, env_id_offset
        self.n, self.C = int(n_envs), int(n_cells)
        self.n_slots = lib().gco_n_slots(C.byref(self.cfg))
        n = self.n
        self.state = np.zeros((self.C, n), np.int8)
        self.t = np.zeros(n, np.int32)
        self.reward = np.zeros(n, np.float64)
        self.index = np.zeros(n, np.uint32)
        self.terminated = np.zeros(n, np.uint8)
        self.truncated = np.zeros(n, np.uint8)
        self.unsafe = np.zeros(n, np.uint8)
        self.count = np.zeros(n, np.uint8)
        self.se_row = np.zeros((self.C, n), np.int8)
        self.stats = np.zeros(N_STATS, np.int64)
        self.global_step = 0
        self.reset()

    def initial_state(self):
        out = np.zeros(self.C, np.int8)
        lib().gco_initial_state(C.byref(self.cfg), _p(out))
        return out

    def reset(self, mask=None):
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        lib().gco_reset(C.byref(self.cfg), self.n, self.n, _p(m), _p(self.state), _p(self.t), _p(self.index))
        return self.state

    def step(self, actions, replay_u=None, lo=0, hi=None):
        """Step envs [lo, hi) (default all).  `actions` is int8 [C][n]."""
        actions = np.ascontiguousarray(actions, np.int8)
        assert actions.shape == (self.C, self.n)
        if self.cfg.flags & F_REPLAY:
            replay_u = np.ascontiguousarray(replay_u, np.float64)
            assert replay_u.shape == (self.n, self.n_slots)
        hi = self.n if hi is None else hi
        off = lo

        def sl(a):
            return None if a is None else C.c_void_p(a.ctypes.data + off * a.itemsize)
        cfg = self.cfg
        if lo:
            cfg = _Config.from_buffer_copy(self.cfg)
            cfg.env_id_offset = self.cfg.env_id_offset + lo
        ru = None if replay_u is None else C.c_void_p(replay_u.ctypes.data + off * self.n_slots * 8)
        rc = lib().gco_step(C.byref(cfg), hi - lo, self.n, sl(actions), sl(self.state), sl(self.t),
                            sl(self.reward), sl(self.index), sl(self.terminated), sl(self.truncated),
                            sl(self.unsafe), sl(self.count), sl(self.se_row), ru, self.global_step,
                            _p(self.stats))
        if rc < 0:
            raise KeyError("position")      # the reference's error for a grid-world action (4, 4)
        if lo == 0 and hi == self.n:
            self.global_step += 1
        return self.state, self.reward, self.terminated, self.truncated

    def policy_actions(self, policy=None):
        """Actions the fused rollout kernel generates for the current step (random or tabular policy)."""
        a = np.zeros((self.C, self.n), np.int8)
        pol = None if policy is None else np.ascontiguousarray(policy, np.int32)
        lib().gco_policy_actions(C.byref(self.cfg), self.n, self.n, 0 if pol is None else 1, _p(pol),
                                 _p(self.state), _p(self.t), self.global_step, _p(a))
        return a

    def rollout(self, n_steps, policy=None):
        """n_steps x (policy_actions -> step); returns (sum of rewards, unsafe steps) per env."""
        ret = np.zeros(self.n, np.float64)
        uns = np.zeros(self.n, np.int64)
        for _ in range(n_steps):
            self.step(self.policy_actions(policy))
            ret += self.reward
            uns += self.unsafe
        return ret, uns

    def step_parallel(self, actions, n_threads):
        """All-core stepping for the CPU baseline: ctypes releases the GIL inside gco_step."""
        bounds = np.linspace(0, self.n, n_threads + 1).astype(np.int64)
        actions = np.ascontiguousarray(actions, np.int8)
        threads = []
        for i in range(n_threads):
            def work(lo=int(bounds[i]), hi=int(bounds[i + 1])):
                if hi > lo:
                    self._step_range(actions, lo, hi)
            th = threading.Thread(target=work)
            threads.append(th)
            th.start()
        for th in threads:
            th.join()
        self.global_step += 1
        return self.state, self.reward, self.terminated, self.truncated

    def _step_range(self, actions, lo, hi):
        cfg = _Config.from_buffer_copy(self.cfg)
        if self._table is not None:
            cfg.reward_table = self._table.ctypes.data_as(C.POINTER(C.c_double))
        cfg.env_id_offset = self.cfg.env_id_offset + lo

        def sl(a):
            return C.c_void_p(a.ctypes.data + lo * a.itemsize)
        lib().gco_step(C.byref(cfg), hi - lo, self.n, sl(actions), sl(self.state), sl(self.t),
                       sl(self.reward), sl(self.index), sl(self.terminated), sl(self.truncated),
                       sl(self.unsafe), sl(self.count), None, None, self.global_step, None)
