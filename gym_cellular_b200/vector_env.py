"""`CellularVectorEnv`: a gymnasium.vector.VectorEnv whose step() launches the sm_100a kernels.

One instance holds `num_envs` independent copies of one environment of the gym-cellular family in
structure-of-arrays device tensors and steps all of them with one ctypes call into
libgymcellular_b200.so (include/gym_cellular_b200.h).  The reference surface it batches:
`Env.reset()` / `Env.step(action)` of gym_cellular/envs/cells3states3actions3.py:99-125,
cells2rest3.py:87-112, cells3resetVdeadlock.py:130-157 and grid_world.py:97-116, with the tabular
index of `prior_knowledge.tabularize` (cells3states3actions3.py:281-284) emitted alongside.

Two ways to drive it:
  * device path -- `step(actions)` with an int8 torch tensor [n_cells, num_envs] on the env's device
    (or anything exporting DLPack); everything stays in HBM and the returned observations are views
    of the env's own buffers (valid until the next step).
  * host path   -- `step(actions)` with numpy arrays: the C library copies the actions in, steps and
    copies observation / reward / flags back through pinned buffers, pipelined in chunks.

There is no CPU implementation behind this class: without the CUDA library or a CUDA device it raises.
"""
import ctypes as C
import weakref
from collections import namedtuple

import numpy as np
import torch

from . import _lib, tables
from ._gym import gym

_FAMILIES = {
    # id suffix: (kind, n_cells, n_states, n_actions, stochastic)
    "Cells3States3Actions3-v0": ("cellular", 3, 3, 3, False),
    "Cells2Rest3-v0": ("cellular", 2, 3, 3, False),
    "Cells3ResetVDeadlock-v0": ("cellular", 3, 3, 3, True),
    "GridWorld-v0": ("gridworld", 2, 20, 5, True),
}


class Transitions(namedtuple("Transitions", "obs action reward flags next_obs")):
    """Experience of `collect(K)`: [K, num_envs] device tensors, row k = step k.
    obs / action / next_obs are int32 tensors carrying the uint32 tabular indices (as `tabular_state(torch.int32)`);
    next_obs is the successor before the time-limit auto-reset (None unless requested); flags is the packed
    layout's flag byte (bit 0 unsafe, bit 1 truncated, bits 2-6 count), decoded by `unsafe`, `truncated`, `count`."""
    __slots__ = ()

    @property
    def unsafe(self):
        return (self.flags & _lib.FLAG_UNSAFE).ne(0)

    @property
    def truncated(self):
        return (self.flags & _lib.FLAG_TRUNCATED).ne(0)

    @property
    def count(self):
        return self.flags >> _lib.FLAG_COUNT_SHIFT


class Counts(namedtuple("Counts", "visits next reward_q24 unsafe cell_next")):
    """Experience counts of `collect_counts`: int64 device tensors the kernel adds to (None = not counted).
    s / a / s' are the tabular `obs`, executed `action` and `next_obs` of `collect` (nS = n_states ** n_cells,
    nA = n_actions ** n_cells; grid world 400 and 25).
      visits      [nS, nA]        N(s, a)
      next        [nS, nA, nS]    N(s, a, s'), s' = successor before the time-limit auto-reset
      reward_q24  [nS, nA]        sum of round(reward * 2**24), the term stats()['reward_sum'] is kept in
      unsafe      [nS, nA]        steps that reported 'unsafe'
      cell_next   [C, S, A, S]    per cell c: N_c(s_c, a_c, s'_c) (cellular family only)
    P_hat(s' | s, a) = next / visits and R_hat(s, a) = reward_q24 * 2**-24 / visits.
    Grouped counts (`zero_counts(groups=P)`) have a leading [P] on every table: `group(g)` is group g's Counts."""
    __slots__ = ()

    def group(self, g):
        """Counts of group g of grouped counts: views of row g of every table (None stays None)."""
        return Counts(*(None if t is None else t[g] for t in self))


_JOINT_LIMIT = 2 ** 31              # entries of one joint count table (32-bit indices in the kernels)


def _round_up(n, m):
    return (n + m - 1) // m * m


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _check_policy_stack(policy, policy_of_env, n_states_joint, num_envs, device):
    """Shapes, dtypes and device of a policy stack: `policy` [P, nS] of int tabular actions (P >= 1), `policy_of_env`
    an integer tensor [num_envs] on `device`.  Returns policy as a contiguous int32 tensor on `device`.  (The range of
    the map is checked on the device by the caller.)"""
    if policy is None:
        raise ValueError("policy_of_env needs a stack of policy tables: the random policy has no table to pick from")
    ptab = torch.as_tensor(policy, device=device)
    if ptab.dtype.is_floating_point or ptab.dtype.is_complex or ptab.dtype == torch.bool:
        raise ValueError(f"policy must hold integer tabular actions, not {ptab.dtype}")
    if ptab.dim() != 2 or ptab.shape[0] < 1 or ptab.shape[1] != n_states_joint:
        raise ValueError(f"with policy_of_env, policy must have shape [n_tables, {n_states_joint}] (n_tables >= 1); "
                         f"got {tuple(ptab.shape)}")
    if ptab.shape[0] >= 2 ** 31:
        raise ValueError("a policy stack holds fewer than 2**31 tables")
    m = policy_of_env
    if not isinstance(m, torch.Tensor):
        raise ValueError("policy_of_env must be a torch tensor on the env's device")
    if m.dtype not in (torch.int32, torch.int64, torch.int16, torch.int8, torch.uint8):
        raise ValueError(f"policy_of_env must be an integer tensor, not {m.dtype}")
    if m.device != torch.device(device):
        raise ValueError(f"policy_of_env lives on {m.device}, the env on {device}")
    if tuple(m.shape) != (num_envs,):
        raise ValueError(f"policy_of_env must have shape ({num_envs},); got {tuple(m.shape)}")
    return ptab.to(torch.int32).contiguous()


_TYPESTR = {torch.int8: "|i1", torch.uint8: "|u1", torch.int32: "<i4", torch.float32: "<f4"}


class _CompressibleBlock:
    """One gc_alloc_compressible allocation, seen by torch through __cuda_array_interface__.  A tensor made from it
    holds a reference to it, so the memory is freed (gc_free_compressible) when the last tensor and view is gone."""

    def __init__(self, lib, shape, dtype, device):
        self._lib, self._device = lib, device.index
        self.nbytes = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        stream = torch.cuda.current_stream(device).cuda_stream
        self.ptr = lib.gc_alloc_compressible(self.nbytes, self._device, stream)
        if not self.ptr:
            raise torch.cuda.OutOfMemoryError(f"gc_alloc_compressible could not allocate {self.nbytes} bytes")
        self.__cuda_array_interface__ = {"data": (self.ptr, False), "shape": tuple(shape), "typestr": _TYPESTR[dtype],
                                         "version": 2, "strides": None}

    def __del__(self):
        if getattr(self, "ptr", None):
            self._lib.gc_free_compressible(self.ptr, self.nbytes, self._device, None)     # synchronises the device
            self.ptr = None


class CellularVectorEnv(gym.vector.VectorEnv):
    """Batched polarisation / grid-world environment on one CUDA device.

    Parameters mirror the reference's `gymnasium.make` kwargs (`difficulty`, `reward_func`,
    `env_seed`, `deadlock`; cells3states3actions3.py:61-64,91-94, cells3resetVdeadlock.py:77-82,
    122-125) plus the batching ones.

    kind            'cellular' (polarisation family) or 'gridworld'
    num_envs        envs on THIS device
    n_cells/n_states/n_actions   cellular family shape (reference: 3/3/3 and 2/3/3; config 4: 16/4/4)
    stochastic      cellular: per-cell "reset" noise of Cells3ResetVDeadlock (p = noise_prob)
    deadlock        cellular + stochastic: polarised cells stay polarised
    rng_episodic    RNG counter = episode step, i.e. every episode replays the same noise, which is
                    what the reference's re-seeding reset() does (cells3resetVdeadlock.py:131)
    max_episode_steps   None/0 = never truncate (reference); > 0 = time limit with fused auto-reset
    emit_final_obs  also write the observation BEFORE a time-limit auto-reset: infos['final_obs'] (valid where
                    infos['_final_obs'], i.e. truncated) and infos['final_info'] -- gymnasium's SAME_STEP
                    convention; the reference itself never ends an episode (gym_cellular/__init__.py:7)
    compressible_buffers   the env-owned step buffers (state, time step, reward, index, flags) in generic
                    compressible memory, where L2 <-> DRAM transfers of low-entropy lines move fewer bytes
                    (config 4 on a B200: 178 against 192 us per step, profiles/r05_compression.md); results are
                    identical.  None = on where the device supports it and the step buffers exceed 1/16 of its
                    L2.  `compressible` tells what was granted
    env_id_offset   global id of env 0: Philox streams are keyed by global id, so a batch sharded
                    over ranks reproduces the single-device results env by env
    """

    metadata = {"render_modes": []}
    if hasattr(gym.vector, "AutoresetMode"):
        metadata["autoreset_mode"] = gym.vector.AutoresetMode.SAME_STEP

    def __init__(self, kind="cellular", num_envs=1, n_cells=3, n_states=3, n_actions=None,
                 difficulty="easy", reward_func=None, stochastic=False, deadlock=False,
                 noise_prob=0.1, dispersal_prob=0.01, env_seed=0, rng_episodic=None,
                 max_episode_steps=None, device=None, env_id_offset=0, emit_side_effects=True,
                 collect_stats=True, host_chunk_envs=1 << 20, cell_tables=None, force_generic_kernel=False,
                 emit_final_obs=False, cell_radix=None, compressible_buffers=None):
        self._lib = _lib.load()                      # raises ImportError when the .so is missing
        if not torch.cuda.is_available():
            raise RuntimeError("CellularVectorEnv needs a CUDA device: there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise ValueError("device must be a CUDA device")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.kind = kind
        self._cell_tables = cell_tables
        if cell_tables is not None:          # explicit table set (tables.debug_tables() etc.)
            n_cells, n_states, n_actions = (cell_tables[k] for k in ("n_cells", "n_states", "n_actions"))
            stochastic = cell_tables.get("draws") is not None
            noise_prob = cell_tables.get("noise_prob", noise_prob)
            reward_func = cell_tables["reward"] if reward_func is None else reward_func
        if kind == "gridworld":
            n_cells, n_states, n_actions, stochastic = 2, 20, 5, True
        elif kind != "cellular":
            raise ValueError("kind must be 'cellular' or 'gridworld'")
        self.num_envs = int(num_envs)
        self.n_cells, self.n_states = int(n_cells), int(n_states)
        self.n_actions = int(n_actions) if n_actions is not None else int(n_states)
        self.difficulty = difficulty
        self.stochastic, self.deadlock = bool(stochastic), bool(deadlock)
        if rng_episodic is None:
            rng_episodic = (kind == "cellular")      # the polarisation env re-seeds on reset, grid world never seeds
        self.rng_episodic = bool(rng_episodic)
        self.max_episode_steps = int(max_episode_steps or 0)
        self.env_seed = int(env_seed)
        self.env_id_offset = int(env_id_offset)
        self.emit_side_effects = bool(emit_side_effects)
        self.emit_final_obs = bool(emit_final_obs)
        # ragged state space: levels of each cell for the tabular index (the reference's codec takes one space
        # per cell, generalized_space_transformations.py:1-12); the moves must keep cell c below cell_radix[c]
        self.cell_radix = None if cell_radix is None else [int(r) for r in cell_radix]
        self.host_chunk_envs = int(host_chunk_envs)
        self.ld = _round_up(self.num_envs, 16)

        # --- handle -------------------------------------------------------------------------
        cfg = _lib.GcConfig()
        cfg.struct_size = C.sizeof(_lib.GcConfig)
        cfg.kind = _lib.KIND_CELLULAR if kind == "cellular" else _lib.KIND_GRIDWORLD
        cfg.device = self.device.index
        cfg.n_cells, cfg.n_states, cfg.n_actions = self.n_cells, self.n_states, self.n_actions
        cfg.max_episode_steps = self.max_episode_steps
        flags = 0
        self.reward_log2 = False
        if kind == "cellular":
            if reward_func is None:
                reward_func = tables.nonlinear_right_polarizing if stochastic else tables.right_polarizing
            if isinstance(reward_func, tables.CellReward):     # bind the shape: the host callable must agree with the device table
                reward_func = reward_func.for_shape(self.n_states, self.n_actions)
            self.reward_func = reward_func
            self.reward_table, self.reward_log2 = tables.lower_reward(reward_func, self.n_cells, self.n_states, self.n_actions)
            if stochastic:
                flags |= _lib.F_NOISE
            if self.reward_log2:
                flags |= _lib.F_REWARD_LOG2
        else:
            self.reward_func = reward_func
        if self.rng_episodic:
            flags |= _lib.F_RNG_EPISODIC
        if force_generic_kernel:
            flags |= _lib.F_GENERIC_KERNEL
        cfg.flags = flags
        cfg.n_envs, cfg.ld, cfg.env_id_offset = self.num_envs, self.ld, self.env_id_offset
        cfg.seed = self.env_seed & (2 ** 64 - 1)
        cfg.noise_prob, cfg.dispersal_prob = float(noise_prob), float(dispersal_prob)
        self._cfg = cfg
        handle = C.c_void_p()
        _lib.check(self._lib.gc_create(C.byref(cfg), C.byref(handle)))
        self._h = handle
        if kind == "cellular":
            self._set_tables()

        self._collect_stats = bool(collect_stats)
        if compressible_buffers is None:
            # a small shard's step is bound by latency, not by DRAM bytes, and compressed lines cost latency: on by
            # default above 1/16 of L2 (config 2, 1.2 MB of step buffers: 123-128 against 128-133 G env-steps/s
            # compressed; config 3, 19 MB: 334-336 against 329-330 G)
            l2 = torch.cuda.get_device_properties(self.device).L2_cache_size
            compressible_buffers = (bool(self._lib.gc_compressible_supported(self.device.index))
                                    and self.ld * self._step_bytes_per_env() > l2 // 16)
        self._compressible_buffers = bool(compressible_buffers)
        self._alloc_device_buffers()
        self._host = None                                 # pinned mirrors, allocated on first host step

        # --- spaces -------------------------------------------------------------------------
        sp = gym.spaces
        self.single_observation_space = sp.Tuple([sp.Discrete(self.n_states) for _ in range(self.n_cells)])
        self.single_action_space = sp.Tuple([sp.Discrete(self.n_actions) for _ in range(self.n_cells)])
        self._batched_spaces = None          # built on first access: 2 x n_cells arrays of num_envs int64
        self.closed = False
        self._build_views()
        self.reset()

    def _step_buffer_zeros(self):
        """zeros(*shape, dtype=...) for the env-owned step buffers: generic compressible memory when
        `compressible_buffers` is on (gc_alloc_compressible, which falls back to ordinary device memory where the
        device grants none), ordinary torch memory otherwise."""
        dev = self.device
        if not self._compressible_buffers:
            return lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)

        def zeros(*shape, dtype):
            t = torch.as_tensor(_CompressibleBlock(self._lib, shape, dtype, dev), device=dev)
            return t.zero_()
        return zeros

    @property
    def compressible(self):
        """True when every env-owned step buffer (state, time step, reward, index, flags) lives in generic
        compressible memory: L2 <-> DRAM transfers of its low-entropy lines move fewer bytes."""
        return all(self._lib.gc_is_compressible(_ptr(t)) for t in self._step_buffers())

    def _step_buffers(self):
        return (self._state, self._t, self._reward, self._index, self._terminated, self._truncated, self._unsafe,
                self._count)

    def _step_bytes_per_env(self):
        return self.n_cells + 16

    def _alloc_device_buffers(self):
        """Device buffers (caller-owned as far as the library is concerned)."""
        dev, ld, Cn = self.device, self.ld, self.n_cells
        z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
        step = self._step_buffer_zeros()
        self._state = step(Cn, ld, dtype=torch.int8)
        self._actions = z(Cn, ld, dtype=torch.int8)
        self._t = step(ld, dtype=torch.int32)
        self._reward = step(ld, dtype=torch.float32)
        self._index = step(ld, dtype=torch.int32)        # uint32 payload (see tabular_state())
        self._terminated = step(ld, dtype=torch.uint8)
        self._truncated = step(ld, dtype=torch.uint8)
        self._unsafe = step(ld, dtype=torch.uint8)
        self._count = step(ld, dtype=torch.uint8)
        self._se_row = z(Cn, ld, dtype=torch.int8) if self.emit_side_effects else None
        self._stats = z(_lib.N_STATS, dtype=torch.int64) if self._collect_stats else None
        self._final = z(Cn, ld, dtype=torch.int8) if self.emit_final_obs else None
        if self._final is not None:          # an extra output of every following step of the handle
            _lib.check(self._lib.gc_set_final_obs(self._h, _ptr(self._final)))

    def _spaces(self):
        if self._batched_spaces is None:
            sp = gym.spaces
            self._batched_spaces = tuple(
                sp.Tuple([sp.MultiDiscrete(np.full(self.num_envs, k)) for _ in range(self.n_cells)])
                for k in (self.n_states, self.n_actions))
        return self._batched_spaces

    @property
    def observation_space(self):
        """Batched space (gymnasium convention: a Tuple of n_cells MultiDiscrete([n_states] * num_envs));
        built lazily -- at 2^24 envs it is gigabytes of metadata nobody on the hot path needs."""
        return self._spaces()[0]

    @observation_space.setter
    def observation_space(self, value):
        pass                                   # gymnasium.vector.VectorEnv's class attribute protocol

    @property
    def action_space(self):
        return self._spaces()[1]

    @action_space.setter
    def action_space(self, value):
        pass

    # ------------------------------------------------------------------------------------------
    def _set_tables(self):
        S, A, Cn = self.n_states, self.n_actions, self.n_cells
        ct = self._cell_tables
        reward_noisy, counted, init = None, tables.counted_levels(S), np.zeros(Cn)
        if ct is not None:
            move, noisy, draws, se = ct["move"], ct.get("noisy"), ct.get("draws"), ct["side_effects"]
            reward_noisy, counted = ct.get("reward_noisy"), ct["counted"]
            if ct.get("initial_state") is not None:
                init = ct["initial_state"]
        elif self.stochastic:
            move, noisy, draws = tables.noise_tables(S, A, self.deadlock)
            se = tables.side_effect_tables(Cn, S, self.difficulty)
        else:
            move, noisy, draws = tables.move_table(S, A), None, None
            se = tables.side_effect_tables(Cn, S, self.difficulty)
        keep = [np.ascontiguousarray(move, np.int8),
                None if noisy is None else np.ascontiguousarray(noisy, np.int8),
                None if draws is None else np.ascontiguousarray(draws, np.uint8),
                np.ascontiguousarray(self.reward_table, np.float32),
                np.ascontiguousarray(se, np.int8),
                np.ascontiguousarray(counted, np.uint8),
                np.ascontiguousarray(init, np.int8),
                None if reward_noisy is None else np.ascontiguousarray(reward_noisy, np.float32),
                None if self.cell_radix is None else np.ascontiguousarray(self.cell_radix, np.int32)]
        if self.cell_radix is not None and len(self.cell_radix) != Cn:
            raise ValueError("cell_radix needs one entry per cell")
        if len(keep[6]) != Cn:
            raise ValueError("initial_state needs one entry per cell")
        t = _lib.GcCellTables(*[None if a is None else a.ctypes.data for a in keep])
        _lib.check(self._lib.gc_set_tables(self._h, C.byref(t)))
        self.side_effect_table = se

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ---- views -------------------------------------------------------------------------------
    @property
    def state(self):
        """int8 [n_cells, num_envs] view of the resident state (assignable through set_state)."""
        return self._state[:, :self.num_envs]

    def set_state(self, cells, t=None, validate=True):
        """Overwrite the resident state (and optionally the episode steps), as tests and agents do with
        `env.state = ...` on the reference; the tabular index is refreshed.  `validate` checks the level
        range (one host synchronisation)."""
        cells = torch.as_tensor(cells, device=self.device).to(torch.int8).reshape(self.n_cells, self.num_envs)
        if validate:
            levels = self.n_states if self.cell_radix is None else \
                torch.tensor(self.cell_radix, dtype=torch.int8, device=self.device)[:, None]
            if bool((cells < 0).any()) or bool((cells >= levels).any()):
                raise ValueError(f"state levels must lie in [0, {self.n_states if self.cell_radix is None else self.cell_radix})")
        self._state[:, :self.num_envs].copy_(cells)
        if t is not None:
            self._t[:self.num_envs].copy_(torch.as_tensor(t, device=self.device).to(torch.int32))
        self._encode_state(self._state, self._index, self.num_envs, self.ld)

    def _encode_state(self, cells, index, n, ld):
        """Tabular index of int8 [n_cells, ld] device levels, with the place values the step kernels use: the
        uniform radix n_states, or the per-cell `cell_radix` of a ragged state space."""
        if self.cell_radix is None:
            _lib.check(self._lib.gc_encode(self.device.index, n, ld, self.n_cells, self.n_states, _ptr(cells),
                                           _ptr(index), self._stream()))
        else:
            radix = np.ascontiguousarray(self.cell_radix, np.int32)
            _lib.check(self._lib.gc_encode_mixed(self.device.index, n, ld, self.n_cells, radix.ctypes.data, None,
                                                 _ptr(cells), _ptr(index), self._stream()))

    def tabular_state(self, dtype=torch.int64):
        """Tabular index of the current observation (uint32 payload widened to `dtype`)."""
        idx = self._index[:self.num_envs]
        if dtype == torch.int32:
            return idx
        return idx.to(torch.int64) & 0xFFFFFFFF

    # ---- batched codec (SURVEY 8 f1): both directions, states and actions -----------------------
    def tabularize(self, cells, space="state"):
        """int8 [n_cells, n] device tensor (n a multiple of 16, contiguous) -> int64 [n] tabular indices.
        `space`: 'state' or 'action' (radix n_states or n_actions; grid world 20 / 5), i.e. the batched
        `prior_knowledge.tabularize` (cells3states3actions3.py:281-284, grid_world.py:397-407)."""
        cells = torch.as_tensor(cells, device=self.device).to(torch.int8).contiguous()
        n = cells.shape[1]
        ld = _round_up(n, 16)
        if ld != n:
            pad = torch.zeros(cells.shape[0], ld, dtype=torch.int8, device=self.device)
            pad[:, :n] = cells
            cells = pad
        out = torch.empty(ld, dtype=torch.int32, device=self.device)
        if space == "state" and self.cell_radix is not None:
            self._encode_state(cells, out, n, ld)
        else:
            radix = self.n_states if space == "state" else self.n_actions
            _lib.check(self._lib.gc_encode(self.device.index, n, ld, cells.shape[0], radix, _ptr(cells), _ptr(out),
                                           self._stream()))
        return out[:n].to(torch.int64) & 0xFFFFFFFF

    def detabularize(self, index, space="state"):
        """int64/int32 [n] tabular indices -> int8 [n_cells, n] cells: the batched
        `prior_knowledge.detabularize` (generalized_space_transformations.py:15-23)."""
        index = torch.as_tensor(index, device=self.device)
        n = index.shape[0]
        ld = _round_up(n, 16)
        idx = torch.zeros(ld, dtype=torch.int32, device=self.device)
        idx[:n] = (index.to(torch.int64) & 0xFFFFFFFF).to(torch.int32) if index.dtype != torch.int32 else index
        out = torch.empty(self.n_cells, ld, dtype=torch.int8, device=self.device)
        if space == "state" and self.cell_radix is not None:
            radix = np.ascontiguousarray(self.cell_radix, np.int32)
            _lib.check(self._lib.gc_decode_mixed(self.device.index, n, ld, self.n_cells, radix.ctypes.data, None,
                                                 _ptr(idx), _ptr(out), self._stream()))
        else:
            radix = self.n_states if space == "state" else self.n_actions
            _lib.check(self._lib.gc_decode(self.device.index, n, ld, self.n_cells, radix, _ptr(idx), _ptr(out),
                                           self._stream()))
        return out[:, :n]

    def materialise(self, i):
        """Observation of env i in the reference's own Python type: a tuple of ints (polarisation
        family) or a tuple of {'agt': ..., 'living_trees': ...} dicts (grid world, grid_world.py:364-394)."""
        codes = [int(x) for x in self._state[:, i].cpu().tolist()]
        if self.kind == "gridworld":
            from .envs import GridWorldPriorKnowledge
            return GridWorldPriorKnowledge().decellularize(codes, "state")
        return tuple(codes)

    @property
    def time_step(self):
        return self._t[:self.num_envs]

    def stats(self, reset=False):
        """Episode statistics accumulated in-kernel since the last reset of the accumulators."""
        if self._stats is None:
            raise RuntimeError("collect_stats=False")
        s = self._stats.cpu().numpy().copy()
        if reset:
            self._stats.zero_()
        return {"env_steps": int(s[_lib.STAT_STEPS]), "unsafe_steps": int(s[_lib.STAT_UNSAFE]),
                "count_sum": int(s[_lib.STAT_COUNT]), "episodes_truncated": int(s[_lib.STAT_TRUNCATED]),
                "reward_sum": float(s[_lib.STAT_REWARD_Q24]) / 2.0 ** 24}

    # ---- checkpoint / resume -----------------------------------------------------------------------
    def state_dict(self):
        """Everything needed to resume: the resident state, episode steps, statistics and the global
        step (the RNG itself is stateless: Philox is keyed by seed, global env id and step)."""
        self.sync_step_counter()
        return {"state": self._state.clone(), "t": self._t.clone(),
                "stats": None if self._stats is None else self._stats.clone(),
                "global_step": int(self._lib.gc_get_global_step(self._h)),
                "meta": (self.kind, self.num_envs, self.n_cells, self.n_states, self.env_seed, self.env_id_offset)}

    def load_state_dict(self, sd):
        if tuple(sd["meta"]) != (self.kind, self.num_envs, self.n_cells, self.n_states, self.env_seed, self.env_id_offset):
            raise ValueError("state_dict belongs to a differently configured env")
        self._state.copy_(sd["state"])
        self._t.copy_(sd["t"])
        if self._stats is not None and sd["stats"] is not None:
            self._stats.copy_(sd["stats"])
        # gc_set_global_step is ordered only after blocking streams: a step still queued on a non-blocking current
        # stream would read the restored counter and then overwrite it with its own successor
        torch.cuda.current_stream(self.device).synchronize()
        _lib.check(self._lib.gc_set_global_step(self._h, int(sd["global_step"])))
        # refresh the tabular index of the restored state
        self._encode_state(self._state, self._index, self.num_envs, self.ld)

    @property
    def launch_count(self):
        return int(self._lib.gc_launch_count(self._h))

    # ---- gymnasium.vector API ----------------------------------------------------------------
    def reset(self, *, seed=None, options=None):
        """Reference reset() ignores its seed (cells3states3actions3.py:99); so does this one."""
        _lib.check(self._lib.gc_reset(self._h, None, _ptr(self._state), _ptr(self._t), _ptr(self._index),
                                      self._stream()))
        self._reward.zero_()
        self._truncated.zero_()
        self._unsafe.zero_()
        self._count.zero_()
        if self._se_row is not None:
            # the reference's reset() info: cellular envs hard-code row 0 = ('safe', 'silent', ...)
            # (cells3states3actions3.py:102-109); grid world evaluates side_effects_func (grid_world.py:101)
            self._se_row.zero_()
            if self._cell_tables is not None:
                for c, code in enumerate(self._cell_tables["reset_row"]):
                    self._se_row[c].fill_(int(code))
            elif self.kind == "cellular":
                self._se_row[0].fill_(tables.SAFE)
            else:
                self._se_row.fill_(tables.SAFE)
        if self._final is not None:
            self._final.copy_(self._state)
        # the global step (RNG counter of the non-episodic kinds: grid world, DeepExplorationDebug) is NOT
        # rewound: the reference never re-seeds these envs (grid_world.py:97-104), every episode draws
        # fresh numbers.  The episodic kinds count from the per-env episode step, which reset() zeroes.
        return self._obs_device(), self._infos_device()

    def reset_envs(self, mask):
        """Masked reset: `mask` is a bool/uint8 tensor [num_envs] on the device."""
        m = torch.zeros(self.ld, dtype=torch.uint8, device=self.device)
        m[:self.num_envs] = torch.as_tensor(mask, device=self.device).to(torch.uint8)
        _lib.check(self._lib.gc_reset(self._h, _ptr(m), _ptr(self._state), _ptr(self._t), _ptr(self._index),
                                      self._stream()))

    def step(self, actions, replay_u=None):
        if isinstance(actions, np.ndarray) or (isinstance(actions, (tuple, list)) and len(actions)
                                                and isinstance(actions[0], np.ndarray)):
            return self._step_host(actions)
        self.step_device(actions, replay_u=replay_u)
        return self._v_obs, self._v_reward, self._v_term, self._v_trunc, self._v_infos

    def step_device(self, actions=None, replay_u=None):
        """Launch one step on the current stream; no host synchronisation, no output marshalling.
        `actions`: None = the env's own action buffer (`action_buffer`) already holds them."""
        if replay_u is None and type(actions) is torch.Tensor:
            # hot path: the same action tensor(s) again and again -> a pre-bound launch per buffer
            cache = self.__dict__.setdefault("_bound_cache", {})
            call = cache.get(actions.data_ptr())
            if call is None and len(cache) < 8 and actions.shape == (self.n_cells, self.ld) \
                    and actions.dtype == torch.int8 and actions.is_contiguous() and actions.device == self.device:
                call = cache[actions.data_ptr()] = (self.bind_step(actions), actions)   # keeps the buffer alive
            if call is not None and call[1] is actions:
                call[0]()
                return
        a_ptr = _ptr(self._actions)
        if actions is not None:
            a_ptr = self._load_actions_device(actions)
        ru = None
        if replay_u is not None:
            ru = torch.as_tensor(replay_u, dtype=torch.float64, device=self.device).contiguous()
            slots = self.n_cells if self.kind == "cellular" else 6
            if ru.shape != (self.num_envs, slots):
                raise ValueError(f"replay_u must have shape {(self.num_envs, slots)}")
        _lib.check(self._lib.gc_step(
            self._h, 0, self.num_envs, a_ptr, _ptr(self._state), _ptr(self._t), _ptr(self._reward),
            _ptr(self._index), _ptr(self._terminated), _ptr(self._truncated), _ptr(self._unsafe), _ptr(self._count),
            _ptr(self._se_row), _ptr(ru), _ptr(self._stats), self._stream()))

    def _bind(self, actions=None):
        """Stores the pointer set of a full-shard step in one of the handle's 16 slots; returns the slot."""
        a = self._actions if actions is None else actions
        if a.dtype != torch.int8 or a.shape != (self.n_cells, self.ld) or not a.is_contiguous() or a.device != self.device:
            raise ValueError(f"bind_step needs a contiguous int8 tensor of shape {(self.n_cells, self.ld)} on {self.device}")
        slot = getattr(self, "_n_bound", 0)
        if slot >= 16:                      # GC_MAX_BINDINGS: the pointer set lives in the handle
            raise RuntimeError("all 16 binding slots of the handle are in use")
        self._n_bound = slot + 1
        _lib.check(self._lib.gc_bind_step(self._h, slot, _ptr(a), _ptr(self._state), _ptr(self._t), _ptr(self._reward),
                                          _ptr(self._index), _ptr(self._terminated), _ptr(self._truncated),
                                          _ptr(self._unsafe), _ptr(self._count), _ptr(self._se_row), _ptr(self._stats)))
        self.__dict__.setdefault("_bound_keepalive", []).append(a)
        return slot

    def bind_step(self, actions=None, stream=None):
        """Returns a zero-argument callable that launches one step with all ctypes arguments
        pre-bound (for tight rollout loops: ~4-6 us of host time per step) -- on `stream`
        (a torch.cuda.Stream, its handle looked up once) or, by default, on whatever stream is
        current at each call.  `actions`: an int8 device tensor [n_cells, ld] kept alive by the
        caller, or None for `action_buffer`."""
        check, dev, current_stream = _lib.check, self.device, torch.cuda.current_stream
        if stream is not None:
            if stream.device != self.device:
                raise ValueError(f"stream lives on {stream.device}, the env on {self.device}")
            pinned = stream.cuda_stream
        if getattr(self, "_n_bound", 0) < 16:
            slot = self._bind(actions)
            fn, h = self._lib.gc_step_bound, self._h

            if stream is not None:
                def launch():
                    rc = fn(h, slot, pinned)
                    if rc:
                        check(rc)
                launch.stream, launch.slot = stream, slot     # keeps the stream object alive, too
                return launch

            def launch():
                rc = fn(h, slot, current_stream(dev).cuda_stream)
                if rc:
                    check(rc)
            launch.slot = slot
            return launch
        a = self._actions if actions is None else actions
        if a.dtype != torch.int8 or a.shape != (self.n_cells, self.ld) or not a.is_contiguous() or a.device != self.device:
            raise ValueError(f"bind_step needs a contiguous int8 tensor of shape {(self.n_cells, self.ld)} on {self.device}")
        fn = self._lib.gc_step
        args = (self._h, 0, self.num_envs, _ptr(a), _ptr(self._state), _ptr(self._t), _ptr(self._reward),
                _ptr(self._index), _ptr(self._terminated), _ptr(self._truncated), _ptr(self._unsafe),
                _ptr(self._count), _ptr(self._se_row), None, _ptr(self._stats))
        if stream is not None:
            current_stream = lambda _dev: stream          # noqa: E731

        def launch():
            rc = fn(*args, current_stream(dev).cuda_stream)
            if rc:
                check(rc)
        return launch

    def step_many(self, slots, n_steps, stream=None):
        """`n_steps` pre-bound steps back to back in ONE foreign call (gc_step_many): step i launches the
        binding `slots[i % len(slots)]` (slots from `_bind` / `bind_step(...).slot`).  The launches are
        chained by programmatic dependent launch and no Python runs between them -- the per-step loop of
        launch-bound batch sizes without capturing a CUDA graph.  Shards of up to 2^21 envs whose slots differ only
        in their action tensors (what `_bind` / `bind_step` produce) run all the steps inside ONE kernel, every
        per-step output still written at every step (include/gym_cellular_b200.h: gc_step_many)."""
        arr = self._slot_array(slots)
        st = (torch.cuda.current_stream(self.device) if stream is None else stream).cuda_stream
        _lib.check(self._lib.gc_step_many(self._h, arr, len(arr), int(n_steps), st))

    def _slot_array(self, slots):
        key = tuple(int(x) for x in slots)
        cache = self.__dict__.setdefault("_slot_arrays", {})
        arr = cache.get(key)
        if arr is None:
            arr = cache[key] = (C.c_int32 * len(key))(*key)
        return arr

    def prepare_step_many(self, slots):
        """Builds the CUDA graph `step_many` replays for this slot list ahead of time (small shards only; no step
        is executed), so that the first `step_many` does not pay for the capture."""
        arr = self._slot_array(slots)
        _lib.check(self._lib.gc_prepare_step_many(self._h, arr, len(arr)))

    def rollout(self, n_steps, policy=None, policy_of_env=None):
        """Fused K-step rollout: `n_steps` steps per env inside one kernel, actions generated on the
        device -- uniformly at random (policy=None) or from a tabular policy (int tensor
        [n_states ** n_cells] of tabular action indices).  Returns (returns float32 [num_envs],
        unsafe_steps int32 [num_envs]); state, time_step, tabular_state() and stats() advance exactly as
        if step() had been called n_steps times with those actions.
        policy_of_env: a stack of policies in one launch -- `policy` is then [P, n_states ** n_cells] and env e acts
        by table policy_of_env[e] (an integer tensor [num_envs] on the env's device, values in [0, P)), exactly as it
        would under that table alone.  The map is checked (one host synchronisation) and copied when a new tensor,
        or a new version of it, arrives; a repeated call with the same map adds neither."""
        n = self.num_envs
        if getattr(self, "_ro_ret", None) is None:
            self._ro_ret = torch.zeros(self.ld, dtype=torch.float32, device=self.device)
            self._ro_unsafe = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
        kind, ptab = self._policy_table(policy, policy_of_env)
        _lib.check(self._lib.gc_rollout(self._h, int(n_steps), kind, _ptr(ptab), _ptr(self._state), _ptr(self._t),
                                        _ptr(self._index), _ptr(self._ro_ret), _ptr(self._ro_unsafe), _ptr(self._stats),
                                        self._stream()))
        return self._ro_ret[:n], self._ro_unsafe[:n]

    def collect(self, n_steps, policy=None, epsilon=0.0, next_obs=False, policy_of_env=None):
        """Experience collection: `n_steps` steps per env inside one kernel, as `rollout()`, recording every
        transition.  policy=None: uniformly random actions (epsilon must be 0); a table as for `rollout()`: the
        epsilon-greedy policy that takes policy[obs] and, with probability `epsilon`, a uniformly random joint
        action instead (grid world: the reference sampler's).  Exploration is keyed by global env id and global
        step, so it differs between episodes even when the env's noise replays (`rng_episodic`).
        Returns `Transitions(obs, action, reward, flags, next_obs)` of [n_steps, num_envs] views; state,
        time_step, tabular_state() and stats() advance exactly as `rollout()` advances them.  The views alias
        buffers cached per n_steps: the next `collect` with the same n_steps overwrites them, as a step
        overwrites its outputs.  policy_of_env: a stack of table policies, one per env, as for `rollout()`; an
        exploring env takes the uniformly random joint action whatever its table."""
        return self._collect(n_steps, policy, epsilon, next_obs, self._state, self._index, policy_of_env)

    def _policy_table(self, policy, policy_of_env=None):
        if policy_of_env is not None:
            ptab = _check_policy_stack(policy, policy_of_env, self._joint_sizes()[0], self.num_envs, self.device)
            self._set_policy_map(policy_of_env, ptab.shape[0])
            return _lib.POLICY_TABLE_STACK, ptab
        if policy is None:
            return _lib.POLICY_RANDOM, None
        ptab = torch.as_tensor(policy, device=self.device).to(torch.int32).contiguous()
        if ptab.numel() != self.n_states ** self.n_cells:
            raise ValueError("policy must have one entry per tabular state")
        return _lib.POLICY_TABLE, ptab

    def _set_policy_map(self, policy_of_env, n_tables):
        """Hands the table map of a policy stack to the handle (gc_set_policy_stack): an [ld] int32 copy owned by the
        env, so that the kernels' 4-env reads of the padding stay inside it.  A map tensor seen before, unchanged
        (same object, same `_version`) and for the same number of tables, is neither checked nor copied again, so build
        the map once and pass the same tensor: a map rebuilt on every call is checked on every call (one host
        synchronisation).  The env holds only a weak reference to it."""
        key = getattr(self, "_map_key", None)
        if key is not None and key[0]() is policy_of_env and key[1] == policy_of_env._version and key[2] == n_tables:
            return
        if bool(((policy_of_env < 0) | (policy_of_env >= n_tables)).any()):
            raise ValueError(f"policy_of_env holds table ids outside [0, {n_tables})")
        if getattr(self, "_map", None) is None:
            self._map = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
        self._map[:self.num_envs].copy_(policy_of_env)
        _lib.check(self._lib.gc_set_policy_stack(self._h, _ptr(self._map), int(n_tables)))
        self._map_key = (weakref.ref(policy_of_env), policy_of_env._version, n_tables)

    def _collect(self, n_steps, policy, epsilon, next_obs, state, index, policy_of_env=None):
        n_steps = int(n_steps)
        kind, ptab = self._policy_table(policy, policy_of_env)
        bufs = self.__dict__.setdefault("_record_bufs", {})
        buf = bufs.get(n_steps)
        if buf is None:
            rows = max(n_steps, 1)              # n_steps < 1 is rejected by the library, with its message
            z = lambda dtype: torch.zeros(rows, self.ld, dtype=dtype, device=self.device)     # noqa: E731
            buf = bufs[n_steps] = {"obs": z(torch.int32), "action": z(torch.int32), "reward": z(torch.float32),
                                   "flags": z(torch.uint8), "next_obs": None}
        if next_obs and buf["next_obs"] is None:
            buf["next_obs"] = torch.zeros_like(buf["obs"])
        nx = buf["next_obs"] if next_obs else None
        rec = _lib.GcRecord(C.sizeof(_lib.GcRecord), buf["obs"].data_ptr(), buf["action"].data_ptr(),
                            buf["reward"].data_ptr(), buf["flags"].data_ptr(), None if nx is None else nx.data_ptr())
        _lib.check(self._lib.gc_collect(self._h, n_steps, kind, _ptr(ptab), float(epsilon), _ptr(state), _ptr(self._t),
                                        _ptr(index), C.byref(rec), _ptr(self._stats), self._stream()))
        n = self.num_envs
        return Transitions(buf["obs"][:, :n], buf["action"][:, :n], buf["reward"][:, :n], buf["flags"][:, :n],
                           None if nx is None else nx[:, :n])

    def _joint_sizes(self):
        if self.kind == "gridworld":
            return 400, 25
        return self.n_states ** self.n_cells, self.n_actions ** self.n_cells

    def zero_counts(self, joint=True, transitions=True, groups=None):
        """Zeroed `Counts` tables for `collect_counts`.  joint=False leaves the four joint tables None (for envs too
        large for them, such as 16 cells x 4 levels, only the per-cell `cell_next` is kept); transitions=False leaves
        `next` None.  `cell_next` is None for grid world.  groups=P: grouped counts, one set per table of a policy stack
        of P tables, with a leading [P] on every table (`collect_counts(..., policy_of_env=)`); each table then holds at
        most 2**31 entries in all."""
        nS, nA = self._joint_sizes()
        S, A, Cn = self.n_states, self.n_actions, self.n_cells
        lead = ()
        if groups is not None:
            if isinstance(groups, bool) or not isinstance(groups, (int, np.integer)) or groups < 1:
                raise ValueError(f"groups must be an int >= 1 (got {groups!r})")
            lead = (int(groups),)
        G = lead[0] if lead else 1
        what = f"{G} groups x " if lead else ""
        if joint and (G * nS * nA > _JOINT_LIMIT or (transitions and G * nS * nA * nS > _JOINT_LIMIT)):
            raise ValueError(f"the joint count tables of {what}{nS} states x {nA} actions exceed 2**31 entries: use "
                             "joint=False" + ("" if G * nS * nA > _JOINT_LIMIT else " or transitions=False")
                             + (" or fewer groups" if lead else ""))
        if self.kind == "cellular" and G * Cn * S * A * S > _JOINT_LIMIT:
            raise ValueError(f"the per-cell count table of {what}{Cn} cells exceeds 2**31 entries: use fewer groups")
        z = lambda *shape: torch.zeros(*lead, *shape, dtype=torch.int64, device=self.device)      # noqa: E731
        return Counts(z(nS, nA) if joint else None, z(nS, nA, nS) if joint and transitions else None,
                      z(nS, nA) if joint else None, z(nS, nA) if joint else None,
                      z(Cn, S, A, S) if self.kind == "cellular" else None)

    def collect_counts(self, n_steps, policy=None, epsilon=0.0, counts=None, policy_of_env=None):
        """Experience counts: `n_steps` steps per env inside one kernel, as `collect()` (same policies, same epsilon
        rule, same draws), adding every transition to `counts` instead of recording it.  counts=None allocates
        `zero_counts()`.  Returns `counts`; the counts equal the histogram of the record `collect()` would return, and
        state, time_step, tabular_state() and stats() advance exactly as `collect()` advances them.  The counts are
        integers, so they are exact, independent of the order of the adds and of how the envs are sharded.
        policy_of_env: a stack of table policies, one per env, as for `rollout()`.  All envs add to the one `counts`,
        unless `counts` are grouped (`zero_counts(groups=P)`, P = policy.shape[0]): env e then adds into group
        policy_of_env[e] only, so `counts.group(g)` is the histogram of the record over the envs of table g and the sum
        over the groups is what ungrouped counts would hold.  Still one launch."""
        return self._collect_counts(n_steps, policy, epsilon, counts, self._state, self._index, policy_of_env)

    def _collect_counts(self, n_steps, policy, epsilon, counts, state, index, policy_of_env=None):
        if counts is None:
            counts = self.zero_counts()
        nS, nA = self._joint_sizes()
        shapes = Counts((nS, nA), (nS, nA, nS), (nS, nA), (nS, nA),
                        (self.n_cells, self.n_states, self.n_actions, self.n_states) if self.kind == "cellular" else None)
        if not isinstance(counts, Counts) or all(t is None for t in counts):
            raise ValueError("counts must be a Counts with at least one table (see zero_counts())")
        # grouped counts: one more leading dimension on every table, of the size of the policy stack
        given = [(t, shape) for t, shape in zip(counts, shapes) if isinstance(t, torch.Tensor) and shape is not None]
        grouped = bool(given) and given[0][0].dim() == len(given[0][1]) + 1
        if grouped and policy_of_env is None:
            raise ValueError("grouped counts (a leading group dimension) need policy_of_env: one group per table")
        kind, ptab = self._policy_table(policy, policy_of_env)
        if grouped:
            if given[0][0].shape[0] != ptab.shape[0]:
                raise ValueError(f"grouped counts have {given[0][0].shape[0]} groups; the policy stack has "
                                 f"{ptab.shape[0]} tables (one group per table)")
            shapes = Counts(*(None if sh is None else (ptab.shape[0],) + sh for sh in shapes))
        for name, t, shape in zip(Counts._fields, counts, shapes):
            if t is None:
                continue
            if shape is None:
                raise ValueError(f"counts.{name} must be None for {self.kind}")
            # the kernel adds at flat indices of these shapes: a smaller table would be written past its end
            if tuple(t.shape) != shape:
                raise ValueError(f"counts.{name} has shape {tuple(t.shape)}; this env's is {shape} (see zero_counts())")
            if t.dtype != torch.int64 or t.device != self.device or not t.is_contiguous():
                raise ValueError("count tables must be contiguous int64 tensors on the env's device")
        cs = _lib.GcCounts(C.sizeof(_lib.GcCounts), *(None if t is None else t.data_ptr() for t in counts))
        if grouped:
            _lib.check(self._lib.gc_collect_counts_grouped(self._h, int(n_steps), _ptr(ptab), float(epsilon), _ptr(state),
                                                           _ptr(self._t), _ptr(index), C.byref(cs), _ptr(self._stats),
                                                           self._stream()))
        else:
            _lib.check(self._lib.gc_collect_counts(self._h, int(n_steps), kind, _ptr(ptab), float(epsilon), _ptr(state),
                                                   _ptr(self._t), _ptr(index), C.byref(cs), _ptr(self._stats),
                                                   self._stream()))
        return counts

    def capture_steps(self, action_ring):
        """Captures one step per tensor of `action_ring` (int8 [n_cells, ld] device tensors, kept alive
        by the caller) into a CUDA graph and returns it; `graph.replay()` then runs len(action_ring)
        steps with a single launch.  The RNG step counter lives in device memory and is advanced by the
        kernels themselves, so every replay draws fresh numbers.  For launch-bound batch sizes."""
        calls = [self.bind_step(a) for a in action_ring]
        graph = torch.cuda.CUDAGraph()
        torch.cuda.synchronize(self.device)
        with torch.cuda.graph(graph):
            for call in calls:
                call()
        return graph

    def sync_step_counter(self):
        """Reads the device-resident global step into the host mirror and returns it.  (The kernels of
        every path -- step, bound step, graph replay, host-path chunks -- read the device word; the mirror
        only serves state_dict() and diagnostics.)"""
        _lib.check(self._lib.gc_sync_global_step(self._h, self._stream()))
        return int(self._lib.gc_get_global_step(self._h))

    @property
    def action_buffer(self):
        """int8 [n_cells, num_envs] device view: write actions here and call step_device()."""
        return self._actions[:, :self.num_envs]

    def check_actions(self):
        """Raises KeyError('position') if a grid-world env got an action without any go-to position
        since the last call (the reference raises at grid_world.py:143).  Synchronises."""
        rc = self._lib.gc_poll_status(self._h, self._stream())
        if rc == _lib.ERR_ACTION:
            raise KeyError("position")
        _lib.check(rc)

    def close_extras(self, **kwargs):
        if getattr(self, "_h", None):
            self._lib.gc_destroy(self._h)
            self._h = None

    # ---- helpers -----------------------------------------------------------------------------
    def _load_actions_device(self, actions):
        if isinstance(actions, (tuple, list)):
            actions = torch.stack([torch.as_tensor(a, device=self.device) for a in actions])
        elif not isinstance(actions, torch.Tensor):
            actions = torch.from_dlpack(actions)
        if actions.shape == (self.num_envs, self.n_cells) and self.num_envs != self.n_cells:
            actions = actions.t()
        if actions.shape != (self.n_cells, self.num_envs):
            raise ValueError(f"actions must have shape {(self.n_cells, self.num_envs)}")
        if (actions.dtype == torch.int8 and actions.device == self.device and actions.is_contiguous()
                and self.num_envs == self.ld and actions.data_ptr() % 16 == 0):
            return C.c_void_p(actions.data_ptr())       # the caller's tensor has the kernel's layout: no copy
        if actions.data_ptr() != self._actions.data_ptr():
            self._actions[:, :self.num_envs].copy_(actions.to(self.device, non_blocking=True))
        return _ptr(self._actions)

    def _build_views(self):
        """Zero-copy views handed back by step()/reset(): they alias the env's buffers (valid until the
        next step) and are built once, so a device-path step() launches exactly one kernel."""
        n = self.num_envs
        self._v_obs = tuple(self._state[c, :n] for c in range(self.n_cells))
        self._v_reward = self._reward[:n]
        self._v_term = self._terminated[:n].view(torch.bool)
        self._v_trunc = self._truncated[:n].view(torch.bool)
        self._v_infos = {"unsafe": self._unsafe[:n].view(torch.bool), "count": self._count[:n],
                         "time_step": self._t[:n]}
        # the index is a uint32 payload in an int32 tensor: directly usable whenever it fits 31 bits
        key = "tabular_state" if self.n_states ** self.n_cells <= 2 ** 31 else "tabular_state_u32"
        self._v_infos[key] = self._index[:n]
        if self._se_row is not None:
            self._v_infos["side_effects"] = self._se_row[:, :n]
        if self._final is not None:
            # gymnasium SAME_STEP auto-reset: the observation the episode ended with, valid where `_final_obs`;
            # reward / unsafe / count / side_effects of the returned step already describe that final step
            self._v_infos["final_obs"] = tuple(self._final[c, :n] for c in range(self.n_cells))
            self._v_infos["_final_obs"] = self._v_trunc
            self._v_infos["final_info"] = _FinalInfo(self)
            self._v_infos["_final_info"] = self._v_trunc

    def _obs_device(self):
        return self._v_obs

    def _infos_device(self):
        """`tabular_state` is the int32 index tensor (zero-copy); for spaces above 2^31 states the key
        is `tabular_state_u32` (raw uint32 payload) and `tabular_state()` widens it to int64."""
        return self._v_infos

    def side_effects_incidence(self):
        """count / n_cells, as the reference's data['side_effects_incidence'] (float32 tensor)."""
        return self._count[:self.num_envs].to(torch.float32) / self.n_cells

    def _alloc_host(self):
        ld, Cn = self.ld, self.n_cells
        pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype).pin_memory()
        self._host = {"actions": pin(Cn, ld, dtype=torch.int8), "state": pin(Cn, ld, dtype=torch.int8),
                      "reward": pin(ld, dtype=torch.float32), "index": pin(ld, dtype=torch.int32),
                      "terminated": pin(ld, dtype=torch.uint8), "truncated": pin(ld, dtype=torch.uint8),
                      "unsafe": pin(ld, dtype=torch.uint8), "count": pin(ld, dtype=torch.uint8)}
        if self._se_row is not None:
            self._host["se_row"] = pin(Cn, ld, dtype=torch.int8)
        self._host_np = {k: v.numpy() for k, v in self._host.items()}

    @property
    def host_bytes_per_env_step(self):
        """(host-to-device, device-to-host) bytes the host path of step() moves per env."""
        d2h = self.n_cells + 4 + 4 + 2 + (1 if self.max_episode_steps else 0)
        if self._se_row is not None:
            d2h += self.n_cells
        return self.n_cells, d2h

    @property
    def host_action_buffer(self):
        """Pinned int8 [n_cells, num_envs] numpy view: fill it and call step(host_action_buffer)
        to skip the staging copy of the host path."""
        if self._host is None:
            self._alloc_host()
        return self._host_np["actions"][:, :self.num_envs]

    def _step_host(self, actions):
        if self._host is None:
            self._alloc_host()
        n, h = self.num_envs, self._host_np
        h_actions_ptr = _ptr(self._host["actions"])
        if isinstance(actions, (tuple, list)):
            for c, a in enumerate(actions):
                h["actions"][c, :n] = a
        elif actions.shape == (self.n_cells, n):
            if actions.dtype == np.int8 and actions.flags.c_contiguous and n == self.ld:
                h_actions_ptr = C.c_void_p(actions.ctypes.data)      # caller's buffer (pinned or not), no staging copy
            elif actions.ctypes.data != h["actions"].ctypes.data:
                h["actions"][:, :n] = actions
        elif actions.shape == (n, self.n_cells):
            h["actions"][:, :n] = actions.T
        else:
            raise ValueError(f"actions must have shape {(self.n_cells, n)} or {(n, self.n_cells)}")
        torch.cuda.current_stream(self.device).synchronize()     # resident state must be settled
        H = self._host
        # 'terminated' is constant False (cells3states3actions3.py:122, grid_world.py:113) and 'truncated' is
        # too without a time limit: their zero-initialised mirrors are returned without a device-to-host copy
        _lib.check(self._lib.gc_step_host(
            self._h, h_actions_ptr, _ptr(H["state"]), _ptr(H["reward"]), _ptr(H["index"]),
            None, _ptr(H["truncated"]) if self.max_episode_steps else None, _ptr(H["unsafe"]), _ptr(H["count"]),
            _ptr(H.get("se_row")),
            _ptr(self._actions), _ptr(self._state), _ptr(self._t), _ptr(self._reward), _ptr(self._index),
            _ptr(self._terminated), _ptr(self._truncated), _ptr(self._unsafe), _ptr(self._count),
            _ptr(self._se_row), _ptr(self._stats), self.host_chunk_envs))
        obs = tuple(h["state"][c, :n] for c in range(self.n_cells))
        # zero-copy views of the pinned mirrors (valid until the next step); incidence = count / n_cells
        infos = {"unsafe": h["unsafe"][:n].view(np.bool_), "count": h["count"][:n],
                 "tabular_state": h["index"][:n].view(np.uint32)}
        if "se_row" in h:
            infos["side_effects"] = h["se_row"][:, :n]
        if self._final is not None:        # the final observations stay on the device: one extra copy when asked for
            fin = self._final[:, :n].cpu().numpy()
            infos["final_obs"] = tuple(fin[c] for c in range(self.n_cells))
            infos["_final_obs"] = h["truncated"][:n].view(np.bool_)
        return obs, h["reward"][:n], h["terminated"][:n].view(np.bool_), h["truncated"][:n].view(np.bool_), infos


class _FinalInfo(dict):
    """infos['final_info']: the info of the step an episode ended with.  `unsafe`, `count` and `side_effects`
    are the step's own (they always describe the step taken); `tabular_state` is the index of the final
    observation, encoded on demand."""

    def __init__(self, env):
        super().__init__()
        self._env = env

    def __missing__(self, key):
        env = self._env
        if key == "tabular_state":
            out = torch.empty(env.ld, dtype=torch.int32, device=env.device)
            if env.kind == "gridworld":
                _lib.check(env._lib.gc_encode(env.device.index, env.num_envs, env.ld, env.n_cells, 20,
                                              _ptr(env._final), _ptr(out), env._stream()))
            else:
                env._encode_state(env._final, out, env.num_envs, env.ld)
            return out[:env.num_envs].to(torch.int64) & 0xFFFFFFFF
        if key in ("unsafe", "count", "side_effects"):
            return env._v_infos[key]
        raise KeyError(key)


def make_vector_env(env_id, num_envs, layout="int8", **kwargs):
    """`gymnasium.make_vec`-style constructor from a registered id ('gym_cellular/<Name>-v0'): all seven
    ids of the reference (gym_cellular/__init__.py:4-45).  `layout='packed'` selects the packed-word layout
    (`PackedCellularVectorEnv`; every id but GridWorld)."""
    from . import tables
    name = env_id.split("/")[-1]
    debug = {"Debug-v0": tables.debug_tables, "DeepPlanningDebug-v0": tables.deep_planning_tables,
             "DeepExplorationDebug-v0": tables.deep_exploration_tables}
    if name not in _FAMILIES and name not in debug:
        raise ValueError(f"{env_id} has no batched CUDA implementation (have: {sorted(_FAMILIES) + sorted(debug)})")
    if layout not in ("int8", "packed"):
        raise ValueError("layout must be 'int8' or 'packed'")
    cls = CellularVectorEnv
    if layout == "packed":
        from .packed_env import PackedCellularVectorEnv as cls
    if name in debug:
        if name == "DeepExplorationDebug-v0":
            kwargs.setdefault("rng_episodic", False)    # the reference never re-seeds it (debug/deep_exploration.py:49)
        return cls(kind="cellular", num_envs=num_envs, cell_tables=debug[name](), **kwargs)
    kind, n_cells, n_states, n_actions, stochastic = _FAMILIES[name]
    if kind == "gridworld":
        if layout == "packed":
            raise ValueError("the packed layout covers the cellular family; GridWorld uses the int8 layout")
        return CellularVectorEnv(kind="gridworld", num_envs=num_envs, **kwargs)
    kwargs.setdefault("n_cells", n_cells)
    kwargs.setdefault("n_states", n_states)
    kwargs.setdefault("n_actions", n_actions)
    kwargs.setdefault("stochastic", stochastic)
    return cls(kind="cellular", num_envs=num_envs, **kwargs)
