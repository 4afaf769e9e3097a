"""`PackedCellularVectorEnv`: the cellular (polarisation) vector env in the packed layout.

The joint cell state and the joint action of an env are ONE 32-bit word each, 2 bits per cell, cell c
in bits 2c and 2c+1 (n_states, n_actions <= 4: every polarisation env of the reference and the 16-cell
x 4-level scale-up).  With four levels the state word IS the reference's tabular index
(`prior_knowledge.tabularize`, cells3states3actions3.py:281-284 /
generalized_space_transformations.py:1-12) -- which is all a tabular agent consumes besides the reward
and the safety flag of `step()` (cells3states3actions3.py:116-125).  Compared with the int8
structure-of-arrays layout of `CellularVectorEnv` an env-step moves 25 instead of 3 n_cells + 20 bytes
through HBM and 4 in / 9 out instead of n_cells / n_cells + 10 bytes over the host link.

Same rules, same Philox draws, bit-identical results (tests/test_gpu_packed.py); `pack()` / `unpack()`
convert between the layouts on the device.  No CPU implementation: it raises without the CUDA library
or a CUDA device.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .vector_env import CellularVectorEnv, _ptr, _round_up


def pack_host(cells):
    """numpy int [n_cells, n] levels -> uint32 [n] packed words (2 bits per cell, cell 0 lowest)."""
    cells = np.asarray(cells)
    out = np.zeros(cells.shape[1], np.uint32)
    for c in range(cells.shape[0]):
        out |= (cells[c].astype(np.uint32) & 3) << np.uint32(2 * c)
    return out


def unpack_host(words, n_cells):
    """uint32 [n] packed words -> int8 [n_cells, n] levels."""
    words = np.asarray(words).astype(np.uint32, copy=False)
    return np.stack([((words >> np.uint32(2 * c)) & 3).astype(np.int8) for c in range(n_cells)])


class PackedCellularVectorEnv(CellularVectorEnv):
    """Batched polarisation env whose resident state, actions and host wire format are packed words.

    Constructor arguments as `CellularVectorEnv` (kind is 'cellular'; n_states, n_actions <= 4), plus
      emit_final_obs   also write the next state BEFORE a time-limit auto-reset (`infos['final_obs']`)
    `emit_side_effects` defaults to False here (row 0 of the side-effects matrix then costs nothing).

    step() takes, on the device path, an int32/uint32 tensor [num_envs] of action words (or an int8
    tensor [n_cells, num_envs], packed on the device first) and, on the host path, a numpy uint32/int32
    array [num_envs] (or int8 [n_cells, num_envs], packed on the host first).  It returns
    (state words, reward, terminated, truncated, infos); infos carries `flags` (bit 0 unsafe, bit 1
    truncated, bits 2-6 count), `unsafe`, `count`, `tabular_state` and `time_step` as lazily evaluated
    views, so a device-path step() is exactly one kernel launch.
    """

    def __init__(self, *args, emit_side_effects=False, **kwargs):
        kind = args[0] if args else kwargs.setdefault("kind", "cellular")
        if kind != "cellular":
            raise ValueError("the packed layout covers the cellular (polarisation) family")
        super().__init__(*args, emit_side_effects=emit_side_effects, **kwargs)

    # ---- buffers -----------------------------------------------------------------------------------
    def _alloc_device_buffers(self):
        if self.n_states > 4 or self.n_actions > 4:
            self.close_extras()
            raise ValueError("the packed layout needs n_states, n_actions <= 4 (2 bits per cell)")
        dev, ld = self.device, self.ld
        z = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype, device=dev)
        self._state = z(ld, dtype=torch.int32)            # uint32 payload: 2 bits per cell
        self._actions = z(ld, dtype=torch.int32)
        self._t = z(ld, dtype=torch.int32)
        self._reward = z(ld, dtype=torch.float32)
        self._flags = z(ld, dtype=torch.uint8)
        # four levels: the state word is the tabular index; otherwise the kernel writes it separately
        self._index = self._state if self.n_states == 4 else z(ld, dtype=torch.int32)
        self._final = z(ld, dtype=torch.int32) if self.emit_final_obs else None
        self._se_row = z(ld, dtype=torch.int32) if self.emit_side_effects else None
        self._stats = z(_lib.N_STATS, dtype=torch.int64) if self._collect_stats else None
        self._false = z(ld, dtype=torch.bool)
        self._cells_scratch = None

    def _index_ptr(self):
        return None if self._index is self._state else _ptr(self._index)

    @property
    def hbm_bytes_per_env_step(self):
        """Algorithmic HBM bytes of one env-step in this layout: state r/w, action r, t r/w, reward w,
        flags w (+ index / final state / side-effect words when they are separate outputs)."""
        extra = sum(4 for b in (self._index_ptr(), self._final, self._se_row) if b is not None)
        return 25 + extra

    # ---- conversions -------------------------------------------------------------------------------
    def pack(self, cells):
        """int8 device tensor [n_cells, n] -> int32 [n] packed words (device kernel)."""
        cells = torch.as_tensor(cells, device=self.device).to(torch.int8)
        n = cells.shape[1]
        ld = _round_up(n, 16)
        if ld != n or not cells.is_contiguous():
            pad = torch.zeros(cells.shape[0], ld, dtype=torch.int8, device=self.device)
            pad[:, :n] = cells
            cells = pad
        out = torch.empty(ld, dtype=torch.int32, device=self.device)
        _lib.check(self._lib.gc_pack_cells(self.device.index, n, ld, cells.shape[0], _ptr(cells), _ptr(out), self._stream()))
        return out[:n]

    def unpack(self, words):
        """int32/uint32 device tensor [n] packed words -> int8 [n_cells, n] levels (device kernel)."""
        words = torch.as_tensor(words, device=self.device)
        n = words.shape[0]
        ld = _round_up(n, 16)
        w = torch.zeros(ld, dtype=torch.int32, device=self.device)
        w[:n] = words.view(torch.int32) if words.dtype == torch.uint32 else words.to(torch.int32)
        out = torch.empty(self.n_cells, ld, dtype=torch.int8, device=self.device)
        _lib.check(self._lib.gc_unpack_cells(self.device.index, n, ld, self.n_cells, _ptr(w), _ptr(out), self._stream()))
        return out[:, :n]

    @property
    def state(self):
        """int8 [n_cells, num_envs] levels, unpacked on demand from the resident words."""
        return self.unpack(self._state[:self.num_envs])

    @property
    def packed_state(self):
        """int32 [num_envs] view of the resident state words (uint32 payload)."""
        return self._state[:self.num_envs]

    def set_state(self, cells, t=None, validate=True):
        cells = torch.as_tensor(cells, device=self.device)
        if cells.dim() == 2:
            cells = cells.to(torch.int8).reshape(self.n_cells, self.num_envs)
            if validate and (bool((cells < 0).any()) or bool((cells >= self.n_states).any())):
                raise ValueError(f"state levels must lie in [0, {self.n_states})")
            words = self.pack(cells)
        else:
            words = cells.to(torch.int32)
        self._state[:self.num_envs].copy_(words)
        if t is not None:
            self._t[:self.num_envs].copy_(torch.as_tensor(t, device=self.device).to(torch.int32))
        self._refresh_index()

    def _refresh_index(self):
        if self._index is not self._state:
            cells = self.unpack(self._state)
            _lib.check(self._lib.gc_encode(self.device.index, self.num_envs, self.ld, self.n_cells, self.n_states,
                                           _ptr(cells.contiguous()), _ptr(self._index), self._stream()))

    def materialise(self, i):
        word = int(self._state[i].item()) & 0xFFFFFFFF
        return tuple((word >> (2 * c)) & 3 for c in range(self.n_cells))

    # ---- checkpoint / resume -----------------------------------------------------------------------
    def load_state_dict(self, sd):
        if tuple(sd["meta"]) != (self.kind, self.num_envs, self.n_cells, self.n_states, self.env_seed, self.env_id_offset):
            raise ValueError("state_dict belongs to a differently configured env")
        self._state.copy_(sd["state"])
        self._t.copy_(sd["t"])
        if self._stats is not None and sd["stats"] is not None:
            self._stats.copy_(sd["stats"])
        torch.cuda.current_stream(self.device).synchronize()       # see CellularVectorEnv.load_state_dict
        _lib.check(self._lib.gc_set_global_step(self._h, int(sd["global_step"])))
        self._refresh_index()

    # ---- gymnasium.vector API ----------------------------------------------------------------------
    def reset(self, *, seed=None, options=None):
        """Reference reset() ignores its seed (cells3states3actions3.py:99); so does this one."""
        _lib.check(self._lib.gc_reset_packed(self._h, None, _ptr(self._state), _ptr(self._t), self._index_ptr(),
                                             self._stream()))
        self._reward.zero_()
        self._flags.zero_()
        if self._final is not None:
            self._final.copy_(self._state)
        if self._se_row is not None:
            # the reference's reset() info hard-codes row 0 = ('safe', 'silent', ...) (cells3states3actions3.py:102-109)
            row = [1] + [0] * (self.n_cells - 1) if self._cell_tables is None else self._cell_tables["reset_row"]
            self._se_row.fill_(sum(int(code) << (2 * j) for j, code in enumerate(row)))
        return self._v_obs, self._v_infos

    def reset_envs(self, mask):
        m = torch.zeros(self.ld, dtype=torch.uint8, device=self.device)
        m[:self.num_envs] = torch.as_tensor(mask, device=self.device).to(torch.uint8)
        _lib.check(self._lib.gc_reset_packed(self._h, _ptr(m), _ptr(self._state), _ptr(self._t), self._index_ptr(),
                                             self._stream()))

    def step(self, actions, replay_u=None):
        if replay_u is not None:
            raise ValueError("replayed uniforms are offered by the int8 layout (CellularVectorEnv) only")
        if isinstance(actions, np.ndarray) or (isinstance(actions, (tuple, list)) and len(actions)
                                                and isinstance(actions[0], np.ndarray)):
            return self._step_host(actions)
        self.step_device(actions)
        trunc = self._lazy_truncated() if self.max_episode_steps else self._false[:self.num_envs]
        return self._v_obs, self._v_reward, self._false[:self.num_envs], trunc, self._v_infos

    def _action_words(self, actions):
        """Device pointer of the packed action words for whatever form `actions` has."""
        if actions is None:
            return _ptr(self._actions)
        if isinstance(actions, (tuple, list)):
            actions = torch.stack([torch.as_tensor(a, device=self.device) for a in actions])
        elif not isinstance(actions, torch.Tensor):
            actions = torch.from_dlpack(actions)
        if actions.dim() == 2:                       # per-cell levels: pack on the device
            if actions.shape == (self.num_envs, self.n_cells) and self.num_envs != self.n_cells:
                actions = actions.t()
            if actions.shape != (self.n_cells, self.num_envs):
                raise ValueError(f"actions must have shape {(self.n_cells, self.num_envs)} or be packed words [{self.num_envs}]")
            actions = self.pack(actions.to(self.device))
        if actions.shape[0] not in (self.num_envs, self.ld):
            raise ValueError(f"packed actions must have {self.num_envs} entries")
        if actions.dtype == torch.uint32:
            actions = actions.view(torch.int32)
        if (actions.dtype == torch.int32 and actions.device == self.device and actions.is_contiguous()
                and actions.shape[0] == self.ld and actions.data_ptr() % 16 == 0):
            return C.c_void_p(actions.data_ptr())     # the caller's tensor has the kernel's layout: no copy
        if actions.data_ptr() != self._actions.data_ptr():
            self._actions[:self.num_envs].copy_(actions[:self.num_envs].to(self.device, torch.int32, non_blocking=True))
        return _ptr(self._actions)

    def step_device(self, actions=None, replay_u=None):
        """Launch one step on the current stream; no host synchronisation, no output marshalling."""
        if type(actions) is torch.Tensor and actions.dim() == 1:
            cache = self.__dict__.setdefault("_bound_cache", {})
            call = cache.get(actions.data_ptr())
            if call is None and len(cache) < 8 and actions.shape == (self.ld,) and actions.dtype == torch.int32 \
                    and actions.is_contiguous() and actions.device == self.device:
                call = cache[actions.data_ptr()] = (self.bind_step(actions), actions)
            if call is not None and call[1] is actions:
                call[0]()
                return
        a_ptr = self._action_words(actions)
        _lib.check(self._lib.gc_step_packed(
            self._h, 0, self.num_envs, a_ptr, _ptr(self._state), _ptr(self._t), _ptr(self._reward), self._index_ptr(),
            _ptr(self._flags), _ptr(self._final), _ptr(self._se_row), _ptr(self._stats), self._stream()))

    def _bind(self, actions):
        """Stores the pointer set of a full-shard step in a slot of the handle; returns the slot."""
        a = self._actions if actions is None else actions
        if a.dtype == torch.uint32:
            a = a.view(torch.int32)
        if a.dtype != torch.int32 or a.shape != (self.ld,) or not a.is_contiguous() or a.device != self.device:
            raise ValueError(f"bind_step needs a contiguous int32 tensor of {self.ld} packed action words on {self.device}")
        slot = getattr(self, "_n_bound", 0)
        if slot >= 16:
            raise RuntimeError("all 16 binding slots of the handle are in use")
        self._n_bound = slot + 1
        _lib.check(self._lib.gc_bind_step_packed(self._h, slot, _ptr(a), _ptr(self._state), _ptr(self._t),
                                                 _ptr(self._reward), self._index_ptr(), _ptr(self._flags),
                                                 _ptr(self._final), _ptr(self._se_row), _ptr(self._stats)))
        self.__dict__.setdefault("_bound_keepalive", []).append(a)
        return slot

    def bind_step(self, actions=None, stream=None):
        slot = self._bind(actions)
        check, dev, fn, h = _lib.check, self.device, self._lib.gc_step_bound, self._h
        if stream is not None:
            if stream.device != self.device:
                raise ValueError(f"stream lives on {stream.device}, the env on {self.device}")
            pinned = stream.cuda_stream

            def launch():
                rc = fn(h, slot, pinned)
                if rc:
                    check(rc)
            launch.stream, launch.slot = stream, slot
            return launch
        current_stream = torch.cuda.current_stream

        def launch():
            rc = fn(h, slot, current_stream(dev).cuda_stream)
            if rc:
                check(rc)
        launch.slot = slot
        return launch

    def rollout(self, n_steps, policy=None):
        """Fused K-step rollout (see `CellularVectorEnv.rollout`).  The rollout kernel keeps the per-cell levels in
        registers, so the packed state is unpacked for it and packed again afterwards (two extra launches per
        call, amortised over `n_steps` steps)."""
        n = self.num_envs
        if getattr(self, "_ro_ret", None) is None:
            self._ro_ret = torch.zeros(self.ld, dtype=torch.float32, device=self.device)
            self._ro_unsafe = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
            self._ro_index = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
        kind, ptab = _lib.POLICY_RANDOM, None
        if policy is not None:
            ptab = torch.as_tensor(policy, device=self.device).to(torch.int32).contiguous()
            if ptab.numel() != self.n_states ** self.n_cells:
                raise ValueError("policy must have one entry per tabular state")
            kind = _lib.POLICY_TABLE
        cells = self.unpack(self._state).contiguous()            # int8 [n_cells, ld]
        _lib.check(self._lib.gc_rollout(self._h, int(n_steps), kind, _ptr(ptab), _ptr(cells), _ptr(self._t),
                                        _ptr(self._ro_index), _ptr(self._ro_ret), _ptr(self._ro_unsafe), _ptr(self._stats),
                                        self._stream()))
        self._state.copy_(self.pack(cells))
        if self._index is not self._state:
            self._index.copy_(self._ro_index)
        return self._ro_ret[:n], self._ro_unsafe[:n]

    def collect(self, n_steps, policy=None, epsilon=0.0, next_obs=False):
        """Experience collection (see `CellularVectorEnv.collect`): the recording kernel takes the int8 layout,
        so the packed state is unpacked for it and packed again afterwards, as in `rollout()`."""
        if getattr(self, "_ro_index", None) is None:
            self._ro_index = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
        cells = self.unpack(self._state).contiguous()            # int8 [n_cells, ld]
        tr = self._collect(n_steps, policy, epsilon, next_obs, cells, self._ro_index)
        self._state.copy_(self.pack(cells))
        if self._index is not self._state:
            self._index.copy_(self._ro_index)
        return tr

    def collect_counts(self, n_steps, policy=None, epsilon=0.0, counts=None):
        """Experience counts (see `CellularVectorEnv.collect_counts`): the counting kernel takes the int8 layout, so the
        packed state is unpacked for it and packed again afterwards, as in `collect()`."""
        if getattr(self, "_ro_index", None) is None:
            self._ro_index = torch.zeros(self.ld, dtype=torch.int32, device=self.device)
        cells = self.unpack(self._state).contiguous()            # int8 [n_cells, ld]
        counts = self._collect_counts(n_steps, policy, epsilon, counts, cells, self._ro_index)
        self._state.copy_(self.pack(cells))
        if self._index is not self._state:
            self._index.copy_(self._ro_index)
        return counts

    # ---- views ---------------------------------------------------------------------------------------
    def _lazy_truncated(self):
        return (self._flags[:self.num_envs] & _lib.FLAG_TRUNCATED).ne(0)

    def _build_views(self):
        n = self.num_envs
        self._v_obs = self._state[:n]
        self._v_reward = self._reward[:n]
        env = self

        class _Infos(dict):
            """Zero-copy views; the entries derived from the flag byte are computed when they are read."""
            def __missing__(self, key):
                f = env._flags[:n]
                if key == "unsafe":
                    return (f & _lib.FLAG_UNSAFE).ne(0)
                if key == "truncated":
                    return (f & _lib.FLAG_TRUNCATED).ne(0)
                if key == "count":
                    return f >> _lib.FLAG_COUNT_SHIFT
                if key == "_final_obs":
                    return (f & _lib.FLAG_TRUNCATED).ne(0)
                raise KeyError(key)

        infos = _Infos(flags=self._flags[:n], time_step=self._t[:n], packed_state=self._state[:n])
        key = "tabular_state" if self.n_states ** self.n_cells <= 2 ** 31 else "tabular_state_u32"
        infos[key] = self._index[:n]
        if self._final is not None:
            infos["final_obs"] = self._final[:n]
        if self._se_row is not None:
            infos["side_effects_packed"] = self._se_row[:n]
        self._v_infos = infos

    def side_effects_incidence(self):
        return (self._flags[:self.num_envs] >> _lib.FLAG_COUNT_SHIFT).to(torch.float32) / self.n_cells

    def side_effects_row(self):
        """int8 [n_cells, num_envs] row 0 of the side-effects matrix (0 silent, 1 safe, 2 unsafe), unpacked."""
        if self._se_row is None:
            raise RuntimeError("emit_side_effects=False")
        return self.unpack(self._se_row[:self.num_envs])

    # ---- host path -----------------------------------------------------------------------------------
    def _alloc_host(self):
        ld = self.ld
        pin = lambda *shape, dtype: torch.zeros(*shape, dtype=dtype).pin_memory()
        self._host = {"actions": pin(ld, dtype=torch.int32), "state": pin(ld, dtype=torch.int32),
                      "reward": pin(ld, dtype=torch.float32), "flags": pin(ld, dtype=torch.uint8)}
        if self._index is not self._state:
            self._host["index"] = pin(ld, dtype=torch.int32)
        self._host_np = {k: v.numpy() for k, v in self._host.items()}

    @property
    def host_bytes_per_env_step(self):
        """(host-to-device, device-to-host) bytes the host path of step() moves per env: the action word
        in; the state word, the reward and the flag byte out (+ the index when it is a separate word)."""
        return 4, 9 + (4 if self._index is not self._state else 0)

    @property
    def host_action_buffer(self):
        """Pinned uint32 [num_envs] numpy view: fill it and call step(host_action_buffer)."""
        if self._host is None:
            self._alloc_host()
        return self._host_np["actions"][:self.num_envs].view(np.uint32)

    def _step_host(self, actions):
        if self._final is not None or self._se_row is not None:
            return self._step_host_extras(actions)
        if self._host is None:
            self._alloc_host()
        n, h = self.num_envs, self._host_np
        h_actions_ptr = _ptr(self._host["actions"])
        if isinstance(actions, (tuple, list)):
            actions = np.stack(actions)
        if actions.ndim == 2:
            if actions.shape == (n, self.n_cells) and n != self.n_cells:
                actions = actions.T
            if actions.shape != (self.n_cells, n):
                raise ValueError(f"actions must have shape {(self.n_cells, n)} or be packed words [{n}]")
            h["actions"][:n] = pack_host(actions).view(np.int32)
        elif actions.shape[0] == n:
            if actions.dtype.itemsize == 4 and actions.dtype.kind in "iu" and actions.flags.c_contiguous and n == self.ld:
                h_actions_ptr = C.c_void_p(actions.ctypes.data)      # caller's buffer (pinned or not), no staging copy
            elif actions.ctypes.data != h["actions"].ctypes.data:
                h["actions"][:n] = actions.astype(np.uint32, copy=False).view(np.int32)
        else:
            raise ValueError(f"packed actions must have {n} entries")
        torch.cuda.current_stream(self.device).synchronize()     # resident state must be settled
        H = self._host
        _lib.check(self._lib.gc_step_host_packed(
            self._h, h_actions_ptr, _ptr(H["state"]), _ptr(H["reward"]), _ptr(H.get("index")), _ptr(H["flags"]),
            _ptr(self._actions), _ptr(self._state), _ptr(self._t), _ptr(self._reward), self._index_ptr(),
            _ptr(self._flags), _ptr(self._stats), self.host_chunk_envs))
        flags = h["flags"][:n]
        state = h["state"][:n].view(np.uint32)
        infos = _HostInfos(flags, state, (h["index"] if "index" in h else h["state"])[:n].view(np.uint32), self.n_cells)
        if not hasattr(self, "_h_false"):
            self._h_false = np.zeros(n, np.bool_)
        trunc = (flags & _lib.FLAG_TRUNCATED).astype(np.bool_) if self.max_episode_steps else self._h_false
        return state, h["reward"][:n], self._h_false, trunc, infos


def _step_host_extras(self, actions):
    """Host path when final observations or side-effect rows were asked for: those are outputs of the device path
    (`gc_step_host_packed` carries state words, rewards and flags only), so the step is taken there and the
    arrays are copied to the host one by one -- correct, not pipelined."""
    n = self.num_envs
    if isinstance(actions, (tuple, list)):
        actions = np.stack(actions)
    if actions.ndim == 2:
        if actions.shape == (n, self.n_cells) and n != self.n_cells:
            actions = actions.T
        actions = pack_host(actions)
    self.step_device(torch.from_numpy(np.ascontiguousarray(actions).astype(np.uint32, copy=False).view(np.int32)).to(self.device))
    flags = self._flags[:n].cpu().numpy()
    state = self._state[:n].cpu().numpy().view(np.uint32)
    infos = _HostInfos(flags, state, self._index[:n].cpu().numpy().view(np.uint32), self.n_cells)
    if self._final is not None:
        infos["final_obs"] = self._final[:n].cpu().numpy().view(np.uint32)
        infos["_final_obs"] = (flags & _lib.FLAG_TRUNCATED).astype(np.bool_)
    if self._se_row is not None:
        infos["side_effects_packed"] = self._se_row[:n].cpu().numpy().view(np.uint32)
    false = np.zeros(n, np.bool_)
    trunc = (flags & _lib.FLAG_TRUNCATED).astype(np.bool_) if self.max_episode_steps else false
    return state, self._reward[:n].cpu().numpy(), false, trunc, infos


PackedCellularVectorEnv._step_host_extras = _step_host_extras


class _HostInfos(dict):
    """infos of a host-path step: zero-copy views of the pinned mirrors; what derives from the flag byte or
    needs unpacking is computed when it is read (`unsafe`, `count`, `observation`)."""

    def __init__(self, flags, state, index, n_cells):
        super().__init__(flags=flags, packed_state=state, tabular_state=index)
        self._n_cells = n_cells

    def __missing__(self, key):
        f = self["flags"]
        if key == "unsafe":
            return (f & _lib.FLAG_UNSAFE).astype(np.bool_)
        if key == "truncated":
            return (f & _lib.FLAG_TRUNCATED).astype(np.bool_)
        if key == "count":
            return f >> _lib.FLAG_COUNT_SHIFT
        if key == "observation":          # the reference-shaped observation: int8 [n_cells, num_envs]
            return unpack_host(self["packed_state"], self._n_cells)
        raise KeyError(key)
