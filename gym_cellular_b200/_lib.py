"""ctypes binding of libgymcellular_b200.so (include/gym_cellular_b200.h).

There is no CPU fallback: if the CUDA library has not been built, importing the compute path fails
loudly.  Build it with `python -m gym_cellular_b200.build` (or `__graft_entry__.build()`).
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# GC_B200_LIB_DIR: directory of an alternative in-tree build (A/B runs of tuning variants, gym_cellular_b200/build.py)
LIB_PATH = os.path.join(os.environ.get("GC_B200_LIB_DIR") or os.path.join(_PKG, "lib"), "libgymcellular_b200.so")

ABI_VERSION = 2
KIND_CELLULAR, KIND_GRIDWORLD = 0, 1
F_NOISE, F_RNG_EPISODIC, F_REWARD_LOG2, F_GENERIC_KERNEL = 1, 4, 16, 32
MAX_CELLS, MAX_LEVELS, N_STATS = 16, 8, 8
STAT_STEPS, STAT_UNSAFE, STAT_COUNT, STAT_TRUNCATED, STAT_REWARD_Q24 = range(5)
OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_ACTION = 0, -1, -2, -3, -4
POLICY_RANDOM, POLICY_TABLE, POLICY_TABLE_STACK = 0, 1, 2

EXPORTS = ["gc_abi_version", "gc_last_error", "gc_create", "gc_destroy", "gc_set_tables", "gc_set_final_obs",
           "gc_set_global_step", "gc_get_global_step", "gc_sync_global_step", "gc_launch_count", "gc_reset", "gc_step",
           "gc_bind_step", "gc_step_bound", "gc_step_many", "gc_prepare_step_many", "gc_step_host", "gc_rollout", "gc_collect", "gc_collect_counts", "gc_poll_status", "gc_encode",
           "gc_decode", "gc_encode_mixed", "gc_decode_mixed", "gc_reset_packed", "gc_step_packed", "gc_bind_step_packed",
           "gc_step_host_packed", "gc_pack_cells", "gc_unpack_cells", "gc_compressible_supported", "gc_alloc_compressible",
           "gc_free_compressible", "gc_is_compressible", "gc_set_policy_stack", "gc_collect_counts_grouped"]
FLAG_UNSAFE, FLAG_TRUNCATED, FLAG_COUNT_SHIFT = 1, 2, 2


class GcConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("kind", C.c_int32), ("device", C.c_int32),
                ("n_cells", C.c_int32), ("n_states", C.c_int32), ("n_actions", C.c_int32),
                ("max_episode_steps", C.c_int32), ("flags", C.c_uint32),
                ("n_envs", C.c_int64), ("ld", C.c_int64), ("env_id_offset", C.c_int64),
                ("seed", C.c_uint64), ("noise_prob", C.c_double), ("dispersal_prob", C.c_double)]


class GcCellTables(C.Structure):
    _fields_ = [("move", C.c_void_p), ("noisy", C.c_void_p), ("draws", C.c_void_p),
                ("reward", C.c_void_p), ("side_effects", C.c_void_p), ("counted", C.c_void_p),
                ("initial_state", C.c_void_p), ("reward_noisy", C.c_void_p), ("radix", C.c_void_p)]


class GcRecord(C.Structure):
    """gc_record: step-major [n_steps][ld] device arrays of gc_collect (NULL = not recorded)."""
    _fields_ = [("struct_size", C.c_uint32), ("obs", C.c_void_p), ("action", C.c_void_p), ("reward", C.c_void_p),
                ("flags", C.c_void_p), ("next_obs", C.c_void_p)]


class GcCounts(C.Structure):
    """gc_counts: int64 device count tables of gc_collect_counts (NULL = not counted)."""
    _fields_ = [("struct_size", C.c_uint32), ("visits", C.c_void_p), ("next", C.c_void_p), ("reward_q24", C.c_void_p),
                ("unsafe", C.c_void_p), ("cell_next", C.c_void_p)]


class GcError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libgymcellular_b200 error {code}: {message}")
        self.code = code
        self.message = message


_lib = None


def load():
    """Returns the loaded library; raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no CPU "
            "fallback.  Run `python -m gym_cellular_b200.build` (needs nvcc).")
    L = C.CDLL(LIB_PATH)
    vp, i64 = C.c_void_p, C.c_int64
    L.gc_abi_version.restype = C.c_int
    L.gc_last_error.restype = C.c_char_p
    L.gc_create.argtypes = [C.POINTER(GcConfig), C.POINTER(vp)]
    L.gc_destroy.argtypes = [vp]
    L.gc_set_tables.argtypes = [vp, C.POINTER(GcCellTables)]
    L.gc_set_final_obs.argtypes = [vp, vp]
    L.gc_set_global_step.argtypes = [vp, i64]
    L.gc_get_global_step.argtypes = [vp]
    L.gc_get_global_step.restype = i64
    L.gc_sync_global_step.argtypes = [vp, vp]
    L.gc_launch_count.argtypes = [vp]
    L.gc_launch_count.restype = i64
    L.gc_reset.argtypes = [vp] * 6
    L.gc_step.argtypes = [vp, i64, i64] + [vp] * 13
    L.gc_bind_step.argtypes = [vp, C.c_int32] + [vp] * 11
    L.gc_step_bound.argtypes = [vp, C.c_int32, vp]
    L.gc_step_host.argtypes = [vp] * 21 + [i64]
    L.gc_rollout.argtypes = [vp, C.c_int32, C.c_int32] + [vp] * 8
    L.gc_collect.argtypes = [vp, C.c_int32, C.c_int32, vp, C.c_double, vp, vp, vp, C.POINTER(GcRecord), vp, vp]
    L.gc_collect_counts.argtypes = [vp, C.c_int32, C.c_int32, vp, C.c_double, vp, vp, vp, C.POINTER(GcCounts), vp, vp]
    L.gc_collect_counts_grouped.argtypes = [vp, C.c_int32, vp, C.c_double, vp, vp, vp, C.POINTER(GcCounts), vp, vp]
    L.gc_poll_status.argtypes = [vp, vp]
    L.gc_encode.argtypes = [C.c_int, i64, i64, C.c_int32, C.c_int32, vp, vp, vp]
    L.gc_decode.argtypes = [C.c_int, i64, i64, C.c_int32, C.c_int32, vp, vp, vp]
    i32 = C.c_int32
    L.gc_step_many.argtypes = [vp, vp, i32, i32, vp]
    L.gc_prepare_step_many.argtypes = [vp, vp, i32]
    L.gc_encode_mixed.argtypes = [C.c_int, i64, i64, i32, vp, vp, vp, vp, vp]
    L.gc_decode_mixed.argtypes = [C.c_int, i64, i64, i32, vp, vp, vp, vp, vp]
    L.gc_reset_packed.argtypes = [vp] * 6
    L.gc_step_packed.argtypes = [vp, i64, i64] + [vp] * 10
    L.gc_bind_step_packed.argtypes = [vp, i32] + [vp] * 9
    L.gc_step_host_packed.argtypes = [vp] * 13 + [i64]
    L.gc_pack_cells.argtypes = [C.c_int, i64, i64, i32, vp, vp, vp]
    L.gc_unpack_cells.argtypes = [C.c_int, i64, i64, i32, vp, vp, vp]
    L.gc_compressible_supported.argtypes = [C.c_int]
    L.gc_alloc_compressible.argtypes = [C.c_size_t, C.c_int, vp]
    L.gc_alloc_compressible.restype = vp
    L.gc_free_compressible.argtypes = [vp, C.c_size_t, C.c_int, vp]
    L.gc_free_compressible.restype = None
    L.gc_is_compressible.argtypes = [vp]
    L.gc_set_policy_stack.argtypes = [vp, vp, i32]
    if L.gc_abi_version() != ABI_VERSION:
        raise ImportError(f"ABI version mismatch: library {L.gc_abi_version()} != binding {ABI_VERSION}")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise GcError(rc, load().gc_last_error().decode())
