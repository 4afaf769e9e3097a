"""ctypes binding of libgymcellular_b200_plan.so (include/gym_cellular_b200_plan.h), the planner library.

There is no CPU fallback: if the CUDA library has not been built, loading it fails loudly.  Build it with
`python -m gym_cellular_b200.build` (or `__graft_entry__.build()`), which builds it next to the env library.
"""
import ctypes as C
import os

from ._lib import ERR_INVALID, GcError, OK  # noqa: F401  (the planner returns the env library's gc_status codes)

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.environ.get("GC_B200_LIB_DIR") or os.path.join(_PKG, "lib"), "libgymcellular_b200_plan.so")

ABI_VERSION = 1
MAX_STATES = 4096
MAX_STATE_ACTIONS = 1 << 17
EXPORTS = ["gcp_abi_version", "gcp_last_error", "gcp_value_iteration"]


class GcpModel(C.Structure):
    """gcp_model: the models of one call -- the int64 counts (visits, next, reward_q24) or the float64 (P, R)."""
    _fields_ = [("struct_size", C.c_uint32), ("n_models", C.c_int32), ("n_states", C.c_int32), ("n_actions", C.c_int32),
                ("visits", C.c_void_p), ("next", C.c_void_p), ("reward_q24", C.c_void_p), ("P", C.c_void_p),
                ("R", C.c_void_p)]


_lib = None


def load():
    """Returns the loaded planner library; raises ImportError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the planner's CUDA library has not been built and there is no CPU "
            "fallback.  Run `python -m gym_cellular_b200.build` (needs nvcc).")
    L = C.CDLL(LIB_PATH)
    L.gcp_abi_version.restype = C.c_int
    L.gcp_last_error.restype = C.c_char_p
    L.gcp_value_iteration.argtypes = [C.c_int, C.POINTER(GcpModel), C.c_double, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p]
    if L.gcp_abi_version() != ABI_VERSION:
        raise ImportError(f"ABI version mismatch: planner library {L.gcp_abi_version()} != binding {ABI_VERSION}")
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise GcError(rc, load().gcp_last_error().decode())
