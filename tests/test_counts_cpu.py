"""CPU checks of experience counts (gc_collect_counts): the ctypes struct against the header, and argument validation
before any CUDA call."""
import ctypes as C
import os
import re

from conftest import REPO


def test_counts_struct_matches_header():
    from gym_cellular_b200 import _lib
    header = open(os.path.join(REPO, "include", "gym_cellular_b200.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} gc_counts;", header).group(1)
    fields = re.findall(r"^\s*\w+\s*\*?\s*(\w+);", body, re.M)
    assert fields == [f[0] for f in _lib.GcCounts._fields_]
    # uint32 + padding + 5 pointers on LP64
    assert C.sizeof(_lib.GcCounts) == 8 + 5 * C.sizeof(C.c_void_p) == 48
    assert [getattr(_lib.GcCounts, f).offset for f in fields] == [0, 8, 16, 24, 32, 40]
    assert "gc_collect_counts" in _lib.EXPORTS


def test_collect_counts_rejects_null_handle():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    L = _lib.load()
    cs = _lib.GcCounts(C.sizeof(_lib.GcCounts))
    assert L.gc_collect_counts(None, 4, _lib.POLICY_RANDOM, None, 0.0, None, None, None, C.byref(cs), None, None) == _lib.ERR_INVALID
    assert b"NULL" in L.gc_last_error()
    assert L.gc_collect_counts(None, 4, _lib.POLICY_RANDOM, None, 0.0, None, None, None, None, None, None) == _lib.ERR_INVALID


def test_counts_is_exported():
    import gym_cellular_b200 as B
    assert "Counts" in B.__all__
    assert B.Counts._fields == ("visits", "next", "reward_q24", "unsafe", "cell_next")
