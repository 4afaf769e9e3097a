"""Grouped experience counts (gc_collect_counts_grouped, `zero_counts(groups=)`) without a device: the export and its
ctypes signature against the header, the refusal of a NULL handle, and the shapes and 2^31 limits of grouped tables."""
import ctypes as C
import os
import re
from types import SimpleNamespace

import pytest

from conftest import REPO

torch = pytest.importorskip("torch")

_CTYPE = {"int32_t": C.c_int32, "double": C.c_double}


def _prototype(name):
    header = open(os.path.join(REPO, "include", "gym_cellular_b200.h")).read()
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", header)
    assert m, name
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_grouped_entry_is_exported_with_the_header_signature():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    assert "gc_collect_counts_grouped" in _lib.EXPORTS and _lib.ABI_VERSION == 2
    L = _lib.load()
    fn = L.gc_collect_counts_grouped
    params = _prototype("gc_collect_counts_grouped")
    assert len(fn.argtypes) == len(params) == 10
    for p, t in zip(params, fn.argtypes):
        if "*" in p:
            assert t in (C.c_void_p, C.POINTER(_lib.GcCounts)), p
            assert (t is C.POINTER(_lib.GcCounts)) == p.startswith("const gc_counts"), p
        else:
            assert t is _CTYPE[p.split()[0]], p
    # the same arguments as gc_collect_counts without the policy kind
    assert _prototype("gc_collect_counts")[:2] + _prototype("gc_collect_counts")[3:] == params


def test_grouped_entry_rejects_a_null_handle():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    L = _lib.load()
    cs = _lib.GcCounts(C.sizeof(_lib.GcCounts))
    assert L.gc_collect_counts_grouped(None, 4, None, 0.0, None, None, None, C.byref(cs), None, None) == _lib.ERR_INVALID
    assert b"NULL" in L.gc_last_error()


# ---------------------------------------------------------------------------------------------
# zero_counts(groups=): CellularVectorEnv.zero_counts on a stand-in env with CPU tensors

def _env(kind="cellular", C_=3, S=3, A=3):
    joint = (400, 25) if kind == "gridworld" else (S ** C_, A ** C_)
    return SimpleNamespace(kind=kind, n_cells=C_, n_states=S, n_actions=A, device=torch.device("cpu"),
                           _joint_sizes=lambda: joint)


def _zero(env, **kw):
    from gym_cellular_b200.vector_env import CellularVectorEnv
    return CellularVectorEnv.zero_counts(env, **kw)


def test_zero_counts_groups_shapes():
    z = _zero(_env(), groups=5)
    assert z.visits.shape == (5, 27, 27) and z.next.shape == (5, 27, 27, 27) and z.reward_q24.shape == (5, 27, 27)
    assert z.unsafe.shape == (5, 27, 27) and z.cell_next.shape == (5, 3, 3, 3, 3)
    assert all(t.dtype == torch.int64 and t.is_contiguous() and not t.any() for t in z)
    one = _zero(_env(), groups=1)
    assert one.visits.shape == (1, 27, 27)
    plain = _zero(_env())
    assert plain.visits.shape == (27, 27) and plain.cell_next.shape == (3, 3, 3, 3)
    zt = _zero(_env(), groups=4, transitions=False)
    assert zt.next is None and zt.visits.shape == (4, 27, 27)
    zj = _zero(_env(), groups=4, joint=False)
    assert zj.visits is None and zj.next is None and zj.cell_next.shape == (4, 3, 3, 3, 3)
    zg = _zero(_env("gridworld"), groups=3, transitions=False)
    assert zg.visits.shape == (3, 400, 25) and zg.next is None and zg.cell_next is None


def test_counts_group_is_a_view_of_one_group():
    z = _zero(_env(), groups=3, transitions=False)
    g = z.group(1)
    assert type(g) is type(z) and g.next is None and g.visits.shape == (27, 27) and g.cell_next.shape == (3, 3, 3, 3)
    g.visits[2, 3] = 7
    assert int(z.visits[1, 2, 3]) == 7 and int(z.visits.sum()) == 7


def test_zero_counts_groups_limits():
    """P times each table's size must not pass 2^31 (checked before anything is allocated)."""
    env = _env(C_=5, S=4, A=2)                   # nS nA = 2^15, nS nA nS = 2^25: 'next' of 64 groups is 2^31 exactly
    assert _zero(env, groups=2).next.shape == (2, 1024, 32, 1024)
    with pytest.raises(ValueError, match="65 groups x 1024 states x 32 actions .* or transitions=False or fewer groups"):
        _zero(env, groups=65)
    with pytest.raises(ValueError, match="joint=False or fewer groups"):        # (state, action) tables: 2^16 groups
        _zero(env, groups=2 ** 16 + 1, transitions=False)
    with pytest.raises(ValueError, match="per-cell"):                            # 2^10 entries a group
        _zero(_env(C_=16, S=4, A=4), groups=2 ** 21 + 1, joint=False)
    with pytest.raises(ValueError, match="joint=False"):                         # ungrouped: unchanged
        _zero(_env(C_=16, S=4, A=4))
    for bad in (0, -1, 2.0, True, "3"):
        with pytest.raises(ValueError, match="groups must be an int"):
            _zero(_env(), groups=bad)
