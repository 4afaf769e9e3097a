"""CPU checks of experience collection (gc_collect): the ctypes record struct against the header, argument
validation before any CUDA call, and the test-side restatement of the epsilon-greedy draws (tests/_collect_oracle.py)."""
import ctypes as C
import os
import re

import numpy as np
from scipy import stats as sps

import _collect_oracle as CO
from conftest import REPO


def test_record_struct_matches_header():
    from gym_cellular_b200 import _lib
    header = open(os.path.join(REPO, "include", "gym_cellular_b200.h")).read()
    body = re.search(r"typedef struct \{([^}]*)\} gc_record;", header).group(1)
    fields = re.findall(r"^\s*\w+\s*\*?\s*(\w+);", body, re.M)
    assert fields == [f[0] for f in _lib.GcRecord._fields_]
    # uint32 + padding + 5 pointers on LP64
    assert C.sizeof(_lib.GcRecord) == 8 + 5 * C.sizeof(C.c_void_p) == 48
    assert [getattr(_lib.GcRecord, f).offset for f in fields] == [0, 8, 16, 24, 32, 40]


def test_collect_rejects_null_handle():
    import __graft_entry__
    __graft_entry__.build()
    from gym_cellular_b200 import _lib
    L = _lib.load()
    rec = _lib.GcRecord(C.sizeof(_lib.GcRecord))
    assert L.gc_collect(None, 4, _lib.POLICY_RANDOM, None, 0.0, None, None, None, C.byref(rec), None, None) == _lib.ERR_INVALID
    assert b"NULL" in L.gc_last_error()


def test_numpy_philox_matches_the_oracle():
    from oracle import oracle as O
    rng = np.random.default_rng(7)
    for _ in range(20):
        ctr = rng.integers(0, 2 ** 32, 4, dtype=np.uint64)
        seed = int(rng.integers(0, 2 ** 63))
        ref = O.philox4x32_10(ctr.astype(np.uint32), [seed & 0xFFFFFFFF, seed >> 32])
        assert [int(w) for w in CO.philox(*ctr, seed)] == [int(x) for x in ref]


def test_epsilon_quarter_fraction_and_global_step():
    """ε = 0.25: the non-greedy fraction is ε (1 - 1/A^C); the draws follow the global step, not the episode step."""
    from oracle import oracle as O
    pol = np.zeros(27, np.int32)
    o = O.OracleEnv(n_envs=4096, seed=12, rng_episodic=True, max_episode_steps=16)
    _, act, _, _ = CO.collect(o, 32, pol, 0.25)
    p, N = 0.25 * (1 - 1 / 27), act.size
    assert abs((act != 0).mean() - p) < 5 * np.sqrt(p * (1 - p) / N)
    assert ((act[:16] != 0) != (act[16:] != 0)).any(axis=0).mean() > 0.99


def _chi2_uniform(counts):
    exp = np.full(len(counts), counts.sum() / len(counts))
    return sps.chisquare(counts, exp).pvalue


def test_oracle_epsilon_zero_is_the_table_policy():
    from oracle import oracle as O
    pol = np.random.default_rng(1).integers(0, 27, 27).astype(np.int32)
    o = O.OracleEnv(n_envs=1001, noise=True, seed=3, rng_episodic=True, max_episode_steps=6, reward="nonlinear_rp")
    ref = O.OracleEnv(n_envs=1001, noise=True, seed=3, rng_episodic=True, max_episode_steps=6, reward="nonlinear_rp")
    obs, act, rew, flags = CO.collect(o, 9, pol, 0.0)
    assert (act == pol[obs]).all()
    ret, uns = ref.rollout(9, pol)
    np.testing.assert_allclose(rew.sum(0), ret)
    assert ((flags & 1).sum(0) == uns).all() and (o.state == ref.state).all() and (o.t == ref.t).all()


def test_oracle_epsilon_one_is_uniform():
    from oracle import oracle as O
    pol = np.zeros(27, np.int32)
    o = O.OracleEnv(n_envs=4096, seed=11)
    _, act, _, _ = CO.collect(o, 8, pol, 1.0)
    assert _chi2_uniform(np.bincount(act.ravel(), minlength=27)) > 1e-4
    g = O.OracleEnv(kind="gridworld", n_envs=4096, seed=11)
    _, act, _, _ = CO.collect(g, 8, np.zeros(400, np.int32), 1.0)
    codes = [4 + 5 * p for p in range(4)] + [p + 20 for p in range(4)]      # (4, pos) and (pos, 4)
    counts = np.bincount(act.ravel(), minlength=25)
    assert counts[codes].sum() == act.size
    assert _chi2_uniform(counts[codes]) > 1e-4
