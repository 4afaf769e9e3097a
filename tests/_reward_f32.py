"""The float32 reward arithmetic of the cellular kernels restated in numpy: the exact bits of the pre-log reward.

The float64 table reference (_table_reference.py) sums the cells' rewards exactly; the kernels add float32 table
entries in a fixed order, and the order and grouping decide the rounding.  The LUT builders (gc_tables.cu) and the
kernels give, per family (the library is built without --use_fast_math, so every FADD rounds to nearest like numpy's
float32 addition):

  pair     cell_pair_kernel, cell_packed_kernel, both many-step kernels, cell_rollout_kernel (rollout, collect,
           counts), cell_pair8_kernel without noise.  Entry k = f32(f64(r_2k) + f64(r_2k+1)), an odd last cell the
           single entry f32(r_C-1); the entries added in float32 in pair order.
  single   cell_step_kernel (generic) and cell_pair8_kernel with noise: the entries f32(r_c) added in cell order.

r_c is reward_noisy[s][a] where cell c's draw fired (and draws[s][a] is set), else reward[s][a].  A sum that is zero
is +0.0: the LUT builders store +0.0 for an entry that compares equal to zero, and float32 sums of non-negative-zero
terms are never -0.0.
"""
import numpy as np

PAIR, SINGLE = "pair", "single"


def cell_rewards(ref):
    """float32 [C, n]: the reward of each cell in the last step of TableEnv `ref`, as the device tables hold it."""
    s, a, fire = ref.last_s, ref.last_a, ref.last_fire
    r = np.where(fire, ref.reward_noisy[s, a], ref.reward[s, a])
    return r.astype(np.float32)


def entries(cell, family):
    """float32 [L, n]: the table entries a kernel of `family` adds for per-cell rewards `cell` [C, n]."""
    cell = np.asarray(cell, np.float32)
    if family == SINGLE:
        out = list(cell)
    else:
        assert family == PAIR, family
        C = cell.shape[0]
        out = [(cell[2 * k].astype(np.float64) + cell[2 * k + 1].astype(np.float64)).astype(np.float32)
               for k in range(C // 2)]
        if C % 2:
            out.append(cell[C - 1])
    # +0.0 for an entry equal to zero (gc_tables.cu)
    return np.stack([np.where(e == 0, np.float32(0.0), e) for e in out])


def prelog(ref, family):
    """float32 [n]: the pre-log reward of every env of the last step of `ref` in kernel family `family`."""
    acc = np.zeros(ref.n, np.float32)
    for e in entries(cell_rewards(ref), family):
        acc = acc + e
    return acc


def bits(x):
    return np.ascontiguousarray(x, np.float32).view(np.uint32)


def q24(x):
    """int64 [n]: rint(reward * 2^24) per env, as the reward statistic adds it."""
    return np.rint(np.asarray(x, np.float32).astype(np.float64) * 2.0 ** 24).astype(np.int64)


def sum_bound(ref):
    """The float32 rounding bound of a C-term sum against the exact float64 sum of the float32 cell rewards."""
    return (ref.C + 1) * 2.0 ** -24 * ref.reward_abs + 2.0 ** -149
