"""The Philox draws that decide every random event of the step, rollout and collect kernels, restated in numpy from
DESIGN.md §4 (RNG table) on top of `_collect_oracle.philox`: a derivation independent of both the kernels and the
oracle's `draw_uniform`.  Everything random reduces to a compare of a 32-bit value v against ceil(p * 2^32), so for
one chosen draw v the probabilities v * 2^-32 (must not fire) and (v + 1) * 2^-32 (must fire) put that compare at
its exact boundary; `search` finds draws of a wanted shape.

  narrow cellular draw (<= 4 cells), cell c, env g, counter T:  philox(g, T, c // 4)[c % 4]
  wide cellular draw (> 4 cells):   half (c % 8) of philox(g, T, c // 8) << 16  |  philox(g, T, 0x20000000 + c)[0] >> 16
                                    (half h = the low half of word h // 2 for even h, the high half for odd h)
  grid-world dispersal trigger:     philox(g // 4, T, 0)[g % 4]
  collect explore test:             philox(g // 4, G, 0x50000000)[g % 4]  (G = the global step)
T is the episode step of the env under rng_episodic, else the global step.  The cellular draws take T as a scalar or as
a per-env array [n] (episodic envs at different episode steps).
"""
from types import SimpleNamespace

import numpy as np

from _collect_oracle import _words, philox

NARROW_CELLS = 4
NOISE_LOW_STREAM = 0x20000000
EXPLORE_STREAM = 0x50000000
_LO = np.uint64(0xFFFFFFFF)


def _ids(first, n):
    g = np.arange(n, dtype=np.uint64) + np.uint64(first)
    return g & _LO, g >> np.uint64(32)


def wide_tops(seed, n_cells, first, n, T):
    """uint32 [n_cells, n]: top halves of the wide draws of envs first .. first + n - 1 at counter T (scalar or [n])."""
    lo, hi = _ids(first, n)
    blocks = [np.stack(philox(lo, hi, T, b, seed)) for b in range((n_cells + 7) // 8)]
    return np.stack([(blocks[c // 8][(c % 8) // 2] >> np.uint32(16 * (c % 2))) & np.uint32(0xFFFF)
                     for c in range(n_cells)])


def wide_lows(seed, cells, first, n, T):
    """uint32 [len(cells), n]: low halves of the wide draws of the given cells (T scalar or [n])."""
    lo, hi = _ids(first, n)
    return np.stack([philox(lo, hi, T, NOISE_LOW_STREAM + c, seed)[0] >> np.uint32(16) for c in cells])


def cell_draws(seed, n_cells, first, n, T):
    """uint32 [n_cells, n]: the 32-bit noise draw of every cell of envs first .. first + n - 1 at counter T (scalar or
    [n])."""
    if n_cells <= NARROW_CELLS:
        lo, hi = _ids(first, n)
        return np.stack(philox(lo, hi, T, 0, seed))[:n_cells]
    return (wide_tops(seed, n_cells, first, n, T) << np.uint32(16)) | wide_lows(seed, range(n_cells), first, n, T)


def grouped_words(seed, first, n, T, stream):
    """uint32 [n]: word g % 4 of philox(g // 4, T, stream) for g = first .. first + n - 1 (first a multiple of 4)."""
    batch = SimpleNamespace(n=int(n), cfg=SimpleNamespace(seed=seed, env_id_offset=int(first)))
    return _words(batch, np.uint64(T), stream)


def grid_triggers(seed, first, n, T):
    return grouped_words(seed, first, n, T, 0)


def explore_words(seed, first, n, G):
    return grouped_words(seed, first, n, G, EXPLORE_STREAM)


def top(v):
    return int(v) >> 16


def low(v):
    return int(v) & 0xFFFF


def search(draws, pred, first=0, n=1 << 18, chunk=1 << 16, limit=16):
    """Up to `limit` candidates (g, c, v) with pred(v) true (pred works on uint32 arrays), in order of env id, among
    envs first .. first + n - 1.  `draws(first, n)` returns the uint32 [rows, n] draws of those envs (row = cell)."""
    out = []
    for f in range(first, first + n, chunk):
        d = np.atleast_2d(draws(f, chunk))
        rows, cols = np.nonzero(pred(d))
        for j in np.argsort(cols, kind="stable"):
            out.append((f + int(cols[j]), int(rows[j]), int(d[rows[j], cols[j]])))
            if len(out) >= limit:
                return out
    return out


def search_wide(seed, n_cells, T, top_is=None, low_is=None, first=0, n=1 << 18, limit=16):
    """Wide draws whose top half equals `top_is` and/or whose low half equals `low_is` (searching only the half that
    is constrained, then completing the hits)."""
    if top_is is not None:
        hits = search(lambda f, m: wide_tops(seed, n_cells, f, m, T), lambda d: d == top_is, first, n, limit=limit * 4)
        hits = [(g, c, (t << 16) | int(wide_lows(seed, [c], g, 1, T)[0, 0])) for g, c, t in hits]
    else:
        hits = search(lambda f, m: wide_lows(seed, range(n_cells), f, m, T), lambda d: d == low_is, first, n, limit=limit * 4)
        hits = [(g, c, (int(wide_tops(seed, n_cells, g, 1, T)[c, 0]) << 16) | lo) for g, c, lo in hits]
    return [h for h in hits if low_is is None or low(h[2]) == low_is][:limit]
