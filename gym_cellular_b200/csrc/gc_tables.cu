// Host-side builders of the lookup tables the fast kernels stage into shared memory.
// (Compiled by nvcc with the rest of the library; no device code here.)
#include <cstring>

#include "gc_internal.h"

// ---------------------------------------------------------------------------------------------
// Grid world: closed form of grid_world.py:119-179 on the reference's own cellular codes
// (grid_world.py:349-359): code_j = T_j + 4 * pos_j, T_j = tree bits (bit 0 = tree at (1,0),
// bit 1 = tree at (0,0)), pos_j = row*2+col of the agent or 4 if it is not in jurisdiction j.
//   site(p): tree bit under position p  (p=2 -> (1,0) -> bit 0, p=0 -> (0,0) -> bit 1, else none)
//   1. all trees regrow (N_j = 3)                                                     :122-127
//   2. the agent (first jurisdiction J holding one) moves to (G, q): its own jurisdiction if the
//      action names a position there, else the first jurisdiction whose action does   :128-137
//   3. a dead tree under the origin stays dead; a live tree under the destination dies :141-151
//   4. jurisdictions that were barren BEFORE the step stay barren                      :154-158
//   reward = trees that died (pre-step minus post-step, clipped at 0)                  :30-39
//   side effects row 0 = ('safe' if N_0>0 and N_1>0, 'safe' if N_0>0); never 'unsafe'  :168-179
// Seed dispersal (:160-162) is the only stochastic part and is applied in the kernel on top of the
// table entry.  All 20 x 20 x 5 x 5 code combinations are tabulated, including states the
// reference never reaches (no agent / two agents), with the reference's behaviour for them.
static uint32_t site_of(uint32_t p) { return (p == 0u ? 2u : 0u) | (p == 2u ? 1u : 0u); }

void gc_build_grid_lut(uint32_t *lut)
{
    for (uint32_t c1 = 0; c1 < 20; ++c1)
        for (uint32_t c0 = 0; c0 < 20; ++c0)
            for (uint32_t a1 = 0; a1 < 5; ++a1)
                for (uint32_t a0 = 0; a0 < 5; ++a0) {
                    const uint32_t T0 = c0 & 3u, T1 = c1 & 3u, P0 = c0 >> 2, P1 = c1 >> 2;
                    const bool has0 = P0 < 4u, has1 = P1 < 4u, agent = has0 || has1;
                    const uint32_t J = has0 ? 0u : 1u, p = has0 ? P0 : P1, TJ = has0 ? T0 : T1;
                    const uint32_t aJ = J ? a1 : a0;
                    uint32_t G = J, q = p, bad = 0;
                    if (aJ < 4u) { G = J; q = aJ; }
                    else if (a0 < 4u) { G = 0u; q = a0; }
                    else if (a1 < 4u) { G = 1u; q = a1; }
                    else if (agent) bad = 1u;                       // reference: KeyError('position'), :143
                    uint32_t N0 = 3u, N1 = 3u;
                    if (agent) {
                        const uint32_t TG = G ? T1 : T0;
                        const uint32_t kill_origin = site_of(p) & ~TJ, kill_dest = site_of(q) & TG;
                        if (J == 0u) N0 &= ~kill_origin; else N1 &= ~kill_origin;
                        if (G == 0u) N0 &= ~kill_dest; else N1 &= ~kill_dest;
                    }
                    const uint32_t nb = (T0 == 0u) + (T1 == 0u);
                    if (T0 == 0u) N0 = 0u;
                    if (T1 == 0u) N1 = 0u;
                    const uint32_t reward = __builtin_popcount(T0 & ~N0) + __builtin_popcount(T1 & ~N1);
                    const uint32_t nc0 = N0 + 4u * ((agent && G == 0u) ? q : 4u);
                    const uint32_t nc1 = N1 + 4u * ((agent && G == 1u) ? q : 4u);
                    const uint32_t se0 = (N0 > 0u && N1 > 0u) ? 1u : 0u, se1 = (N0 > 0u) ? 1u : 0u;
                    lut[(c0 + 20u * c1) * 25u + a0 + 5u * a1] =
                        nc0 | (nc1 << 8) | (reward << 16) | (nb << 18) | (se0 << 20) | (se1 << 21) | (bad << 22);
                }
}

// ---------------------------------------------------------------------------------------------
// Reward entries of the cellular LUTs: the float32 sum of the cells' rewards in double, +0.0 where it is zero.
// The kernels take the first entry of an env as its initial sum, so a -0.0 entry would give a -0.0 reward where
// the paths that add from 0.0f (rollout, pair8, generic) give +0.0; with no -0.0 entry no float32 sum is -0.0.
static float reward_entry(double r)
{
    return r == 0.0 ? 0.0f : (float)r;
}

// Cellular family, S, A <= 4: pair / single-cell entries (layout in gc_cell_fast.cu).
void gc_build_pair_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut, uint32_t *unsafe_rows)
{
    auto ok = [&](int s, int a) { return s < S && a < A; };
    auto nxt = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0;
        if (noise && fire && t->draws[s * A + a]) return (int)t->noisy[s * A + a];
        return (int)t->move[s * A + a];
    };
    auto rw = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0.0;
        if (noise && fire && t->draws[s * A + a] && t->reward_noisy) return (double)t->reward_noisy[s * A + a];
        return (double)t->reward[s * A + a];
    };
    auto se = [&](int j, int s0, int sp) { return (int)t->side_effects[((size_t)j * S + s0) * S + sp]; };
    auto cn = [&](int n) { return t->counted[n] ? 1u : 0u; };
    for (int p = 0; p < GC_PAIR_LUT_PAIRS; ++p) {
        const int sc = p & 3, ac = (p >> 2) & 3, sd = (p >> 4) & 3, ad = (p >> 6) & 3;
        const int nc = nxt(sc, ac, (p >> 8) & 1), nd = nxt(sd, ad, (p >> 9) & 1);
        const uint32_t uns01 = (C >= 2 && (se(0, nc, nd) == 2 || se(1, nc, nd) == 2)) ? 1u : 0u;
        lut[p].x = (cn(nc) + cn(nd)) | (((1u << nc) | (1u << nd)) << 8) | (uns01 << 12) |
                   ((uint32_t)nc << 16) | ((uint32_t)nd << 24);
        const float f = reward_entry(rw(sc, ac, (p >> 8) & 1) + rw(sd, ad, (p >> 9) & 1));
        std::memcpy(&lut[p].y, &f, sizeof(f));
    }
    for (int p = 0; p < 32; ++p) {
        const int s = p & 3, a = (p >> 2) & 3, n = nxt(s, a, (p >> 4) & 1);
        const uint32_t uns0 = (C == 1 && se(0, n, n) == 2) ? 1u : 0u;
        lut[GC_PAIR_LUT_PAIRS + p].x = cn(n) | ((1u << n) << 8) | (uns0 << 12) | ((uint32_t)n << 16);
        const float f = reward_entry(rw(s, a, (p >> 4) & 1));
        std::memcpy(&lut[GC_PAIR_LUT_PAIRS + p].y, &f, sizeof(f));
    }
    *unsafe_rows = 0;
    if (C >= 3)
        for (int s0 = 0; s0 < S; ++s0)
            for (int x = 0; x < S; ++x)
                if (se(2, s0, x) == 2) *unsafe_rows |= (1u << x) << (8 * s0);
}

// ---------------------------------------------------------------------------------------------
// Cellular family, packed layout (gc_cell_packed.cu): the same pair / single-cell rules, indexed the way
// the packed words deliver the digits and with the info word laid out for whole-word accumulation.
//   pair index   p = (s_c | s_d << 2) | (a_c | a_d << 2) << 4 | fire_c << 8 | fire_d << 9
//   single index p = s | a << 2 | fire << 4                       (entries GC_PAIR_LUT_PAIRS ..)
//   .x  bits  5k .. 5k+4 (k = 0..3)   how many of the entry's next levels x have SE[j >= 2][k][x] == 'unsafe',
//                   i.e. would be reported unsafe if cell 0 ended at level k             (:157-212)
//       bits 20-24  how many of them count towards the incidence          (cells3states3actions3.py:159-162)
//       bit  25     row-0 entries 0 and 1 of the side-effects matrix hold 'unsafe' for (s'_c, s'_d)
//                   (meaningful for the pair (cell 0, cell 1); single entry: for a 1-cell env)   (:157-212)
//       bits 28-31  next levels s'_c | s'_d << 2                                                 (:133-154)
//   .y  reward contribution (float)                                                              (:9-45)
// The sum of the .x words of an env's entries has no carries between the fields (<= 16 cells), and the
// nibble sits on top so that whatever its sum carries out of is discarded.
void gc_build_packed_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut)
{
    auto ok = [&](int s, int a) { return s < S && a < A; };
    auto nxt = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0;
        if (noise && fire && t->draws[s * A + a]) return (int)t->noisy[s * A + a];
        return (int)t->move[s * A + a];
    };
    auto rw = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0.0;
        if (noise && fire && t->draws[s * A + a] && t->reward_noisy) return (double)t->reward_noisy[s * A + a];
        return (double)t->reward[s * A + a];
    };
    auto se = [&](int j, int s0, int sp) { return (int)t->side_effects[((size_t)j * S + s0) * S + sp]; };
    auto info = [&](int n) {
        uint32_t w = t->counted[n] ? (1u << 20) : 0u;
        if (C >= 3)
            for (int k = 0; k < S; ++k)
                if (se(2, k, n) == 2) w |= 1u << (5 * k);
        return w;
    };
    for (int p = 0; p < GC_PAIR_LUT_PAIRS; ++p) {
        const int sc = p & 3, sd = (p >> 2) & 3, ac = (p >> 4) & 3, ad = (p >> 6) & 3;
        const int fc = (p >> 8) & 1, fd = (p >> 9) & 1;
        const int nc = nxt(sc, ac, fc), nd = nxt(sd, ad, fd);
        const uint32_t uns01 = (C >= 2 && (se(0, nc, nd) == 2 || se(1, nc, nd) == 2)) ? 1u : 0u;
        lut[p].x = (info(nc) + info(nd)) | (uns01 << 25) | ((uint32_t)(nc | (nd << 2)) << 28);
        const float f = reward_entry(rw(sc, ac, fc) + rw(sd, ad, fd));
        std::memcpy(&lut[p].y, &f, sizeof(f));
    }
    for (int p = 0; p < 32; ++p) {
        const int s = p & 3, a = (p >> 2) & 3, n = nxt(s, a, (p >> 4) & 1);
        const uint32_t uns0 = (C == 1 && se(0, n, n) == 2) ? 1u : 0u;
        lut[GC_PAIR_LUT_PAIRS + p].x = info(n) | (uns0 << 25) | ((uint32_t)n << 28);
        const float f = reward_entry(rw(s, a, (p >> 4) & 1));
        std::memcpy(&lut[GC_PAIR_LUT_PAIRS + p].y, &f, sizeof(f));
    }
}

// ---------------------------------------------------------------------------------------------
// Cellular family, 5..8 levels / actions (gc_cell_pair8.cu): the pair entries of gc_build_pair_lut with 3-bit
// digits (no noise: deterministic launches only), then the single-cell entries with the fire bit on top.
// pair index p = s_c | a_c << 3 | s_d << 6 | a_d << 9, single index p = s | a << 3 | fire << 6.
//   .x  bits 0-4 counted next levels, bit 7 pair-(0, 1) 'unsafe' flag, bits 8-15 one-hot set of the next levels,
//       bits 16-23 next level of cell c, bits 24-31 next level of cell d;  .y reward contribution (float)
void gc_build_pair8_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut, unsigned long long *unsafe_rows8,
                        unsigned long long *unsafe01_rows8)
{
    auto ok = [&](int s, int a) { return s < S && a < A; };
    auto nxt = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0;
        if (noise && fire && t->draws[s * A + a]) return (int)t->noisy[s * A + a];
        return (int)t->move[s * A + a];
    };
    auto rw = [&](int s, int a, int fire) {
        if (!ok(s, a)) return 0.0;
        if (noise && fire && t->draws[s * A + a] && t->reward_noisy) return (double)t->reward_noisy[s * A + a];
        return (double)t->reward[s * A + a];
    };
    auto se = [&](int j, int s0, int sp) { return (int)t->side_effects[((size_t)j * S + s0) * S + sp]; };
    auto cn = [&](int n) { return t->counted[n] ? 1u : 0u; };
    for (int p = 0; p < GC_PAIR8_PAIRS; ++p) {
        const int sc = p & 7, ac = (p >> 3) & 7, sd = (p >> 6) & 7, ad = (p >> 9) & 7;
        const int nc = nxt(sc, ac, 0), nd = nxt(sd, ad, 0);
        const uint32_t uns01 = (C >= 2 && (se(0, nc, nd) == 2 || se(1, nc, nd) == 2)) ? 1u : 0u;
        lut[p].x = (cn(nc) + cn(nd)) | (uns01 << 7) | (((1u << nc) | (1u << nd)) << 8) | ((uint32_t)nc << 16) | ((uint32_t)nd << 24);
        const float f = reward_entry(rw(sc, ac, 0) + rw(sd, ad, 0));
        std::memcpy(&lut[p].y, &f, sizeof(f));
    }
    for (int p = 0; p < 128; ++p) {
        const int s = p & 7, a = (p >> 3) & 7, n = nxt(s, a, p >> 6);
        const uint32_t uns0 = (C == 1 && se(0, n, n) == 2) ? 1u : 0u;
        lut[GC_PAIR8_PAIRS + p].x = cn(n) | (uns0 << 7) | ((1u << n) << 8) | ((uint32_t)n << 16);
        const float f = reward_entry(rw(s, a, p >> 6));
        std::memcpy(&lut[GC_PAIR8_PAIRS + p].y, &f, sizeof(f));
    }
    *unsafe_rows8 = 0;
    if (C >= 3)
        for (int s0 = 0; s0 < S; ++s0)
            for (int x = 0; x < S; ++x)
                if (se(2, s0, x) == 2) *unsafe_rows8 |= (unsigned long long)(1u << x) << (8 * s0);
    *unsafe01_rows8 = 0;
    for (int s0 = 0; s0 < S; ++s0)
        for (int s1 = 0; s1 < S; ++s1) {
            const bool uns = C >= 2 ? (se(0, s0, s1) == 2 || se(1, s0, s1) == 2) : (s0 == s1 && se(0, s0, s0) == 2);
            if (uns) *unsafe01_rows8 |= 1ull << (8 * s0 + s1);
        }
}
