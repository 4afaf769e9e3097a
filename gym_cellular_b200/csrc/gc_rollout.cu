// K-step fused rollout (SURVEY.md 8 f2): n_steps consecutive env.step() calls per env inside ONE kernel.
//
// The caller's loop around step() -- pick an action, step, accumulate the return -- is what agents and
// the synthetic random-action sweep do on both sides of the hot path.  Here the state of the four
// envs a thread owns stays in registers for all n_steps steps; actions are generated in the kernel,
// either uniformly at random or from a tabular policy (`initial_policy` as a table,
// cells3states3actions3.py:293-295, grid_world.py:423-438).  HBM traffic is one read and one write of
// the state per n_steps steps, so the kernel is bound by instruction issue, not by memory: it is the
// remedy for batches too small to be HBM-bound (BASELINE configs 2 and 3).
//
// The transition itself is the one of gc_cell_fast.cu / gc_grid.cu (same tables, same Philox words
// for the noise), so a rollout is bit-identical to n_steps calls of gc_step with the same actions.
//
// Random actions (part of the RNG layer, restated in oracle/gc_oracle.c: gco_policy_actions):
//   the action word of env g for cell c at RNG counter T is word (g % 4) of
//       philox(key, ctr = ((g/4)_lo, (g/4)_hi, T, 0x40000000 + c))
//   cellular: action = floor(word * 2^-32 * A);  grid world (c = 0): jurisdiction = bit 31, position =
//   bits 29-30, the other jurisdiction names no position (the reference sampler's distribution,
//   grid_world.py:191-195).  T is the counter the step's noise uses (episode step or global step).
//
// Experience collection (gc_collect): the RECORD instantiations also write every transition (obs, executed
// action, reward, flags, next_obs) into step-major [n_steps][ld] arrays and take the table policy
// epsilon-greedily (restated in tests/_collect_oracle.py).  For env g at global step G:
//   explore iff word (g % 4) of philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000000)) < ceil(eps * 2^32);
//   explore action = word (g % 4) of philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000001)): cellular joint action
//   floor(word * A^C / 2^32), grid world the random policy's rule.
// G is the global step even for episodic envs: exploration belongs to the agent, and keying it by the episode
// step would make every episode explore at the same steps with the same actions.
//
// Experience counts (gc_collect_counts): the COUNT instantiations take the same actions and draws as the RECORD
// ones and add each transition to per-(state, action) counters instead of writing it out; no draw is added.
//   joint tables: one warp-aggregated 64-bit global atomic per group of lanes on the same bin (__match_any_sync),
//     since after a reset every env of a warp sits in the same state and, under a table policy, acts alike;
//   per-cell N_c(s_c, a_c, s'_c): a 32-bit shared-memory histogram per block, [C][4][4][4], flushed at block exit.
//     The add that takes a bin across 2^31 moves 2^31 to global memory, so no shared bin wraps as long as fewer than
//     2^31 further adds land on it before that subtraction does (each add is at most 4, and the subtraction is the
//     next instruction of the thread that crossed).
// Grouped counts (gc_collect_counts_grouped, policy stacks only): a runtime branch of the same COUNT instantiations.
// Every table has a leading group dimension and env e adds into group min(table_of_env[e], n_tables - 1); the joint
// tables match lanes on the group-offset bin, the per-cell table uses warp-aggregated global atomics on (group, cell, bin).
#include "gc_device.cuh"

namespace {

constexpr uint32_t kActionStream = 0x40000000u;
constexpr uint32_t kExploreStream = 0x50000000u;     // + 0: explore test, + 1: explore action

// what a rollout kernel does with the transitions: nothing (gc_rollout), record them (gc_collect), count them
// (gc_collect_counts).  RECORD and COUNT take the table policy epsilon-greedily.
constexpr int kRollout = 0, kRecord = 1, kCount = 2;
constexpr uint32_t kCellFlush = 1u << 31;           // per-cell shared bin: moved to global memory at 2^31

__device__ __forceinline__ bool same4(const int (&t)[kEPT]) { return t[0] == t[1] && t[1] == t[2] && t[2] == t[3]; }

// action words of the 4 envs of a thread for cell c: one shared Philox block when the counters agree
__device__ __forceinline__ void action_words(const RolloutIO &io, uint32_t grp_lo, uint32_t grp_hi, const uint32_t (&T)[kEPT],
                                             bool shared, uint32_t c, uint32_t (&w)[kEPT])
{
    if (shared) {
        philox4x32_10(grp_lo, grp_hi, T[0], kActionStream + c, io.round_key, w);
    } else {
#pragma unroll 1
        for (int e = 0; e < kEPT; ++e) {
            uint32_t x[4];
            philox4x32_10(grp_lo, grp_hi, T[e], kActionStream + c, io.round_key, x);
            w[e] = x[e];
        }
    }
}

// grid world, the reference sampler's distribution: (a_0, a_1) = (4, pos) or (pos, 4) as a_0 + 5 a_1
__device__ __forceinline__ uint32_t random_grid_action(uint32_t w)
{
    const uint32_t pos = (w >> 29) & 3u;
    return (w >> 31) ? (4u + 5u * pos) : (pos + 20u);
}

// per-cell bin s * 16 + a * 4 + s' of cell c -> flat index of the caller's [C][S][A][S] table
__device__ __forceinline__ uint32_t cell_bin(const CellTables &tab, uint32_t c, uint32_t bin)
{
    const uint32_t S = static_cast<uint32_t>(tab.n_states), A = static_cast<uint32_t>(tab.n_actions);
    return ((c * S + (bin >> 4)) * A + ((bin >> 2) & 3u)) * S + (bin & 3u);
}

// epsilon-greedy (RECORD kernels): bit e of the result is set when env e of the thread explores at global step G;
// w then holds the explore-action words (drawn only when one of the 4 envs explores)
__device__ __forceinline__ uint32_t explore_words(const RolloutIO &io, uint32_t grp_lo, uint32_t grp_hi, uint32_t G,
                                                  uint32_t (&w)[kEPT])
{
    if (!io.explore_thr_nz) return 0u;
    uint32_t x[4];
    philox4x32_10(grp_lo, grp_hi, G, kExploreStream, io.round_key, x);
    uint32_t m = 0;
#pragma unroll
    for (int e = 0; e < kEPT; ++e) m |= (x[e] <= io.explore_thr_m1 ? 1u : 0u) << e;
    if (m) philox4x32_10(grp_lo, grp_hi, G, kExploreStream + 1u, io.round_key, w);
    return m;
}

// GC_POLICY_TABLE_STACK: the table ids of the 4 envs of a thread, re-read at every step (an L1 hit) rather than held in
// registers across the step loop
__device__ __forceinline__ int4 stack_map(const RolloutIO &io, int64_t e0)
{
    return __ldg(reinterpret_cast<const int4 *>(io.table_of_env + e0));
}

// first entry of table `id` of the stack; an id outside [0, n_tables) is clamped, so only the rows [0, n_tables) are read
// whatever the map holds.  64-bit offset: a table has up to 2^32 entries (16 cells x 4 levels)
__device__ __forceinline__ const int32_t *stack_row(const RolloutIO &io, int32_t id)
{
    const uint32_t j = min(static_cast<uint32_t>(id), io.n_tables - 1u);
    return io.policy + j * io.table_stride;
}

// count group of env e0 + e (gc_collect_counts_grouped): its table id clamped as stack_row clamps it, read at each use
// (an L1 hit) so that no group is held in registers across the count adds
__device__ __forceinline__ uint32_t count_group(const RolloutIO &io, int64_t e0, int e)
{
    return min(static_cast<uint32_t>(__ldg(io.table_of_env + e0 + e)), io.n_tables - 1u);
}

// lanes of this warp inside the env loop at this iteration (a prefix: lane l owns env e0 + 4 (l - lane))
__device__ __forceinline__ unsigned live_lanes(int64_t e0, int64_t n)
{
    const int64_t left = n - (e0 - kEPT * static_cast<int64_t>(threadIdx.x & 31));
    return left > 31 * kEPT ? 0xFFFFFFFFu : (1u << static_cast<uint32_t>((left + kEPT - 1) / kEPT)) - 1u;   // shift < 32
}

// one env per lane of the joint tables: bin sa = s * nA + a, successor nx, reward term q24 (round(r * 2^24)),
// 'unsafe' uns.  Lanes on the same bin add as one group; valid = false lanes (past the batch) count nothing.  Grouped
// counts pass sa + g * nS nA: the 'next' bin (g nS nA + sa) nS + nx is then g * nS nA nS + sa * nS + nx as well.
__device__ __forceinline__ void count_joint(const CountIO &cnt, unsigned lanes, bool valid, uint32_t sa, uint32_t nx,
                                            int32_t q24, uint32_t uns)
{
    const uint32_t lane = threadIdx.x & 31;
    const unsigned peers = __match_any_sync(lanes, valid ? sa : 0xFFFFFFFFu);
    const bool leader = valid && static_cast<uint32_t>(__ffs(peers) - 1) == lane;
    if (cnt.visits && leader) atomicAdd(cnt.visits + sa, static_cast<unsigned long long>(__popc(peers)));
    if (cnt.unsafe) {
        const unsigned u = __ballot_sync(lanes, uns != 0u) & peers;
        if (leader && u) atomicAdd(cnt.unsafe + sa, static_cast<unsigned long long>(__popc(u)));
    }
    if (cnt.reward_q24) {                 // |q24| < 2^31: 16-bit halves, so that a group of 32 cannot overflow
        const uint32_t lo = __reduce_add_sync(peers, static_cast<uint32_t>(q24) & 0xFFFFu);
        const int hi = __reduce_add_sync(peers, q24 >> 16);
        const long long sum = static_cast<long long>(hi) * 65536 + lo;
        if (leader && sum) atomicAdd(cnt.reward_q24 + sa, static_cast<unsigned long long>(sum));
    }
    if (cnt.next) {
        const uint32_t sas = sa * cnt.n_states + nx;
        const unsigned p2 = __match_any_sync(lanes, valid ? sas : 0xFFFFFFFFu);
        if (valid && static_cast<uint32_t>(__ffs(p2) - 1) == lane)
            atomicAdd(cnt.next + sas, static_cast<unsigned long long>(__popc(p2)));
    }
}

// grouped per-cell counts: one env per lane, flat index `at` of the grouped [G][C][S][A][S] table.  The per-block shared
// histogram holds one group only, so lanes on the same (group, cell, bin) add as one 64-bit global atomic instead.  Out
// of line: inlined into the 128-register count kernels of 11 to 16 cells, this path made them spill more.
__device__ __noinline__ void count_cell_grouped(unsigned long long *cell_next, unsigned lanes, bool valid, uint32_t at)
{
    const unsigned peers = __match_any_sync(lanes, valid ? at : 0xFFFFFFFFu);
    if (valid && static_cast<uint32_t>(__ffs(peers) - 1) == (threadIdx.x & 31))
        atomicAdd(cell_next + at, static_cast<unsigned long long>(__popc(peers)));
}

// ---------------------------------------------------------------------------------------------
template <int C, bool NOISE, int MODE>
__global__ void __launch_bounds__(kThreads, 2)
cell_rollout_kernel(const __grid_constant__ CellTables tab, const __grid_constant__ RolloutIO io,
                    const uint2 *__restrict__ lut, const __grid_constant__ CountIO cnt)
{
    constexpr bool RECORD = MODE == kRecord, EXPLORE = MODE != kRollout;
    constexpr int N_PAIR = NOISE ? GC_PAIR_LUT_PAIRS : 256;
    constexpr int N_SINGLE = NOISE ? 32 : 16;
    constexpr int NPAIR = C / 2;
    constexpr bool ODD = (C & 1) != 0;
    __shared__ uint2 s_pair[N_PAIR];
    __shared__ uint2 s_single[N_SINGLE];
    __shared__ unsigned long long s_stats[5];
    __shared__ uint32_t s_cell[MODE == kCount ? C * 64 : 1];        // N_c(s, a, s') at c * 64 + s * 16 + a * 4 + s'
    const uint32_t step0 = io.step_ctr ? *reinterpret_cast<const volatile uint32_t *>(io.step_ctr) : 0u;
    if constexpr (MODE == kCount)
        for (int i = threadIdx.x; i < C * 64; i += blockDim.x) s_cell[i] = 0;
    for (int i = threadIdx.x; i < N_PAIR; i += blockDim.x) s_pair[i] = lut[i];
    if (threadIdx.x < N_SINGLE) s_single[threadIdx.x] = lut[GC_PAIR_LUT_PAIRS + threadIdx.x];
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    __syncthreads();

    uint32_t st_steps = 0, st_unsafe = 0, st_count = 0, st_trunc = 0;
    long long st_reward = 0;
    const int64_t ld = io.ld;
    const uint32_t A = static_cast<uint32_t>(tab.n_actions);
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * kEPT;
    for (int64_t e0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * kEPT; e0 < io.n; e0 += stride) {
        const int rem = static_cast<int>(io.n - e0 < kEPT ? io.n - e0 : kEPT);
        const uint32_t vb = valid_bytes(rem);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset + e0);
        const uint32_t gid_lo = static_cast<uint32_t>(gid0), gid_hi = static_cast<uint32_t>(gid0 >> 32);
        const uint32_t grp_lo = static_cast<uint32_t>(gid0 >> 2), grp_hi = static_cast<uint32_t>(gid0 >> 34);
        uint32_t sw[C];
#pragma unroll
        for (int c = 0; c < C; ++c) sw[c] = ld_stream_u32(io.state + c * ld + e0) & 0x03030303u;
        const int4 t4 = ld_stream_v4(io.t + e0);
        int t[kEPT] = {t4.x, t4.y, t4.z, t4.w};
        float ret[kEPT] = {0.f, 0.f, 0.f, 0.f};
        uint32_t nuns[kEPT] = {0, 0, 0, 0};
        uint32_t idx[kEPT];

        auto fold_words = [&](const uint32_t (&w)[C], uint32_t (&out)[kEPT]) {   // tabular index of the 4 envs
#pragma unroll
            for (int e = 0; e < kEPT; ++e) out[e] = 0;
#pragma unroll
            for (int g = 0; g < (C + 3) / 4; ++g) {
                uint32_t q = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (4 * g + i < C) q += w[4 * g + i] * tab.place4[i];
#pragma unroll
                for (int e = 0; e < kEPT; ++e) out[e] += byte_of(q, e) * tab.place[4 * g];
            }
        };
        auto fold_index = [&]() { fold_words(sw, idx); };

#pragma unroll 1
        for (int k = 0; k < io.n_steps; ++k) {
            uint32_t T[kEPT];
#pragma unroll
            for (int e = 0; e < kEPT; ++e) T[e] = io.episodic ? static_cast<uint32_t>(t[e]) : step0 + static_cast<uint32_t>(k);
            const bool shared = !io.episodic || same4(t);
            // ---- actions ------------------------------------------------------------------------
            uint32_t aw[C];
            // the table action p[e] of each env -> epsilon-greedy -> per-cell digits aw
            auto table_actions = [&](uint32_t (&p)[kEPT]) {
                if constexpr (EXPLORE) {
                    uint32_t xw[kEPT];
                    const uint32_t xm = explore_words(io, grp_lo, grp_hi, step0 + static_cast<uint32_t>(k), xw);
#pragma unroll
                    for (int e = 0; e < kEPT; ++e)
                        if ((xm >> e) & 1u) p[e] = static_cast<uint32_t>((static_cast<unsigned long long>(xw[e]) * io.joint_actions) >> 32);
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    aw[c] = 0;
#pragma unroll
                    for (int e = 0; e < kEPT; ++e) { aw[c] |= (p[e] % A) << (8 * e); p[e] /= A; }
                }
            };
            if (io.policy_kind == GC_POLICY_TABLE) {
                fold_index();
                uint32_t p[kEPT];
#pragma unroll
                for (int e = 0; e < kEPT; ++e) p[e] = static_cast<uint32_t>(__ldg(io.policy + idx[e]));
                table_actions(p);
            } else if (io.policy_kind == GC_POLICY_TABLE_STACK) {
                fold_index();
                const int4 m = stack_map(io, e0);
                uint32_t p[kEPT] = {static_cast<uint32_t>(__ldg(stack_row(io, m.x) + idx[0])),
                                    static_cast<uint32_t>(__ldg(stack_row(io, m.y) + idx[1])),
                                    static_cast<uint32_t>(__ldg(stack_row(io, m.z) + idx[2])),
                                    static_cast<uint32_t>(__ldg(stack_row(io, m.w) + idx[3]))};
                table_actions(p);
            } else {
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    uint32_t w[kEPT];
                    action_words(io, grp_lo, grp_hi, T, shared, c, w);
                    aw[c] = __umulhi(w[0], A) | (__umulhi(w[1], A) << 8) | (__umulhi(w[2], A) << 16) | (__umulhi(w[3], A) << 24);
                }
            }
            const int64_t kofs = static_cast<int64_t>(k) * ld;        // record row of this step (K * ld may pass 2^31)
            if constexpr (RECORD) {
                if (io.rec_obs) {
                    if (io.policy_kind == GC_POLICY_RANDOM) fold_index();
                    st_stream_v4(io.rec_obs + kofs + e0, make_int4(idx[0], idx[1], idx[2], idx[3]));
                }
                if (io.rec_action) {                                   // sum_c a_c A^c of the executed digits
                    const uint32_t A2 = A * A, pl4[4] = {1u, A, A2, A2 * A};
                    uint32_t ai[kEPT] = {0, 0, 0, 0}, plg = 1u;
#pragma unroll
                    for (int g = 0; g < (C + 3) / 4; ++g) {
                        uint32_t q = 0;                                // digits <= 3, A <= 4: bytes do not carry
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (4 * g + i < C) q += aw[4 * g + i] * pl4[i];
#pragma unroll
                        for (int e = 0; e < kEPT; ++e) ai[e] += byte_of(q, e) * plg;
                        plg *= A2 * A2;
                    }
                    st_stream_v4(io.rec_action + kofs + e0, make_int4(ai[0], ai[1], ai[2], ai[3]));
                }
            }
            // ---- transition, reward, side effects (pair table, as in gc_cell_fast.cu) ----------------
            float r[kEPT] = {0.f, 0.f, 0.f, 0.f};
            uint32_t add[kEPT] = {0, 0, 0, 0}, orr[kEPT] = {0, 0, 0, 0}, first[kEPT] = {0, 0, 0, 0};
            uint32_t rows[C];
            uint32_t rnd[kEPT][4];
            uint32_t fire16[kEPT] = {0, 0, 0, 0};
            constexpr bool WIDE = C > GC_NARROW_CELLS;        // wide env: one Philox block per env (fire_bits_wide)
            if (NOISE && WIDE && tab.noise_thr_nz) {
#pragma unroll
                for (int e = 0; e < kEPT; ++e)
                    fire16[e] = fire_bits_wide<(C + 7) / 8>(tab, gid_lo | e, gid_hi, T[e], io.round_key);
            }
#pragma unroll
            for (int kk = 0; kk < NPAIR + (ODD ? 1 : 0); ++kk) {
                const int c = 2 * kk, d = 2 * kk + 1;
                const bool pair = kk < NPAIR;
                if (NOISE && !WIDE && (c & 3) == 0) {
#pragma unroll
                    for (int e = 0; e < kEPT; ++e)
                        philox4x32_10(gid_lo | e, gid_hi, T[e], static_cast<uint32_t>(c >> 2), io.round_key, rnd[e]);
                }
                auto fire = [&](int e, int cell) -> uint32_t {
                    if (WIDE) return (fire16[e] >> cell) & 1u;
                    return (NOISE && tab.noise_thr_nz && rnd[e][cell & 3] <= tab.noise_thr_m1) ? 1u : 0u;
                };
                uint32_t inf[kEPT];
                if (pair) {
                    const uint32_t pidx = (aw[d] * 4u + sw[d]) * 16u + aw[c] * 4u + sw[c];
#pragma unroll
                    for (int e = 0; e < kEPT; ++e) {
                        uint32_t ix = byte_of(pidx, e);
                        if (NOISE) ix |= (fire(e, c) << 8) | (fire(e, d) << 9);
                        const uint2 ent = s_pair[ix];
                        r[e] += __uint_as_float(ent.y);
                        inf[e] = ent.x;
                    }
                } else {
                    const uint32_t sidx = aw[c] * 4u + sw[c];
#pragma unroll
                    for (int e = 0; e < kEPT; ++e) {
                        uint32_t ix = byte_of(sidx, e) & 15u;
                        if (NOISE) ix |= fire(e, c) << 4;
                        const uint2 ent = s_single[ix];
                        r[e] += __uint_as_float(ent.y);
                        inf[e] = ent.x;
                    }
                }
#pragma unroll
                for (int e = 0; e < kEPT; ++e) {
                    add[e] += inf[e];
                    if (kk == 0) first[e] = inf[e]; else orr[e] |= inf[e];
                }
                const uint32_t u = prmt(inf[0], inf[1], 0x7362), v = prmt(inf[2], inf[3], 0x7362);
                rows[c] = prmt(u, v, 0x5410);
                if (pair) rows[d] = prmt(u, v, 0x7632);
            }
            // ---- bookkeeping --------------------------------------------------------------------
            uint32_t keep = 0xFFFFFFFFu, unsafe_w = 0, count_w = 0, trunc_w = 0;
            float rlog[kEPT];
            log2_1p_x4(tab.reward_log2, r, rlog);
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                const uint32_t s0n = (first[e] >> 16) & 3u;
                const uint32_t rowmask = (tab.unsafe_rows >> (8 * s0n)) & 0xFFu;
                const uint32_t uns = ((first[e] >> 12) & 1u) | ((((orr[e] >> 8) & rowmask) != 0u) ? 1u : 0u);
                const float rr = rlog[e];
                ret[e] += rr;
                nuns[e] += uns;
                unsafe_w |= uns << (8 * e); count_w |= (add[e] & 31u) << (8 * e);
                if (e < rem) st_reward += __float2int_rn(rr * 16777216.0f);
                t[e] += 1;
                if (io.max_episode_steps > 0 && t[e] >= io.max_episode_steps) {
                    t[e] = 0; trunc_w |= 1u << (8 * e); keep &= ~(0xFFu << (8 * e));
                }
            }
            st_steps += rem;
            st_unsafe = add_bytes(unsafe_w & vb, st_unsafe);
            st_count = add_bytes(count_w & vb, st_count);
            st_trunc = add_bytes(trunc_w & vb, st_trunc);
            if constexpr (RECORD) {
                if (io.rec_reward)
                    st_stream_v4(io.rec_reward + kofs + e0, make_int4(__float_as_int(rlog[0]), __float_as_int(rlog[1]),
                                                                      __float_as_int(rlog[2]), __float_as_int(rlog[3])));
                if (io.rec_flags)
                    st_stream_u32(io.rec_flags + kofs + e0,
                                  unsafe_w * GC_FLAG_UNSAFE | trunc_w * GC_FLAG_TRUNCATED | (count_w << GC_FLAG_COUNT_SHIFT));
                if (io.rec_next_obs) {                                 // successor before the auto-reset
                    uint32_t nx[kEPT];
                    fold_words(rows, nx);
                    st_stream_v4(io.rec_next_obs + kofs + e0, make_int4(nx[0], nx[1], nx[2], nx[3]));
                }
            }
            if constexpr (MODE == kCount) {
                if (cnt.cell_next && cnt.n_groups) {
                    const unsigned lanes = live_lanes(e0, io.n);
#pragma unroll 2
                    for (int e = 0; e < kEPT; ++e) {
                        const uint32_t S = static_cast<uint32_t>(tab.n_states), A = static_cast<uint32_t>(tab.n_actions);
                        uint32_t at = count_group(io, e0, e) * cnt.cell_stride;       // (group, cell 0) of env e
                        const uint32_t SAS = S * A * S;
#pragma unroll
                        for (int c = 0; c < C; ++c) {
                            count_cell_grouped(cnt.cell_next, lanes, e < rem,
                                               at + (((sw[c] >> (8 * e)) & 3u) * A + ((aw[c] >> (8 * e)) & 3u)) * S + ((rows[c] >> (8 * e)) & 3u));
                            at += SAS;
                        }
                    }
                } else if (cnt.cell_next) {
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const uint32_t b = (sw[c] << 4) | (aw[c] << 2) | rows[c];     // bytes s * 16 + a * 4 + s'
                        auto add = [&](uint32_t bin, uint32_t v) {
                            const uint32_t old = atomicAdd(&s_cell[c * 64 + bin], v);
                            if (old < kCellFlush && old + v >= kCellFlush) {
                                atomicSub(&s_cell[c * 64 + bin], kCellFlush);
                                atomicAdd(cnt.cell_next + cell_bin(tab, c, bin), static_cast<unsigned long long>(kCellFlush));
                            }
                        };
                        if (rem == kEPT && b == __byte_perm(b, 0, 0x0000)) {
                            add(b & 0xFFu, 4u);
                        } else {
#pragma unroll
                            for (int e = 0; e < kEPT; ++e)
                                if (e < rem) add(byte_of(b, e), 1u);
                        }
                    }
                }
                if (cnt.visits || cnt.next || cnt.reward_q24 || cnt.unsafe) {
                    if (io.policy_kind == GC_POLICY_RANDOM) fold_index();
                    // executed action sum_c a_c A^c, as recorded above (kept apart so that the RECORD kernels stay as
                    // they were compiled before the COUNT mode existed)
                    const uint32_t A2 = A * A, pl4[4] = {1u, A, A2, A2 * A};
                    uint32_t ai[kEPT] = {0, 0, 0, 0}, nx[kEPT] = {0, 0, 0, 0}, plg = 1u;
#pragma unroll
                    for (int g = 0; g < (C + 3) / 4; ++g) {
                        uint32_t q = 0;
#pragma unroll
                        for (int i = 0; i < 4; ++i)
                            if (4 * g + i < C) q += aw[4 * g + i] * pl4[i];
#pragma unroll
                        for (int e = 0; e < kEPT; ++e) ai[e] += byte_of(q, e) * plg;
                        plg *= A2 * A2;
                    }
                    if (cnt.next) fold_words(rows, nx);
                    const unsigned lanes = live_lanes(e0, io.n);
#pragma unroll
                    for (int e = 0; e < kEPT; ++e)
                        count_joint(cnt, lanes, e < rem,
                                    (cnt.n_groups ? count_group(io, e0, e) * cnt.sa_stride : 0u) + idx[e] * cnt.n_actions + ai[e],
                                    nx[e], __float2int_rn(rlog[e] * 16777216.0f), byte_of(unsafe_w, e));
                }
            }
#pragma unroll
            for (int c = 0; c < C; ++c)
                sw[c] = (rows[c] & keep) | ((0x01010101u * static_cast<uint8_t>(tab.init[c])) & ~keep);
        }
        fold_index();
#pragma unroll
        for (int c = 0; c < C; ++c) st_stream_u32(io.state + c * ld + e0, sw[c]);
        st_stream_v4(io.t + e0, make_int4(t[0], t[1], t[2], t[3]));
        st_stream_v4(io.index + e0, make_int4(idx[0], idx[1], idx[2], idx[3]));
        if constexpr (MODE == kRollout) {
            st_stream_v4(io.ret + e0, make_int4(__float_as_int(ret[0]), __float_as_int(ret[1]),
                                                __float_as_int(ret[2]), __float_as_int(ret[3])));
            st_stream_v4(io.n_unsafe + e0, make_int4(nuns[0], nuns[1], nuns[2], nuns[3]));
        }
    }
    if constexpr (MODE == kCount) {
        if (cnt.cell_next) {
            __syncthreads();
            for (int i = threadIdx.x; i < C * 64; i += blockDim.x)
                if (s_cell[i]) atomicAdd(cnt.cell_next + cell_bin(tab, i >> 6, i & 63u), static_cast<unsigned long long>(s_cell[i]));
        }
    }
    if (io.stats) {
        const ThreadStats ts = {st_steps, st_unsafe, st_count, st_trunc, st_reward};
        block_flush_stats(ts, s_stats, io.stats);
    }
    tick_step_counter(io.step_ctr, io.done_ctr, static_cast<uint32_t>(io.n_steps));
}

// ---------------------------------------------------------------------------------------------
// COUNT: the warp-aggregated adds need registers that 4 blocks per SM (64 per thread) do not leave
template <int MODE>
__global__ void __launch_bounds__(kThreads, MODE == kCount ? 2 : 4)
grid_rollout_kernel(const __grid_constant__ GridParams gp, const __grid_constant__ RolloutIO io,
                    const __grid_constant__ CountIO cnt)
{
    constexpr bool RECORD = MODE == kRecord, EXPLORE = MODE != kRollout;
    __shared__ uint32_t s_lut[GC_GRID_LUT_ENTRIES];
    __shared__ unsigned long long s_stats[5];
    const uint32_t step0 = io.step_ctr ? *reinterpret_cast<const volatile uint32_t *>(io.step_ctr) : 0u;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(gp.lut);
        uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
        for (int i = threadIdx.x; i < GC_GRID_LUT_ENTRIES / 4; i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    __syncthreads();

    uint32_t st_steps = 0, st_count = 0, st_trunc = 0, st_reward = 0, bad_bits = 0;
    const int64_t ld = io.ld;
    const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x * kEPT;
    for (int64_t e0 = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * kEPT; e0 < io.n; e0 += stride) {
        const int rem = static_cast<int>(io.n - e0 < kEPT ? io.n - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset + e0);
        const uint32_t grp_lo = static_cast<uint32_t>(gid0 >> 2), grp_hi = static_cast<uint32_t>(gid0 >> 34);
        const uint32_t s0w = ld_stream_u32(io.state + e0), s1w = ld_stream_u32(io.state + ld + e0);
        const int4 t4 = ld_stream_v4(io.t + e0);
        int t[kEPT] = {t4.x, t4.y, t4.z, t4.w};
        uint32_t c0[kEPT], c1[kEPT];
        float ret[kEPT] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int e = 0; e < kEPT; ++e) { c0[e] = byte_of(s0w, e); c1[e] = byte_of(s1w, e); }

#pragma unroll 1
        for (int k = 0; k < io.n_steps; ++k) {
            uint32_t T[kEPT];
#pragma unroll
            for (int e = 0; e < kEPT; ++e) T[e] = io.episodic ? static_cast<uint32_t>(t[e]) : step0 + static_cast<uint32_t>(k);
            const bool shared = !io.episodic || same4(t);
            uint32_t act[kEPT];                                   // a_0 + 5 a_1
            if (io.policy_kind != GC_POLICY_RANDOM) {                  // GC_POLICY_TABLE or GC_POLICY_TABLE_STACK
                if (io.policy_kind == GC_POLICY_TABLE) {
#pragma unroll
                    for (int e = 0; e < kEPT; ++e) {
                        const uint32_t tab = c0[e] + 20u * c1[e];
                        act[e] = static_cast<uint32_t>(__ldg(io.policy + (tab < 400u ? tab : 0u)));
                        if (act[e] > 24u) act[e] = 24u;
                    }
                } else {
                    const int4 m = stack_map(io, e0);
                    const int32_t *row[kEPT] = {stack_row(io, m.x), stack_row(io, m.y), stack_row(io, m.z), stack_row(io, m.w)};
#pragma unroll
                    for (int e = 0; e < kEPT; ++e) {
                        const uint32_t tab = c0[e] + 20u * c1[e];
                        act[e] = static_cast<uint32_t>(__ldg(row[e] + (tab < 400u ? tab : 0u)));
                        if (act[e] > 24u) act[e] = 24u;
                    }
                }
                if constexpr (EXPLORE) {
                    uint32_t xw[kEPT];
                    const uint32_t xm = explore_words(io, grp_lo, grp_hi, step0 + static_cast<uint32_t>(k), xw);
#pragma unroll
                    for (int e = 0; e < kEPT; ++e)
                        if ((xm >> e) & 1u) act[e] = random_grid_action(xw[e]);
                }
            } else {
                uint32_t w[kEPT];
                action_words(io, grp_lo, grp_hi, T, shared, 0u, w);
#pragma unroll
                for (int e = 0; e < kEPT; ++e) act[e] = random_grid_action(w[e]);
            }
            const int64_t kofs = static_cast<int64_t>(k) * ld;        // record row of this step (K * ld may pass 2^31)
            if constexpr (RECORD) {
                if (io.rec_obs)
                    st_stream_v4(io.rec_obs + kofs + e0, make_int4(c0[0] + 20u * c1[0], c0[1] + 20u * c1[1],
                                                                   c0[2] + 20u * c1[2], c0[3] + 20u * c1[3]));
                if (io.rec_action) st_stream_v4(io.rec_action + kofs + e0, make_int4(act[0], act[1], act[2], act[3]));
            }
            uint32_t trig[kEPT];
            if (shared) {
                philox4x32_10(grp_lo, grp_hi, T[0], 0u, io.round_key, trig);
            } else {
#pragma unroll 1
                for (int e = 0; e < kEPT; ++e) {
                    uint32_t x[4];
                    philox4x32_10(grp_lo, grp_hi, T[e], 0u, io.round_key, x);
                    trig[e] = x[e];
                }
            }
            uint32_t count_w = 0, trunc_w = 0, rew_w = 0;
            uint32_t nx[kEPT], ob[kEPT];
#pragma unroll
            for (int e = 0; e < kEPT; ++e) ob[e] = c0[e] + 20u * c1[e];
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                const uint32_t ix = (c0[e] + 20u * c1[e]) * 25u + act[e];
                uint32_t ent = s_lut[ix < GC_GRID_LUT_ENTRIES ? ix : 0];
                const uint32_t nb = (ent >> 18) & 3u;
                if (nb < 2u && gp.dispersal_thr_nz && trig[e] <= gp.dispersal_thr_m1) {      // grid_world.py:160-162
                    const uint32_t T0 = c0[e] & 3u, T1 = c1[e] & 3u;
                    uint32_t nc0 = ent & 0xFFu, nc1 = (ent >> 8) & 0xFFu;
                    const uint32_t Nk = ((trig[e] >> 1) & 1u) | ((trig[e] & 1u) << 1);
                    if (((trig[e] >> 2) & 1u) == 0u) nc0 = (nc0 & ~3u) | Nk; else nc1 = (nc1 & ~3u) | Nk;
                    const uint32_t rew = __popc(T0 & ~(nc0 & 3u)) + __popc(T1 & ~(nc1 & 3u));
                    ent = nc0 | (nc1 << 8) | (rew << 16) | (nb << 18) | (ent & (1u << 22));
                }
                if (e < rem) bad_bits |= ent;
                const uint32_t rew = (ent >> 16) & 3u;
                ret[e] += static_cast<float>(rew);
                c0[e] = ent & 0xFFu; c1[e] = (ent >> 8) & 0xFFu;
                nx[e] = c0[e] + 20u * c1[e];                              // successor before the auto-reset
                t[e] += 1;
                uint32_t tr = 0;
                if (io.max_episode_steps > 0 && t[e] >= io.max_episode_steps) { tr = 1; t[e] = 0; c0[e] = 15u; c1[e] = 18u; }
                count_w |= nb << (8 * e); trunc_w |= tr << (8 * e); rew_w |= rew << (8 * e);
            }
            const uint32_t vb = valid_bytes(rem);
            st_steps += rem;
            st_count = add_bytes(count_w & vb, st_count);
            st_trunc = add_bytes(trunc_w & vb, st_trunc);
            st_reward = add_bytes(rew_w & vb, st_reward);
            if constexpr (RECORD) {
                if (io.rec_reward)
                    st_stream_v4(io.rec_reward + kofs + e0, make_int4(__float_as_int(static_cast<float>(byte_of(rew_w, 0))),
                                                                      __float_as_int(static_cast<float>(byte_of(rew_w, 1))),
                                                                      __float_as_int(static_cast<float>(byte_of(rew_w, 2))),
                                                                      __float_as_int(static_cast<float>(byte_of(rew_w, 3)))));
                if (io.rec_flags)                                      // never 'unsafe'
                    st_stream_u32(io.rec_flags + kofs + e0, trunc_w * GC_FLAG_TRUNCATED | (count_w << GC_FLAG_COUNT_SHIFT));
                if (io.rec_next_obs) st_stream_v4(io.rec_next_obs + kofs + e0, make_int4(nx[0], nx[1], nx[2], nx[3]));
            }
            if constexpr (MODE == kCount) {                        // never 'unsafe'; reward term rew * 2^24
                const unsigned lanes = live_lanes(e0, io.n);
#pragma unroll
                for (int e = 0; e < kEPT; ++e)
                    count_joint(cnt, lanes, e < rem, (cnt.n_groups ? count_group(io, e0, e) * cnt.sa_stride : 0u) + ob[e] * 25u + act[e],
                                nx[e], static_cast<int32_t>(byte_of(rew_w, e) << 24), 0u);
            }
        }
        st_stream_u32(io.state + e0, c0[0] | (c0[1] << 8) | (c0[2] << 16) | (c0[3] << 24));
        st_stream_u32(io.state + ld + e0, c1[0] | (c1[1] << 8) | (c1[2] << 16) | (c1[3] << 24));
        st_stream_v4(io.t + e0, make_int4(t[0], t[1], t[2], t[3]));
        st_stream_v4(io.index + e0, make_int4(c0[0] + 20u * c1[0], c0[1] + 20u * c1[1], c0[2] + 20u * c1[2], c0[3] + 20u * c1[3]));
        if constexpr (MODE == kRollout) {
            st_stream_v4(io.ret + e0, make_int4(__float_as_int(ret[0]), __float_as_int(ret[1]),
                                                __float_as_int(ret[2]), __float_as_int(ret[3])));
            st_stream_v4(io.n_unsafe + e0, make_int4(0, 0, 0, 0));                   // never 'unsafe'
        }
    }
    if (bad_bits & (1u << 22)) atomicOr(io.status, 1ull);
    if (io.stats) {
        const ThreadStats ts = {st_steps, 0, st_count, st_trunc, static_cast<long long>(st_reward) << 24};
        block_flush_stats(ts, s_stats, io.stats);
    }
    tick_step_counter(io.step_ctr, io.done_ctr, static_cast<uint32_t>(io.n_steps));
}

// A rollout is compute-bound, so a small batch should occupy every SM: when the batch does not fill the
// GPU with 256-thread blocks, 64-thread blocks are launched instead (the kernels size themselves by
// blockDim.x).
inline int rollout_threads(int64_t n, int n_sm) { return (n + kEPT - 1) / kEPT < static_cast<int64_t>(n_sm) * kThreads * 2 ? 64 : kThreads; }

inline int rollout_grid(int64_t n, int threads, int n_sm, int blocks_per_sm_256)
{
    const int64_t need = (n + threads * kEPT - 1) / (threads * kEPT);
    const int64_t cap = static_cast<int64_t>(n_sm) * blocks_per_sm_256 * (kThreads / threads);
    return static_cast<int>(need < cap ? (need < 1 ? 1 : need) : cap);
}

template <int C, int MODE>
cudaError_t launch_rollout_c(const CellTables &tab, const RolloutIO &io, const CountIO &cnt, const uint2 *lut, bool noise,
                             int n_sm, cudaStream_t st)
{
    const int threads = rollout_threads(io.n, n_sm), grid = rollout_grid(io.n, threads, n_sm, 2);
    if (noise)
        cell_rollout_kernel<C, true, MODE><<<grid, threads, 0, st>>>(tab, io, lut, cnt);
    else
        cell_rollout_kernel<C, false, MODE><<<grid, threads, 0, st>>>(tab, io, lut, cnt);
    return cudaGetLastError();
}

template <int MODE>
cudaError_t launch_cell_rollout(const CellTables &tab, const RolloutIO &io, const CountIO &cnt, const uint2 *lut, bool noise,
                                int n_sm, cudaStream_t st)
{
    switch (tab.n_cells) {
#define GC_CASE(C) case C: return launch_rollout_c<C, MODE>(tab, io, cnt, lut, noise, n_sm, st);
        GC_CASE(1) GC_CASE(2) GC_CASE(3) GC_CASE(4) GC_CASE(5) GC_CASE(6) GC_CASE(7) GC_CASE(8)
        GC_CASE(9) GC_CASE(10) GC_CASE(11) GC_CASE(12) GC_CASE(13) GC_CASE(14) GC_CASE(15) GC_CASE(16)
#undef GC_CASE
    default: return cudaErrorInvalidValue;
    }
}

template <int MODE>
cudaError_t launch_grid_rollout(const GridParams &gp, const RolloutIO &io, const CountIO &cnt, int n_sm, cudaStream_t st)
{
    // the 40 KB table is staged per block: keep 256-thread blocks unless the batch is really small
    const int threads = (io.n + kEPT - 1) / kEPT < static_cast<int64_t>(n_sm) * kThreads / 2 ? 64 : kThreads;
    grid_rollout_kernel<MODE><<<rollout_grid(io.n, threads, n_sm, MODE == kCount ? 2 : 4), threads, 0, st>>>(gp, io, cnt);
    return cudaGetLastError();
}

}  // namespace

cudaError_t gc_launch_cell_rollout(const CellTables &tab, const RolloutIO &io, const uint2 *lut, bool noise, int n_sm,
                                   cudaStream_t st)
{
    return launch_cell_rollout<kRollout>(tab, io, CountIO{}, lut, noise, n_sm, st);
}

cudaError_t gc_launch_cell_collect(const CellTables &tab, const RolloutIO &io, const uint2 *lut, bool noise, int n_sm,
                                   cudaStream_t st)
{
    return launch_cell_rollout<kRecord>(tab, io, CountIO{}, lut, noise, n_sm, st);
}

cudaError_t gc_launch_cell_count(const CellTables &tab, const RolloutIO &io, const CountIO &cnt, const uint2 *lut, bool noise,
                                 int n_sm, cudaStream_t st)
{
    return launch_cell_rollout<kCount>(tab, io, cnt, lut, noise, n_sm, st);
}

cudaError_t gc_launch_grid_rollout(const GridParams &gp, const RolloutIO &io, int n_sm, cudaStream_t st)
{
    return launch_grid_rollout<kRollout>(gp, io, CountIO{}, n_sm, st);
}

cudaError_t gc_launch_grid_collect(const GridParams &gp, const RolloutIO &io, int n_sm, cudaStream_t st)
{
    return launch_grid_rollout<kRecord>(gp, io, CountIO{}, n_sm, st);
}

cudaError_t gc_launch_grid_count(const GridParams &gp, const RolloutIO &io, const CountIO &cnt, int n_sm, cudaStream_t st)
{
    return launch_grid_rollout<kCount>(gp, io, cnt, n_sm, st);
}
