// Fast path of the cellular (polarisation) step for S, A <= 4 levels, deterministic or stochastic.
//
// Two cells at a time: the four 2-bit digits (s_c, a_c, s_d, a_d) of a cell pair form one byte that,
// together with one "the noise draw of this cell fired" bit per cell in the stochastic case
// (cells3resetVdeadlock.py:35-61; Philox word < threshold, or a replayed uniform < p), indexes a table
// staged in shared memory (256 entries deterministic, 1024 stochastic; built on the host by
// gc_build_pair_lut).  One 64-bit shared load returns, for the pair,
//   .y  the reward contribution R[s_c][a_c] + R[s_d][a_d]                (cells3states3actions3.py:9-45)
//   .x  bits  0-4   how many of the two next levels count towards the incidence     (:159-162)
//       bits  8-11  one-hot set of the two next levels ("presence", for the side-effect report)
//       bit   12    row-0 entries 0 and 1 of the side-effects matrix hold 'unsafe' for (s'_c, s'_d)
//                   (meaningful for the pair (cell 0, cell 1) only)                 (:157-212)
//       bits 16-23  next level of cell c, bits 24-31 next level of cell d           (:133-154)
// so the per-(env, pair) work is: byte extract, LDS.64, FADD, IADD, LOP.  The 4 envs a thread owns
// travel through the pair-index arithmetic together (byte SWAR in one 32-bit word), and the next-state
// rows are rebuilt in SoA order with PRMT byte shuffles.  'unsafe' for the cells j >= 2 is evaluated
// per env from the presence set: unsafe iff some present level x has SE[j][s'_0][x] == unsafe, which
// needs the side-effect tables of all cells j >= 2 to be equal (they are for every table set
// gym_cellular_b200/tables.py builds; otherwise the generic kernel in gc_kernels.cu is used).
#include "gc_device.cuh"

namespace {

// Resident blocks per SM the register budget is sized for: all 2C row words of a thread's 4 envs are
// requested up front (memory-level parallelism), so wide envs trade occupancy for loads in flight.  The
// Philox variants of wide envs carry 16 more registers (one random block per env) and get the budget of
// three blocks.  (Five blocks of the narrow kernels, at 48 registers, measured 0.732 against 0.775 of the
// roofline: profiles/r01_tuning_log.md.)
constexpr int pair_min_blocks(int c, int rng)
{
    if (rng != GC_RNG_NONE && c > 4) return 3;
    if (rng == GC_RNG_NONE && ((c >= 4 && c <= 8) || c == 10 || c == 11)) return 3;
    return 4;
}

// The pair table is staged once per block, not replicated per lane.  Sixteen replicas (lane l reading replica
// l % 16) would keep the lanes of a half-warp off each other's bank pairs -- profiles/r01_kernel_cfg4.md counted
// 70 % of the shared-memory wavefronts of config 4 as conflicts -- but these kernels wait for HBM, and the
// replicated table measured slower: 190.9 us per step plain, 191.5 with 8 replicas, 193.7-195.3 with 16
// (profiles/r02_tuning_log.md).

// Everything a thread carries across the cell groups of its four envs.  The low halves of the info
// words (count byte, presence / flag byte) are accumulated two envs per register (16-bit lanes: envs
// 0, 1 and envs 2, 3): up to 8 pairs of count <= 2 and of presence / flag bytes <= 0x1F never carry
// out of a lane, so one add per register and pair does the four envs' counts.
struct EnvAcc {
    float r[kEPT];          // reward sums
    uint32_t sum01, sum23;  // sums of the info low halves: bits 0-4 of a lane = counted cells
    uint32_t or01, or23;    // bit 12 of a lane: pair (cell 0, cell 1) is 'unsafe'; bits 8-11: levels present in cells j >= 2
    uint32_t idx[kEPT];     // tabular index
    uint32_t s0w, s1w;      // next level of cell 0 / cell 1 (before an auto-reset), byte lane e = env e

    __device__ __forceinline__ void clear()
    {
#pragma unroll
        for (int e = 0; e < kEPT; ++e) { r[e] = 0.f; idx[e] = 0; }
        sum01 = sum23 = or01 = or23 = s0w = s1w = 0;
    }
};

// One group of N <= 4 consecutive cells starting at cell c0 (c0 % 4 == 0) for the 4 envs of a thread.
//   sw / aw : state / action words of the N cells (byte lane e = env e)
//   FIRST   : the group holds cell 0
template <int N, int C, int RNG, bool WITH_SE, bool FIRST>
__device__ __forceinline__ void do_cells(const CellTables &tab, const StepIO &io, const uint2 *s_pair,
                                         const uint2 *s_single, const uint8_t (*s_se)[GC_TBL], int c0,
                                         uint32_t e0, int rem, uint32_t gid_lo, uint32_t gid_hi, uint32_t step_counter,
                                         const int (&tin)[kEPT], uint32_t keep, const uint32_t (&sw)[4],
                                         const uint32_t (&aw)[4], const uint32_t (&fire16)[kEPT], EnvAcc &acc,
                                         uint32_t (&next)[4])
{
    // fb[e]: bit i = the noise draw of cell (c0 + i) of env e fired (the table ignores the bit where the
    // (level, action) pair consumes no draw).  The four random words are reduced to four bits at once so
    // that only one register per env stays live.
    uint32_t fb[kEPT] = {0, 0, 0, 0};
    if (RNG == GC_RNG_PHILOX && C > GC_NARROW_CELLS) {
        // wide env: the fire bits of all cells were drawn from ONE Philox block per env (fire_bits_wide)
#pragma unroll
        for (int e = 0; e < kEPT; ++e) fb[e] = (fire16[e] >> c0) & 15u;
    } else if (RNG == GC_RNG_PHILOX) {
#pragma unroll
        for (int e = 0; e < kEPT; ++e) {
            uint32_t w[4];
            const uint32_t ctr = io.episodic ? static_cast<uint32_t>(tin[e]) : step_counter;
            philox4x32_10(gid_lo | e, gid_hi, ctr, static_cast<uint32_t>(c0 >> 2), io.round_key, w);
            const uint32_t thr = tab.noise_thr_m1;            // threshold - 1; a zero threshold never gets here (gc_api.cu)
            fb[e] = (w[0] <= thr ? 1u : 0u) | (w[1] <= thr ? 2u : 0u) | (w[2] <= thr ? 4u : 0u) | (w[3] <= thr ? 8u : 0u);
        }
    } else if (RNG == GC_RNG_REPLAY) {
#pragma unroll
        for (int e = 0; e < kEPT; ++e)
            if (e < rem)
#pragma unroll
                for (int i = 0; i < N; ++i)
                    fb[e] |= (io.replay[static_cast<size_t>(e0 + e) * C + c0 + i] < tab.noise_prob ? 1u : 0u) << i;
    }
    // 32-bit element indexes (n_cells * ld <= 2^31, gc_create): an address is one IMAD.WIDE.U32 on the FMA pipe
    const uint32_t ld = static_cast<uint32_t>(io.ld);
    uint32_t q = 0;                       // index digits of the group folded into one byte per env
    uint32_t rows[4];
#pragma unroll
    for (int i = 0; i < N; i += 2) {
        const bool pair = i + 1 < N;
        uint32_t inf[kEPT];
        if (pair) {
            const uint32_t pidx = ((aw[i + 1] & 0x03030303u) * 4u + (sw[i + 1] & 0x03030303u)) * 16u +
                                  (aw[i] & 0x03030303u) * 4u + (sw[i] & 0x03030303u);
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                uint32_t ix = byte_of(pidx, e);
                if (RNG != GC_RNG_NONE) ix |= ((fb[e] >> i) & 3u) << 8;
                const uint2 ent = s_pair[ix];
                if (FIRST && i == 0) acc.r[e] = __uint_as_float(ent.y); else acc.r[e] += __uint_as_float(ent.y);
                inf[e] = ent.x;
            }
        } else {
            const uint32_t sidx = (aw[i] & 0x03030303u) * 4u + (sw[i] & 0x03030303u);
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                uint32_t ix = byte_of(sidx, e) & 15u;
                if (RNG != GC_RNG_NONE) ix |= ((fb[e] >> i) & 1u) << 4;
                const uint2 ent = s_single[ix];
                if (FIRST && i == 0) acc.r[e] = __uint_as_float(ent.y); else acc.r[e] += __uint_as_float(ent.y);
                inf[e] = ent.x;
            }
        }
        const uint32_t w01 = prmt(inf[0], inf[1], 0x5410), w23 = prmt(inf[2], inf[3], 0x5410);
        acc.sum01 += w01; acc.sum23 += w23;
        const uint32_t keep_bits = (FIRST && i == 0) ? 0x10001000u : 0x0F000F00u;
        acc.or01 |= w01 & keep_bits; acc.or23 |= w23 & keep_bits;
        // SoA rows of the next state: byte 2 (cell c0+i) and byte 3 (cell c0+i+1) of the four info words
        const uint32_t u = prmt(inf[0], inf[1], 0x7362), v = prmt(inf[2], inf[3], 0x7362);
        rows[i] = prmt(u, v, 0x5410);
        if (pair) rows[i + 1] = prmt(u, v, 0x7632);
        if (FIRST && i == 0) { acc.s0w = rows[0]; acc.s1w = pair ? rows[1] : rows[0]; }
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {
        if (WITH_SE) {
            // row 0 of the side-effects matrix from the (pre-reset) next state: entry j from
            // (s'_0, s'_p), p = 1 for j = 0 (cell 0 and its partner live in the first group)
            uint32_t sew = 0;
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                const uint32_t s0n = byte_of(acc.s0w, e);
                const uint32_t partner = (FIRST && i == 0) ? byte_of(acc.s1w, e) : byte_of(rows[i], e);
                sew |= static_cast<uint32_t>(s_se[c0 + i][(s0n * GC_LVL_PAD + partner) & (GC_TBL - 1)]) << (8 * e);
            }
            st_stream_u32(io.se_row + ((c0 + i) * ld + e0), sew);
        }
        const uint32_t out = (rows[i] & keep) | ((0x01010101u * static_cast<uint8_t>(tab.init[c0 + i])) & ~keep);
        next[i] = out;                    // (used by the many-step kernel only: the state stays in registers there)
        st_stream_u32(io.state + ((c0 + i) * ld + e0), out);
        if (io.final_state) st_stream_u32(io.final_state + ((c0 + i) * ld + e0), rows[i]);
        q += out * tab.place4[i];
    }
    const uint32_t place = tab.place[c0];
#pragma unroll
    for (int e = 0; e < kEPT; ++e) acc.idx[e] += byte_of(q, e) * place;
}

template <int N>
__device__ __forceinline__ void load_cells(const StepIO &io, int c0, uint32_t e0, uint32_t (&sw)[4], uint32_t (&aw)[4])
{
    const uint32_t ld = static_cast<uint32_t>(io.ld);
#pragma unroll
    for (int i = 0; i < N; ++i) {
        sw[i] = ld_stream_u32(io.state + ((c0 + i) * ld + e0));
        aw[i] = ld_stream_u32(io.actions + ((c0 + i) * ld + e0));
    }
}

// What the step kernel and the many-step kernel do per 4-env word around the cell groups (do_cells): the time
// limit and the wide-env draws before, the flags, statistics and stores after.

// Episode steps after this step (0 where the time limit is reached), the truncated flags (byte lane e = env e)
// and keep, the byte mask of the envs NOT reset.
__device__ __forceinline__ void time_limit(const StepIO &io, const int (&tin)[kEPT], int (&tn)[kEPT], uint32_t &trunc_w,
                                           uint32_t &keep)
{
#pragma unroll
    for (int e = 0; e < kEPT; ++e) tn[e] = tin[e] + 1;
    trunc_w = 0;
    keep = 0xFFFFFFFFu;
    if (io.max_episode_steps > 0) {
#pragma unroll
        for (int e = 0; e < kEPT; ++e)
            if (tn[e] >= io.max_episode_steps) { tn[e] = 0; trunc_w |= 1u << (8 * e); keep &= ~(0xFFu << (8 * e)); }
    }
}

// The fire bits of every cell of a wide env with Philox draws; zero otherwise (narrow envs draw in do_cells).
template <int C, int RNG>
__device__ __forceinline__ void wide_fire_bits(const CellTables &tab, const StepIO &io, uint32_t gid_lo, uint32_t gid_hi,
                                               uint32_t step_counter, const int (&tin)[kEPT], uint32_t (&fire16)[kEPT])
{
#pragma unroll
    for (int e = 0; e < kEPT; ++e) fire16[e] = 0;
    if (RNG == GC_RNG_PHILOX && C > GC_NARROW_CELLS) {
#pragma unroll
        for (int e = 0; e < kEPT; ++e)
            fire16[e] = fire_bits_wide<(C + 7) / 8>(tab, gid_lo | e, gid_hi, io.episodic ? static_cast<uint32_t>(tin[e]) : step_counter,
                                                    io.round_key);
    }
}

// Unsafe / count for the four envs at once (byte lanes): the count and the presence / flag bytes of the 16-bit
// lanes, and the unsafe-levels mask of each env's s'_0 picked out of tab.unsafe_rows with one byte permute
// (selector nibble e = s'_0 of env e); then the statistics and the per-env outputs other than the state rows.
__device__ __forceinline__ void finish_word(const CellTables &tab, const StepIO &io, uint32_t e0, int rem, const EnvAcc &acc,
                                            const int (&tn)[kEPT], uint32_t trunc_w, uint32_t &st_steps, uint32_t &st_unsafe,
                                            uint32_t &st_count, uint32_t &st_trunc, long long &st_reward)
{
    float rout[kEPT];
    log2_1p_x4(tab.reward_log2, acc.r, rout);
    const uint32_t count_w = prmt(acc.sum01, acc.sum23, 0x6420) & 0x1F1F1F1Fu;
    const uint32_t present = prmt(acc.or01, acc.or23, 0x7531);            // bits 0-3 levels present, bit 4 pair-(0,1) flag
    const uint32_t nib = acc.s0w | (acc.s0w >> 4);                        // byte 0: s0_0 | s0_1 << 4, byte 2: s0_2 | s0_3 << 4
    const uint32_t rowmask = prmt(tab.unsafe_rows, 0u, prmt(nib, 0u, 0x4420) & 0x3333u);
    const uint32_t unsafe_w = ((((present & rowmask) + 0x0F0F0F0Fu) | present) >> 4) & 0x01010101u;
#pragma unroll
    for (int e = 0; e < kEPT; ++e)
        if (e < rem) st_reward += __float2int_rn(rout[e] * 16777216.0f);     // |reward| < 128: gc_set_tables
    {
        const uint32_t vb = valid_bytes(rem);
        st_steps += rem;
        st_unsafe = add_bytes(unsafe_w & vb, st_unsafe);
        st_count = add_bytes(count_w & vb, st_count);
        st_trunc = add_bytes(trunc_w & vb, st_trunc);
    }
    st_stream_v4(io.t + e0, make_int4(tn[0], tn[1], tn[2], tn[3]));
    st_stream_v4(io.reward + e0, make_int4(__float_as_int(rout[0]), __float_as_int(rout[1]),
                                           __float_as_int(rout[2]), __float_as_int(rout[3])));
    st_stream_v4(io.index + e0, make_int4(acc.idx[0], acc.idx[1], acc.idx[2], acc.idx[3]));
    st_stream_u32(io.terminated + e0, 0u);
    st_stream_u32(io.truncated + e0, trunc_w);
    st_stream_u32(io.unsafe + e0, unsafe_w);
    st_stream_u32(io.count + e0, count_w);
}

// The cells of an env are walked in groups of four (two table lookups per env and group) by a
// software-pipelined loop: the rows of group g+1 are requested before group g is computed, so a
// thread keeps 8-16 row words in flight with ~60 registers and four blocks stay resident per SM.
template <int C, int RNG, bool WITH_SE>
__global__ void __launch_bounds__(kThreads, pair_min_blocks(C, RNG))
cell_pair_kernel(const __grid_constant__ CellTables tab, const __grid_constant__ StepIO io,
                 const uint2 *__restrict__ lut)
{
    constexpr int NG = C / 4, R = C % 4;                        // full groups, cells in the tail group
    constexpr int N_PAIR = (RNG == GC_RNG_NONE) ? 256 : GC_PAIR_LUT_PAIRS;
    constexpr int N_SINGLE = (RNG == GC_RNG_NONE) ? 16 : 32;
    __shared__ uint2 s_pair[N_PAIR];
    __shared__ uint2 s_single[N_SINGLE];
    __shared__ uint8_t s_se[WITH_SE ? C : 1][GC_TBL];
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;

    const uint32_t stride = gridDim.x * kThreads * kEPT, e_end = static_cast<uint32_t>(io.end);
    // Narrow envs (C < 4: a thread reads only ~10 words per 4 envs) prefetch the inputs of their next
    // 4-env word before computing the current one, to keep enough bytes in flight per SM; the first
    // word's inputs are requested before the tables are staged, so that the two latencies overlap.  Wide
    // envs do not: their prefetched rows spill or cost a resident block (profiles/r01_tuning_log.md).
    constexpr bool PREFETCH = NG == 0;
    constexpr int G0 = NG > 0 ? 4 : R;                       // cells in the first group
    uint32_t e0 = static_cast<uint32_t>(io.begin) + (blockIdx.x * kThreads + threadIdx.x) * kEPT;
    // the immutable tables are requested first (they may be read while the previous step kernel of the
    // stream is still running), then the data the previous kernel wrote, then the tables are stored
    constexpr int LUT_PER_THREAD = N_PAIR / kThreads;
    uint2 lut_pair[LUT_PER_THREAD], lut_single = make_uint2(0u, 0u);
#pragma unroll
    for (int k = 0; k < LUT_PER_THREAD; ++k) lut_pair[k] = lut[threadIdx.x + k * kThreads];
    if (threadIdx.x < N_SINGLE) lut_single = lut[GC_PAIR_LUT_PAIRS + threadIdx.x];
    pdl_launch_dependents();
    pdl_wait();
    uint32_t ps[4], pa[4];
    int4 pt = make_int4(0, 0, 0, 0);
    if constexpr (PREFETCH) if (e0 < e_end) {
        load_cells<G0>(io, 0, e0, ps, pa);
        pt = ld_stream_v4(io.t + e0);
    }
    step_counter_read(io, &s_ctr);
#pragma unroll
    for (int k = 0; k < LUT_PER_THREAD; ++k) s_pair[threadIdx.x + k * kThreads] = lut_pair[k];
    if (threadIdx.x < N_SINGLE) s_single[threadIdx.x] = lut_single;
    if (WITH_SE)
        for (int i = threadIdx.x; i < C * GC_TBL; i += kThreads) s_se[i / GC_TBL][i % GC_TBL] = tab.se[i / GC_TBL][i % GC_TBL];
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    __syncthreads();

    const uint32_t step_now = step_counter_arrive(io, &s_ctr);
    const uint32_t step_counter = (RNG == GC_RNG_PHILOX) ? step_now : 0u;
    uint32_t st_steps = 0, st_unsafe = 0, st_count = 0, st_trunc = 0;   // < 2^32 per thread and launch
    long long st_reward = 0;
#pragma unroll 1
    for (; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);    // envs of this word in range
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;           // multiple of 4: | e never carries
        const uint32_t gid_lo = static_cast<uint32_t>(gid0), gid_hi = static_cast<uint32_t>(gid0 >> 32);

        uint32_t sa[4], aa[4], sb[4], ab[4];
        int4 t4;
        if constexpr (PREFETCH) {
#pragma unroll
            for (int i = 0; i < 4; ++i) { sa[i] = ps[i]; aa[i] = pa[i]; }
            t4 = pt;
            if (NG > 1) load_cells<4>(io, 4, e0, sb, ab); else if (NG == 1 && R > 0) load_cells<R>(io, 4, e0, sb, ab);
            if (e0 + stride < e_end) {
                load_cells<G0>(io, 0, e0 + stride, ps, pa);
                pt = ld_stream_v4(io.t + (e0 + stride));
            }
        } else {
            load_cells<4>(io, 0, e0, sa, aa);
            t4 = ld_stream_v4(io.t + e0);
            if (NG > 1) load_cells<4>(io, 4, e0, sb, ab); else if (R > 0) load_cells<R>(io, 4, e0, sb, ab);
        }

        const int tin[kEPT] = {t4.x, t4.y, t4.z, t4.w};
        int tn[kEPT];
        uint32_t trunc_w, keep, fire16[kEPT];
        time_limit(io, tin, tn, trunc_w, keep);
        wide_fire_bits<C, RNG>(tab, io, gid_lo, gid_hi, step_counter, tin, fire16);
        EnvAcc acc;
        acc.clear();
        uint32_t nx[4];                   // next rows of a group: not needed here (every step reloads its state)

        if (NG == 0) {
            do_cells<R, C, RNG, WITH_SE, true>(tab, io, s_pair, s_single, s_se, 0, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sa, aa, fire16, acc, nx);
        } else {
            do_cells<4, C, RNG, WITH_SE, true>(tab, io, s_pair, s_single, s_se, 0, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sa, aa, fire16, acc, nx);
#pragma unroll 1
            for (int g = 1; g < NG; ++g) {
#pragma unroll
                for (int i = 0; i < 4; ++i) { sa[i] = sb[i]; aa[i] = ab[i]; }
                if (g + 1 < NG) load_cells<4>(io, 4 * (g + 1), e0, sb, ab);
                else if (R > 0) load_cells<R>(io, 4 * NG, e0, sb, ab);
                do_cells<4, C, RNG, WITH_SE, false>(tab, io, s_pair, s_single, s_se, 4 * g, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sa, aa, fire16, acc, nx);
            }
            if (R > 0)
                do_cells<R, C, RNG, WITH_SE, false>(tab, io, s_pair, s_single, s_se, 4 * NG, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sb, ab, fire16, acc, nx);
        }

        finish_word(tab, io, e0, rem, acc, tn, trunc_w, st_steps, st_unsafe, st_count, st_trunc, st_reward);
    }
    if (io.stats) {
        const ThreadStats ts = {st_steps, st_unsafe, st_count, st_trunc, st_reward};
        block_flush_stats(ts, s_stats, io.stats);
    }
    step_counter_finish(io, &s_ctr);
}

template <int C, int RNG>
cudaError_t launch_pair_cr(const CellTables &tab, const StepIO &io, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const int64_t n = io.end - io.begin;
    if (io.se_row)
        return launch_step_kernel(cell_pair_kernel<C, RNG, true>, grid_for<cell_pair_kernel<C, RNG, true>>(n, n_sm), kThreads, 0, st, tab, io, lut);
    else
        return launch_step_kernel(cell_pair_kernel<C, RNG, false>, grid_for<cell_pair_kernel<C, RNG, false>>(n, n_sm), kThreads, 0, st, tab, io, lut);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// gc_step_many in ONE launch (small shards, gc_api.cu: many_fusable): the n_steps bound steps of a handle whose
// slots differ only in their action buffers.  A step of a 65,536-env shard is a 3 us launch around 0.3 us of work
// (BASELINE config 2), so the steps are run back to back by the thread that owns the envs: state and episode step
// stay in registers between two steps, the actions of step k + 1 are requested before step k is computed, and
// EVERY per-step output (state, t, reward, index, flags, side-effect row, statistics) is written at every step
// exactly as the n_steps separate launches write it -- same time_limit, wide_fire_bits, do_cells and finish_word as
// cell_pair_kernel, same Philox counters (global step of the launch + k) -- so the results are bit-identical to them
// (tests/test_gpu_many.py).
template <int C, int RNG, bool WITH_SE, int THREADS>
__global__ void __launch_bounds__(THREADS, 256 / THREADS * 2)
cell_pair_many_kernel(const __grid_constant__ CellTables tab, const __grid_constant__ ManyIO mio, const uint2 *__restrict__ lut)
{
    const StepIO &io = mio.io;
    constexpr int NG = C / 4, R = C % 4, G = (C + 3) / 4;
    constexpr int N_PAIR = (RNG == GC_RNG_NONE) ? 256 : GC_PAIR_LUT_PAIRS;
    constexpr int N_SINGLE = (RNG == GC_RNG_NONE) ? 16 : 32;
    __shared__ uint2 s_pair[N_PAIR];
    __shared__ uint2 s_single[N_SINGLE];
    __shared__ uint8_t s_se[WITH_SE ? C : 1][GC_TBL];
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;

    for (int i = threadIdx.x; i < N_PAIR; i += THREADS) s_pair[i] = lut[i];
    if (threadIdx.x < N_SINGLE) s_single[threadIdx.x] = lut[GC_PAIR_LUT_PAIRS + threadIdx.x];
    if (WITH_SE)
        for (int i = threadIdx.x; i < C * GC_TBL; i += THREADS) s_se[i / GC_TBL][i % GC_TBL] = tab.se[i / GC_TBL][i % GC_TBL];
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    pdl_launch_dependents();
    pdl_wait();
    step_counter_read(io, &s_ctr);
    __syncthreads();
    const uint32_t step0 = step_counter_arrive(io, &s_ctr);

    const uint32_t ld = static_cast<uint32_t>(io.ld);
    const uint32_t stride = gridDim.x * THREADS * kEPT, e_end = static_cast<uint32_t>(io.end);
    uint32_t st_steps = 0, st_unsafe = 0, st_count = 0, st_trunc = 0;
    long long st_reward = 0;
#pragma unroll 1
    for (uint32_t e0 = static_cast<uint32_t>(io.begin) + (blockIdx.x * THREADS + threadIdx.x) * kEPT; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;
        const uint32_t gid_lo = static_cast<uint32_t>(gid0), gid_hi = static_cast<uint32_t>(gid0 >> 32);
        uint32_t sw[G][4], an[G][4];                       // state rows; action rows of the NEXT step
#pragma unroll
        for (int c = 0; c < C; ++c) {
            sw[c / 4][c % 4] = ld_stream_u32(io.state + (c * ld + e0));
            an[c / 4][c % 4] = ld_stream_u32(mio.tape[0] + (c * ld + e0));
        }
        const int4 t4 = ld_stream_v4(io.t + e0);
        int t[kEPT] = {t4.x, t4.y, t4.z, t4.w};
        int slot = 0;
#pragma unroll 1
        for (int k = 0; k < mio.n_steps; ++k) {
            uint32_t aa[G][4];
#pragma unroll
            for (int c = 0; c < C; ++c) aa[c / 4][c % 4] = an[c / 4][c % 4];
            slot = slot + 1 == mio.n_tape ? 0 : slot + 1;
            if (k + 1 < mio.n_steps) {
                const int8_t *const nxt = mio.tape[slot];
#pragma unroll
                for (int c = 0; c < C; ++c) an[c / 4][c % 4] = ld_stream_u32(nxt + (c * ld + e0));
            }
            const int tin[kEPT] = {t[0], t[1], t[2], t[3]};
            int tn[kEPT];
            uint32_t trunc_w, keep, fire16[kEPT];
            time_limit(io, tin, tn, trunc_w, keep);
            const uint32_t step_counter = (RNG == GC_RNG_PHILOX) ? step0 + static_cast<uint32_t>(k) : 0u;
            wide_fire_bits<C, RNG>(tab, io, gid_lo, gid_hi, step_counter, tin, fire16);
            EnvAcc acc;
            acc.clear();
            uint32_t nx[G][4];
            if constexpr (NG == 0) {
                do_cells<R, C, RNG, WITH_SE, true>(tab, io, s_pair, s_single, s_se, 0, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sw[0], aa[0], fire16, acc, nx[0]);
            } else {
                do_cells<4, C, RNG, WITH_SE, true>(tab, io, s_pair, s_single, s_se, 0, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sw[0], aa[0], fire16, acc, nx[0]);
#pragma unroll
                for (int g = 1; g < NG; ++g)
                    do_cells<4, C, RNG, WITH_SE, false>(tab, io, s_pair, s_single, s_se, 4 * g, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sw[g], aa[g], fire16, acc, nx[g]);
                if constexpr (R > 0)
                    do_cells<R, C, RNG, WITH_SE, false>(tab, io, s_pair, s_single, s_se, 4 * NG, e0, rem, gid_lo, gid_hi, step_counter, tin, keep, sw[NG], aa[NG], fire16, acc, nx[NG]);
            }
            finish_word(tab, io, e0, rem, acc, tn, trunc_w, st_steps, st_unsafe, st_count, st_trunc, st_reward);
#pragma unroll
            for (int c = 0; c < C; ++c) sw[c / 4][c % 4] = nx[c / 4][c % 4];
#pragma unroll
            for (int e = 0; e < kEPT; ++e) t[e] = tn[e];
        }
    }
    if (io.stats) {
        const ThreadStats ts = {st_steps, st_unsafe, st_count, st_trunc, st_reward};
        block_flush_stats(ts, s_stats, io.stats);
    }
    step_counter_finish(io, &s_ctr, static_cast<uint32_t>(mio.n_steps));
}

template <int C, int RNG, bool WITH_SE, int THREADS>
cudaError_t launch_pair_many_t(const CellTables &tab, const ManyIO &mio, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const int64_t n = mio.io.end - mio.io.begin;
    return launch_step_kernel(cell_pair_many_kernel<C, RNG, WITH_SE, THREADS>,
                              grid_for<cell_pair_many_kernel<C, RNG, WITH_SE, THREADS>, THREADS>(n, n_sm), THREADS, 0, st, tab, mio, lut);
}

// shards that do not fill every SM with 256-thread blocks take smaller blocks (kManySmallThreads)
template <int C, int RNG>
cudaError_t launch_pair_many_cr(const CellTables &tab, const ManyIO &mio, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const int64_t n = mio.io.end - mio.io.begin;
    const bool small = (n + kThreads * kEPT - 1) / (kThreads * kEPT) < n_sm;
    if (mio.io.se_row)
        return small ? launch_pair_many_t<C, RNG, true, kManySmallThreads>(tab, mio, lut, n_sm, st)
                     : launch_pair_many_t<C, RNG, true, kThreads>(tab, mio, lut, n_sm, st);
    return small ? launch_pair_many_t<C, RNG, false, kManySmallThreads>(tab, mio, lut, n_sm, st)
                 : launch_pair_many_t<C, RNG, false, kThreads>(tab, mio, lut, n_sm, st);
}

template <int C>
cudaError_t launch_pair_c(const CellTables &tab, const StepIO &io, const uint2 *lut, int rng_mode, int n_sm,
                          cudaStream_t st)
{
    switch (rng_mode) {
    case GC_RNG_NONE: return launch_pair_cr<C, GC_RNG_NONE>(tab, io, lut, n_sm, st);
    case GC_RNG_PHILOX: return launch_pair_cr<C, GC_RNG_PHILOX>(tab, io, lut, n_sm, st);
    default: return launch_pair_cr<C, GC_RNG_REPLAY>(tab, io, lut, n_sm, st);
    }
}

}  // namespace

cudaError_t gc_launch_cell_pair_step(const CellTables &tab, const StepIO &io, const uint2 *lut, int rng_mode,
                                     int n_sm, cudaStream_t st)
{
    switch (tab.n_cells) {
#define GC_CASE(C) case C: return launch_pair_c<C>(tab, io, lut, rng_mode, n_sm, st);
        GC_CASE(1) GC_CASE(2) GC_CASE(3) GC_CASE(4) GC_CASE(5) GC_CASE(6) GC_CASE(7) GC_CASE(8)
        GC_CASE(9) GC_CASE(10) GC_CASE(11) GC_CASE(12) GC_CASE(13) GC_CASE(14) GC_CASE(15) GC_CASE(16)
#undef GC_CASE
    default: return cudaErrorInvalidValue;
    }
}

// gc_step_many in one launch: up to GC_MANY_MAX_CELLS cells (wider envs at these batch sizes are not launch-bound)
cudaError_t gc_launch_cell_pair_many(const CellTables &tab, const ManyIO &mio, const uint2 *lut, int rng_mode, int n_sm,
                                     cudaStream_t st)
{
    if (rng_mode != GC_RNG_NONE && rng_mode != GC_RNG_PHILOX) return cudaErrorInvalidValue;
    switch (tab.n_cells) {
#define GC_CASE(C) case C: return rng_mode == GC_RNG_PHILOX ? launch_pair_many_cr<C, GC_RNG_PHILOX>(tab, mio, lut, n_sm, st) \
                                                            : launch_pair_many_cr<C, GC_RNG_NONE>(tab, mio, lut, n_sm, st);
        GC_CASE(1) GC_CASE(2) GC_CASE(3) GC_CASE(4) GC_CASE(5) GC_CASE(6) GC_CASE(7) GC_CASE(8)
#undef GC_CASE
    default: return cudaErrorInvalidValue;
    }
}
