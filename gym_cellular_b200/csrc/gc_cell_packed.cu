// Packed layout of the cellular (polarisation) step for S, A <= 4 levels: ONE 32-bit word per env for the
// joint cell state and one for the joint action, 2 bits per cell (cell c in bits 2c, 2c+1).
//
// Why.  With four levels the reference's tabular index (generalized_space_transformations.py:1-12, cell 0
// least significant) IS this word, and tabular agents consume nothing but the index, the reward and the
// safety flag of cells3states3actions3.py:116-125.  The int8 structure-of-arrays layout moves 3C + 20 bytes
// per env-step (68 at 16 cells); this one moves
//     state 4 r + 4 w, action 4 r, t 4 r + 4 w, reward 4 w, flags 1 w            = 25 bytes
// (+4 for a separate index when S < 4), and on the host wire 4 bytes in, 9 bytes out instead of 16 / 26.
//
// Per env the work is one table lookup per cell PAIR, as in gc_cell_fast.cu, but the pair index falls out of
// the packed words with two LOP3 per eight pairs:
//     x = (aw << 4 & 0xF0F0F0F0) | (sw & 0x0F0F0F0F)     byte k = index of pair 2k     (s nibble | a nibble << 4)
//     y = (aw & 0xF0F0F0F0) | (sw >> 4 & 0x0F0F0F0F)     byte k = index of pair 2k + 1
// and the next state is rebuilt by a funnel shift per pair (the entry carries the pair's next levels in its
// top nibble: new = new << 4 | entry >> 28).  The info words of all pairs are simply ADDED: for each possible
// next level k of cell 0, how many cells would report 'unsafe' (the side-effect report of the cells j >= 2 is
// then one field extract by s'_0), and the polarised-cell count, in carry-free 5-bit fields (gc_tables.cu:
// gc_build_packed_lut).  Per (env, pair) that is PRMT + IMAD (address), LDS.64, FADD, IADD, SHF: the integer
// work is split between the two math pipes, which is what bounds the kernel once the bytes are this few.
//
// Shared-memory bank conflicts.  A warp's 32 random 64-bit table reads would serialise ~6-7-fold (measured on
// the int8 kernel, profiles/r01_kernel_cfg4.md); with 25 bytes per env-step that, not HBM, would bound the
// kernel.  Launches large enough to amortise the staging therefore replicate the table 16 times
// (deterministic, 256 entries -> 32 KB) or 4 times (stochastic, 1024 entries -> 32 KB): entry i of replica r
// sits at word i * REP + r and lane l reads replica l % REP, so the 16 lanes of a half-warp always hit 16
// different bank pairs.
#include "gc_device.cuh"

namespace {

constexpr int kPackThreads = 256;

// (a & m) | (b & ~m) in one LOP3
__device__ __forceinline__ uint32_t bitselect(uint32_t a, uint32_t b, uint32_t m)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(d) : "r"(a), "r"(b), "r"(m));
    return d;
}

// 64-bit shared-memory load from a 32-bit shared address (the tables are immutable after the staging barrier)
__device__ __forceinline__ uint2 lds64(uint32_t addr)
{
    uint2 v;
    asm("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}

// resident blocks per SM the register budget is sized for
#ifndef GC_PACKED_MINB
#define GC_PACKED_MINB 4
#endif

// table replication of a launch: log2 of the replica count (0 = plain table)
__host__ __device__ constexpr int packed_rep_log2(int rng, bool big) { return big ? (rng == GC_RNG_NONE ? 4 : 2) : 0; }
__host__ __device__ constexpr int packed_pairs(int rng) { return rng == GC_RNG_NONE ? 256 : GC_PAIR_LUT_PAIRS; }
__host__ __device__ constexpr int packed_singles(int rng) { return rng == GC_RNG_NONE ? 16 : 32; }
constexpr size_t packed_smem_bytes(int rng, bool big)
{
    return (static_cast<size_t>(packed_pairs(rng) + packed_singles(rng)) << packed_rep_log2(rng, big)) * sizeof(uint2) +
           GC_MAX_CELLS * GC_TBL;
}

// EXTRA: the launch also writes some of the optional outputs (separate tabular index for S < 4, final
// state before the auto-reset, row-0 side-effect codes); the plain variant carries no registers for them.
// the Philox and the optional-output variants carry ~16 more registers: budget of three blocks (85 registers)
__host__ __device__ constexpr int packed_min_blocks(int c, int rng, bool extra)
{
    // (15 cells: the 64-register build of the plain variant spills 8 bytes)
    return (rng != GC_RNG_NONE || extra || c == 15) ? (GC_PACKED_MINB < 3 ? GC_PACKED_MINB : 3) : GC_PACKED_MINB;
}

// One 4-env word of the packed step: everything between the loads of the inputs and the stores of the outputs,
// shared by the step kernel and the many-step kernel (the state words and episode steps a thread hands on to its
// next step come back in nstate / tn).
template <int C, int RNG, bool EXTRA>
__device__ __forceinline__ void packed_word(const CellTables &tab, const PackedIO &io, const uint8_t (*s_se)[GC_TBL],
                                            uint32_t pair_base, uint32_t single_base, uint32_t lut_mul, uint32_t e0, int rem,
                                            uint32_t gid_lo, uint32_t gid_hi, uint32_t step_counter,
                                            const uint32_t (&sw4)[kEPT], const uint32_t (&aw4)[kEPT], const int (&tin)[kEPT],
                                            uint32_t &st_steps, uint32_t &st_unsafe, uint32_t &st_count, uint32_t &st_trunc,
                                            long long &st_reward, uint32_t (&nstate)[kEPT], int (&tn)[kEPT])
{
    constexpr int NP = C / 2;                          // full pairs
    constexpr bool ODD = (C & 1) != 0;                 // plus a single last cell
    uint32_t fin[kEPT], idx[kEPT], sew[kEPT];
    uint32_t flags_w = 0;                          // flag bytes of the four envs
    float rew[kEPT];
#pragma unroll
    for (int e = 0; e < kEPT; ++e) {
        const uint32_t sw = sw4[e], aw = aw4[e];
        // fire bits of the env's cells: bit c = the noise draw of cell c fired (the table ignores the bit
        // where the (level, action) pair consumes no draw); same Philox words as the int8 kernels
        uint32_t fire = 0;
        if (RNG == GC_RNG_PHILOX) {
            const uint32_t ctr = io.episodic ? static_cast<uint32_t>(tin[e]) : step_counter;
            if (C > GC_NARROW_CELLS) {             // wide env: one block, a byte per cell (fire_bits_wide)
                fire = fire_bits_wide<(C + 7) / 8>(tab, gid_lo | e, gid_hi, ctr, io.round_key);
            } else {
                const uint32_t thr = tab.noise_thr_m1;
                uint32_t w[4];
                philox4x32_10(gid_lo | e, gid_hi, ctr, 0u, io.round_key, w);
                fire = (w[0] <= thr ? 1u : 0u) | (w[1] <= thr ? 2u : 0u) | (w[2] <= thr ? 4u : 0u) | (w[3] <= thr ? 8u : 0u);
            }
        }
        const uint32_t x = bitselect(aw << 4, sw, 0xF0F0F0F0u);       // (aw << 4 & M) | (sw & ~M)
        const uint32_t y = bitselect(aw, sw >> 4, 0xF0F0F0F0u);
        constexpr int NL = NP + (ODD ? 1 : 0);
        uint32_t info[NL];
        float r = 0.f;
#pragma unroll
        for (int i = 0; i < NP; ++i) {
            uint32_t ix = prmt((i & 1) ? y : x, 0u, 0x4440u + (i >> 1));      // byte i/2: the pair's index
            if (RNG != GC_RNG_NONE) ix |= ((fire >> (2 * i)) & 3u) << 8;
            const uint2 ent = lds64(ix * lut_mul + pair_base);
            r = (i == 0) ? __uint_as_float(ent.y) : r + __uint_as_float(ent.y);
            info[i] = ent.x;
        }
        if (ODD) {
            const uint32_t b = prmt((NP & 1) ? y : x, 0u, 0x4440u + (NP >> 1));
            uint32_t ix = (b & 3u) | ((b >> 2) & 12u);
            if (RNG != GC_RNG_NONE) ix |= ((fire >> (2 * NP)) & 1u) << 4;
            const uint2 ent = lds64(ix * lut_mul + single_base);
            r = (NP == 0) ? __uint_as_float(ent.y) : r + __uint_as_float(ent.y);
            info[NP] = ent.x;
        }
        uint32_t ns = 0, acc = 0;
#pragma unroll
        for (int i = NL - 1; i >= 0; --i) {
            ns = __funnelshift_l(info[i], ns, 4);              // ns << 4 | next nibble of lookup i
            acc += info[i];
        }
        // 'unsafe': the pair (cell 0, cell 1) flag, or some cell j >= 2 whose level the side-effect table of
        // s'_0 marks unsafe (field s'_0 of the summed info words of the lookups >= 1);
        // count: polarised cells of the next state
        const uint32_t lv = acc - info[0];
        const uint32_t uns2 = ((lv >> (5u * (ns & 3u))) & 31u) ? 1u : 0u;
        const uint32_t uns = ((info[0] >> 25) & 1u) | uns2;
        const uint32_t cnt = (acc >> 20) & 31u;
        uint32_t se_code = 0;
        if (EXTRA && io.se_row) {
            // row 0 of the side-effects matrix from the (pre-reset) next state: entry j from (s'_0, s'_p),
            // p = 1 for j = 0 and p = j otherwise
            const uint32_t s0n = ns & 3u;
#pragma unroll
            for (int j = 0; j < C; ++j) {
                const uint32_t p = (j == 0) ? (C > 1 ? 1 : 0) : j;
                const uint32_t sp = (ns >> (2 * p)) & 3u;
                se_code |= static_cast<uint32_t>(s_se[j][s0n * GC_LVL_PAD + sp]) << (2 * j);
            }
        }
        nstate[e] = ns; tn[e] = tin[e] + 1;
        if (EXTRA) { fin[e] = ns; sew[e] = se_code; }
        rew[e] = r;
        flags_w |= (uns | (cnt << 2)) << (8 * e);
    }
    if (io.max_episode_steps > 0) {                // time limit (uniform branch: the reference has none)
#pragma unroll
        for (int e = 0; e < kEPT; ++e)
            if (tn[e] >= io.max_episode_steps) { tn[e] = 0; nstate[e] = tab.init_packed; flags_w |= 2u << (8 * e); }
    }
#pragma unroll
    for (int e = 0; e < kEPT; ++e) {
        const uint32_t out = nstate[e];
        // tabular index of the returned state: the packed word itself for four levels
        if (EXTRA) {
            uint32_t ix = out;
            if (io.index && tab.n_states != 4) {
                ix = 0;
#pragma unroll
                for (int c = 0; c < C; ++c) ix += ((out >> (2 * c)) & 3u) * tab.place[c];
            }
            idx[e] = ix;
        }
    }
    float rout[kEPT];
    log2_1p_x4(tab.reward_log2, rew, rout);
#pragma unroll
    for (int e = 0; e < kEPT; ++e)
        if (e < rem) st_reward += __float2int_rn(rout[e] * 16777216.0f);
    {
        // statistics of the four envs from the flag word (envs beyond the range masked out)
        const uint32_t fw = flags_w & valid_bytes(rem);
        st_steps += rem;
        st_unsafe += __popc(fw & 0x01010101u);
        st_trunc += __popc(fw & 0x02020202u);
        st_count = add_bytes((fw >> 2) & 0x1F1F1F1Fu, st_count);
    }
    st_stream_v4(io.state + e0, make_int4(nstate[0], nstate[1], nstate[2], nstate[3]));
    st_stream_v4(io.t + e0, make_int4(tn[0], tn[1], tn[2], tn[3]));
    st_stream_v4(io.reward + e0, make_int4(__float_as_int(rout[0]), __float_as_int(rout[1]),
                                           __float_as_int(rout[2]), __float_as_int(rout[3])));
    st_stream_u32(io.flags + e0, flags_w);
    if (EXTRA) {
        if (io.index) st_stream_v4(io.index + e0, make_int4(idx[0], idx[1], idx[2], idx[3]));
        if (io.final_state) st_stream_v4(io.final_state + e0, make_int4(fin[0], fin[1], fin[2], fin[3]));
        if (io.se_row) st_stream_v4(io.se_row + e0, make_int4(sew[0], sew[1], sew[2], sew[3]));
    } else if (io.index) {       // four levels: the tabular index is the state word
        st_stream_v4(io.index + e0, make_int4(nstate[0], nstate[1], nstate[2], nstate[3]));
    }
}

template <int C, int RNG, bool EXTRA>
__global__ void __launch_bounds__(kPackThreads, packed_min_blocks(C, RNG, EXTRA))
cell_packed_kernel(const __grid_constant__ CellTables tab, const __grid_constant__ PackedIO io,
                   const uint2 *__restrict__ lut, const int REP_LOG2)
{
    constexpr int N_PAIR = packed_pairs(RNG), N_SINGLE = packed_singles(RNG);
    extern __shared__ __align__(16) uint2 s_tab[];     // [N_PAIR << REP_LOG2] pairs, [N_SINGLE << REP_LOG2] singles, side effects
    uint2 *const s_pair = s_tab;
    uint2 *const s_single = s_tab + (N_PAIR << REP_LOG2);
    uint8_t (*const s_se)[GC_TBL] = reinterpret_cast<uint8_t (*)[GC_TBL]>(s_single + (N_SINGLE << REP_LOG2));
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;
    const uint32_t REP = 1u << REP_LOG2;

    // 32-bit element indexes (n_cells * ld <= 2^31, gc_create): an address is one IMAD.WIDE.U32 on the FMA pipe
    const uint32_t stride = gridDim.x * kPackThreads * kEPT, e_end = static_cast<uint32_t>(io.end);
    uint32_t e0 = static_cast<uint32_t>(io.begin) + (blockIdx.x * kPackThreads + threadIdx.x) * kEPT;
    // immutable tables first (they may be read while the previous step kernel of the stream still runs)
    for (int i = threadIdx.x; i < (N_PAIR << REP_LOG2); i += kPackThreads) s_pair[i] = lut[i >> REP_LOG2];
    for (int i = threadIdx.x; i < (N_SINGLE << REP_LOG2); i += kPackThreads) s_single[i] = lut[GC_PAIR_LUT_PAIRS + (i >> REP_LOG2)];
    if (EXTRA && io.se_row)
        for (int i = threadIdx.x; i < C * GC_TBL; i += kPackThreads) s_se[i / GC_TBL][i % GC_TBL] = tab.se[i / GC_TBL][i % GC_TBL];
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    pdl_launch_dependents();
    pdl_wait();
    int4 ps = make_int4(0, 0, 0, 0), pa = ps, pt = ps;
    if (e0 < e_end) {
        ps = ld_stream_v4(io.state + e0);
        pa = ld_stream_v4(io.actions + e0);
        pt = ld_stream_v4(io.t + e0);
    }
    step_counter_read(io, &s_ctr);
    __syncthreads();
    const uint32_t step_now = step_counter_arrive(io, &s_ctr);
    const uint32_t step_counter = (RNG == GC_RNG_PHILOX) ? step_now : 0u;
    // shared-memory byte addresses: entry ix of this lane's replica sits at ix * lut_mul + lane base
    const uint32_t rep = threadIdx.x & (REP - 1u);
    const uint32_t lut_mul = 8u << REP_LOG2;
    const uint32_t pair_base = static_cast<uint32_t>(__cvta_generic_to_shared(s_pair)) + rep * 8u;
    const uint32_t single_base = static_cast<uint32_t>(__cvta_generic_to_shared(s_single)) + rep * 8u;

    uint32_t st_steps = 0, st_unsafe = 0, st_count = 0, st_trunc = 0;
    long long st_reward = 0;
    for (; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;
        const uint32_t gid_lo = static_cast<uint32_t>(gid0), gid_hi = static_cast<uint32_t>(gid0 >> 32);
        const uint32_t sw4[kEPT] = {(uint32_t)ps.x, (uint32_t)ps.y, (uint32_t)ps.z, (uint32_t)ps.w};
        const uint32_t aw4[kEPT] = {(uint32_t)pa.x, (uint32_t)pa.y, (uint32_t)pa.z, (uint32_t)pa.w};
        const int tin[kEPT] = {pt.x, pt.y, pt.z, pt.w};
        if (e0 + stride < e_end) {                     // the next word's inputs, before this one is computed
            ps = ld_stream_v4(io.state + (e0 + stride));
            pa = ld_stream_v4(io.actions + (e0 + stride));
            pt = ld_stream_v4(io.t + (e0 + stride));
        }
        uint32_t nstate[kEPT];
        int tn[kEPT];
        packed_word<C, RNG, EXTRA>(tab, io, s_se, pair_base, single_base, lut_mul, e0, rem, gid_lo, gid_hi, step_counter, sw4, aw4, tin,
                                   st_steps, st_unsafe, st_count, st_trunc, st_reward, nstate, tn);
    }
    if (io.stats) {
        const ThreadStats ts = {st_steps, st_unsafe, st_count, st_trunc, st_reward};
        block_flush_stats(ts, s_stats, io.stats);
    }
    step_counter_finish(io, &s_ctr);
}

// gc_step_many in ONE launch, packed layout (gc_api.cu: many_fusable; see cell_pair_many_kernel in gc_cell_fast.cu):
// the n_steps bound steps of a small shard whose packed bindings differ only in their action words.  State word
// and episode step stay in registers between two steps, the action words of step k + 1 are requested before step
// k is computed, every per-step output is written at every step by the same packed_word as the step kernel (so
// the results are bit-identical to n_steps launches), and the table is always replicated: its staging is paid
// once per launch.
template <int C, int RNG, bool EXTRA, int THREADS>
__global__ void __launch_bounds__(THREADS, 256 / THREADS * 2)
cell_packed_many_kernel(const __grid_constant__ CellTables tab, const __grid_constant__ PackedManyIO mio,
                        const uint2 *__restrict__ lut, const int REP_LOG2)
{
    const PackedIO &io = mio.io;
    constexpr int N_PAIR = packed_pairs(RNG), N_SINGLE = packed_singles(RNG);
    extern __shared__ __align__(16) uint2 s_tab[];
    uint2 *const s_pair = s_tab;
    uint2 *const s_single = s_tab + (N_PAIR << REP_LOG2);
    uint8_t (*const s_se)[GC_TBL] = reinterpret_cast<uint8_t (*)[GC_TBL]>(s_single + (N_SINGLE << REP_LOG2));
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;
    const uint32_t REP = 1u << REP_LOG2;
    const uint32_t stride = gridDim.x * THREADS * kEPT, e_end = static_cast<uint32_t>(io.end);
    for (int i = threadIdx.x; i < (N_PAIR << REP_LOG2); i += THREADS) s_pair[i] = lut[i >> REP_LOG2];
    for (int i = threadIdx.x; i < (N_SINGLE << REP_LOG2); i += THREADS) s_single[i] = lut[GC_PAIR_LUT_PAIRS + (i >> REP_LOG2)];
    if (EXTRA && io.se_row)
        for (int i = threadIdx.x; i < C * GC_TBL; i += THREADS) s_se[i / GC_TBL][i % GC_TBL] = tab.se[i / GC_TBL][i % GC_TBL];
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    pdl_launch_dependents();
    pdl_wait();
    step_counter_read(io, &s_ctr);
    __syncthreads();
    const uint32_t step0 = step_counter_arrive(io, &s_ctr);
    const uint32_t rep = threadIdx.x & (REP - 1u);
    const uint32_t lut_mul = 8u << REP_LOG2;
    const uint32_t pair_base = static_cast<uint32_t>(__cvta_generic_to_shared(s_pair)) + rep * 8u;
    const uint32_t single_base = static_cast<uint32_t>(__cvta_generic_to_shared(s_single)) + rep * 8u;

    uint32_t st_steps = 0, st_unsafe = 0, st_count = 0, st_trunc = 0;
    long long st_reward = 0;
#pragma unroll 1
    for (uint32_t e0 = static_cast<uint32_t>(io.begin) + (blockIdx.x * THREADS + threadIdx.x) * kEPT; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;
        const uint32_t gid_lo = static_cast<uint32_t>(gid0), gid_hi = static_cast<uint32_t>(gid0 >> 32);
        const int4 ps = ld_stream_v4(io.state + e0), pt = ld_stream_v4(io.t + e0);
        int4 an = ld_stream_v4(mio.tape[0] + e0);
        uint32_t sw4[kEPT] = {(uint32_t)ps.x, (uint32_t)ps.y, (uint32_t)ps.z, (uint32_t)ps.w};
        int tin[kEPT] = {pt.x, pt.y, pt.z, pt.w};
        int slot = 0;
#pragma unroll 1
        for (int k = 0; k < mio.n_steps; ++k) {
            const uint32_t aw4[kEPT] = {(uint32_t)an.x, (uint32_t)an.y, (uint32_t)an.z, (uint32_t)an.w};
            slot = slot + 1 == mio.n_tape ? 0 : slot + 1;
            if (k + 1 < mio.n_steps) an = ld_stream_v4(mio.tape[slot] + e0);
            const uint32_t step_counter = (RNG == GC_RNG_PHILOX) ? step0 + static_cast<uint32_t>(k) : 0u;
            uint32_t nstate[kEPT];
            int tn[kEPT];
            packed_word<C, RNG, EXTRA>(tab, io, s_se, pair_base, single_base, lut_mul, e0, rem, gid_lo, gid_hi, step_counter, sw4, aw4,
                                       tin, st_steps, st_unsafe, st_count, st_trunc, st_reward, nstate, tn);
#pragma unroll
            for (int e = 0; e < kEPT; ++e) { sw4[e] = nstate[e]; tin[e] = tn[e]; }
        }
    }
    if (io.stats) {
        const ThreadStats ts = {st_steps, st_unsafe, st_count, st_trunc, st_reward};
        block_flush_stats(ts, s_stats, io.stats);
    }
    step_counter_finish(io, &s_ctr, static_cast<uint32_t>(mio.n_steps));
}

template <int C, int RNG, bool EXTRA, int THREADS>
cudaError_t launch_packed_many_t(const CellTables &tab, const PackedManyIO &mio, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const auto kernel = cell_packed_many_kernel<C, RNG, EXTRA, THREADS>;
    const int64_t n = mio.io.end - mio.io.begin;
    const size_t smem = packed_smem_bytes(RNG, true);
    static int per_sm = 0;
    if (per_sm == 0 &&
        (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, THREADS, smem) != cudaSuccess || per_sm < 1))
        per_sm = 1;
    const int64_t need = (n + THREADS * kEPT - 1) / (THREADS * kEPT);
    const int64_t cap = static_cast<int64_t>(n_sm) * per_sm;
    const int grid = static_cast<int>(need < cap ? (need < 1 ? 1 : need) : cap);
    return launch_step_kernel(kernel, grid, THREADS, smem, st, tab, mio, lut, packed_rep_log2(RNG, true));
}

// shards that do not fill every SM with 256-thread blocks take smaller blocks (kManySmallThreads)
template <int C, int RNG, bool EXTRA>
cudaError_t launch_packed_many_cre(const CellTables &tab, const PackedManyIO &mio, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const int64_t n = mio.io.end - mio.io.begin;
    const bool small = (n + kPackThreads * kEPT - 1) / (kPackThreads * kEPT) < n_sm;
    return small ? launch_packed_many_t<C, RNG, EXTRA, kManySmallThreads>(tab, mio, lut, n_sm, st)
                 : launch_packed_many_t<C, RNG, EXTRA, kPackThreads>(tab, mio, lut, n_sm, st);
}

template <int C, int RNG>
cudaError_t launch_packed_many_cr(const CellTables &tab, const PackedManyIO &mio, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const PackedIO &io = mio.io;
    const bool extra = io.final_state || io.se_row || (io.index && tab.n_states != 4);
    return extra ? launch_packed_many_cre<C, RNG, true>(tab, mio, lut, n_sm, st)
                 : launch_packed_many_cre<C, RNG, false>(tab, mio, lut, n_sm, st);
}

// launches of at least this many envs replicate the table (staging 32 KB per block pays off)
#ifndef GC_PACKED_BIG_ENVS
#define GC_PACKED_BIG_ENVS (1 << 21)
#endif

template <int C, int RNG, bool EXTRA>
cudaError_t launch_packed_cre(const CellTables &tab, const PackedIO &io, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const auto kernel = cell_packed_kernel<C, RNG, EXTRA>;
    const int64_t n = io.end - io.begin;
    const bool big = n >= GC_PACKED_BIG_ENVS;
    const size_t smem = packed_smem_bytes(RNG, big);
    static int per_sm[2] = {0, 0};          // resident blocks per SM, plain / replicated table (same on every device)
    if (per_sm[big] == 0 &&
        (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[big], kernel, kPackThreads, smem) != cudaSuccess || per_sm[big] < 1))
        per_sm[big] = 1;
    const int64_t need = (n + kPackThreads * kEPT - 1) / (kPackThreads * kEPT);
    const int64_t cap = static_cast<int64_t>(n_sm) * per_sm[big];
    const int grid = static_cast<int>(need < cap ? (need < 1 ? 1 : need) : cap);
    return launch_step_kernel(kernel, grid, kPackThreads, smem, st, tab, io, lut, packed_rep_log2(RNG, big));
}

template <int C, int RNG>
cudaError_t launch_packed_cr(const CellTables &tab, const PackedIO &io, const uint2 *lut, int n_sm, cudaStream_t st)
{
    const bool extra = io.final_state || io.se_row || (io.index && tab.n_states != 4);
    return extra ? launch_packed_cre<C, RNG, true>(tab, io, lut, n_sm, st)
                 : launch_packed_cre<C, RNG, false>(tab, io, lut, n_sm, st);
}

// ---------------------------------------------------------------------------------------------
// reset() in the packed layout (cells3states3actions3.py:99-113): state word, t = 0, tabular index
__global__ void __launch_bounds__(kPackThreads)
reset_packed_kernel(uint32_t init_packed, uint32_t init_index, const uint8_t *__restrict__ mask, uint32_t *state,
                    int32_t *t, uint32_t *index, int64_t n)
{
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kPackThreads;
    for (int64_t e = static_cast<int64_t>(blockIdx.x) * kPackThreads + threadIdx.x; e < n; e += stride) {
        if (mask != nullptr && mask[e] == 0) continue;
        state[e] = init_packed;
        t[e] = 0;
        if (index) index[e] = init_index;
    }
}

// int8 [n_cells][ld] levels <-> packed words [ld] (2 bits per cell): the bridge between the two layouts
__global__ void __launch_bounds__(kPackThreads)
pack_kernel(int64_t n, int64_t ld, int n_cells, const int8_t *__restrict__ cells, uint32_t *__restrict__ packed)
{
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kPackThreads * kEPT;
    for (int64_t e0 = (static_cast<int64_t>(blockIdx.x) * kPackThreads + threadIdx.x) * kEPT; e0 < n; e0 += stride) {
        uint32_t w[kEPT] = {0, 0, 0, 0};
        for (int c = 0; c < n_cells; ++c) {
            const uint32_t row = ld_stream_u32(cells + c * ld + e0);
#pragma unroll
            for (int e = 0; e < kEPT; ++e) w[e] |= (byte_of(row, e) & 3u) << (2 * c);
        }
        st_stream_v4(packed + e0, make_int4(w[0], w[1], w[2], w[3]));
    }
}

__global__ void __launch_bounds__(kPackThreads)
unpack_kernel(int64_t n, int64_t ld, int n_cells, const uint32_t *__restrict__ packed, int8_t *__restrict__ cells)
{
    const int64_t stride = static_cast<int64_t>(gridDim.x) * kPackThreads * kEPT;
    for (int64_t e0 = (static_cast<int64_t>(blockIdx.x) * kPackThreads + threadIdx.x) * kEPT; e0 < n; e0 += stride) {
        const int4 v = ld_stream_v4(packed + e0);
        const uint32_t w[kEPT] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
        for (int c = 0; c < n_cells; ++c) {
            uint32_t row = 0;
#pragma unroll
            for (int e = 0; e < kEPT; ++e) row |= ((w[e] >> (2 * c)) & 3u) << (8 * e);
            st_stream_u32(cells + c * ld + e0, row);
        }
    }
}

int aux_grid(int64_t n, int per_thread)
{
    const int64_t need = (n + static_cast<int64_t>(kPackThreads) * per_thread - 1) / (static_cast<int64_t>(kPackThreads) * per_thread);
    return static_cast<int>(need < 1 ? 1 : (need > 65535 ? 65535 : need));
}

}  // namespace

cudaError_t gc_launch_cell_packed_step(const CellTables &tab, const PackedIO &io, const uint2 *lut, bool noise,
                                       int n_sm, cudaStream_t st)
{
    switch (tab.n_cells) {
#define GC_CASE(C)                                                                                  \
    case C:                                                                                         \
        return noise ? launch_packed_cr<C, GC_RNG_PHILOX>(tab, io, lut, n_sm, st)                   \
                     : launch_packed_cr<C, GC_RNG_NONE>(tab, io, lut, n_sm, st);
        GC_CASE(1) GC_CASE(2) GC_CASE(3) GC_CASE(4) GC_CASE(5) GC_CASE(6) GC_CASE(7) GC_CASE(8)
        GC_CASE(9) GC_CASE(10) GC_CASE(11) GC_CASE(12) GC_CASE(13) GC_CASE(14) GC_CASE(15) GC_CASE(16)
#undef GC_CASE
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t gc_launch_cell_packed_many(const CellTables &tab, const PackedManyIO &mio, const uint2 *lut, bool noise, int n_sm,
                                       cudaStream_t st)
{
    switch (tab.n_cells) {
#define GC_CASE(C)                                                                                  \
    case C:                                                                                         \
        return noise ? launch_packed_many_cr<C, GC_RNG_PHILOX>(tab, mio, lut, n_sm, st)             \
                     : launch_packed_many_cr<C, GC_RNG_NONE>(tab, mio, lut, n_sm, st);
        GC_CASE(1) GC_CASE(2) GC_CASE(3) GC_CASE(4) GC_CASE(5) GC_CASE(6) GC_CASE(7) GC_CASE(8)
#undef GC_CASE
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t gc_launch_reset_packed(uint32_t init_packed, uint32_t init_index, const uint8_t *mask, uint32_t *state,
                                   int32_t *t, uint32_t *index, int64_t n, cudaStream_t st)
{
    reset_packed_kernel<<<aux_grid(n, 1), kPackThreads, 0, st>>>(init_packed, init_index, mask, state, t, index, n);
    return cudaGetLastError();
}

cudaError_t gc_launch_pack(int64_t n, int64_t ld, int n_cells, const int8_t *cells, uint32_t *packed, cudaStream_t st)
{
    pack_kernel<<<aux_grid(n, kEPT), kPackThreads, 0, st>>>(n, ld, n_cells, cells, packed);
    return cudaGetLastError();
}

cudaError_t gc_launch_unpack(int64_t n, int64_t ld, int n_cells, const uint32_t *packed, int8_t *cells, cudaStream_t st)
{
    unpack_kernel<<<aux_grid(n, kEPT), kPackThreads, 0, st>>>(n, ld, n_cells, packed, cells);
    return cudaGetLastError();
}
