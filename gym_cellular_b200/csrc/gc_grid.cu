// Grid-world step (gym_cellular/envs/grid_world.py:107-179) as a table lookup.
//
// The deterministic part of the transition -- movement, tree death, regrowth, erosion, reward and
// the side-effect report -- is a function of (code_0, code_1, a_0, a_1) with 20*20*5*5 = 10,000
// cases; the host tabulates it once (gc_tables.cu: gc_build_grid_lut, closed form of :119-158) and
// each block stages the 40 KB table into shared memory.  Per env-step the kernel does one shared
// load; the seed-dispersal event (:160-162, probability 0.01; the trigger draws of four envs share one
// Philox block) patches the looked-up result in-line.
#include "gc_device.cuh"

namespace {


// Two blocks of 512 threads per SM: the 40 KB table is staged twice per SM instead of once per 256
// threads (staging traffic rivals the useful traffic for launches of a few million envs), and a block
// that drains frees half an SM, so that a kernel of another handle running on a second stream (the mixed
// workload: polarisation and grid world stepped concurrently) can move in.  Measured on that workload:
// 1024 x 1 -> 0.77, 256 x 4 -> 0.80, 384 x 2 -> 0.82, 512 x 2 -> 0.86 of the HBM roofline
// (profiles/r01_tuning_log.md); alone the geometries are within 2 % of each other.
constexpr int kGridThreads = 512;
constexpr int kGridMinBlocks = 2;
// Launches of up to kGridSmallIters 4-env words per thread read the table through L1 (`ld.global.nc`)
// instead of staging it: the staging phase (40 KB per block, serial with the block's work) is ~1 us of
// an 8 us launch there, while for long launches the shared-memory copy is the faster lookup
// (profiles/r01_tuning_log.md: 2^20 envs 130 -> 145 G env-steps/s in a CUDA graph, 2^22 envs 0.866 -> 0.841).
constexpr int kGridSmallIters = 3;
constexpr int kGridLutAlloc = GC_GRID_LUT_ALLOC;
constexpr int kGridSmemBytes = kGridLutAlloc * 4;

// One 4-env word of the grid-world step: everything from the table index to the last store, shared by the step
// kernel and the many-step kernel.  s0w / s1w and a0w / a1w are the code and action rows of the four envs (byte
// lane e = env e), tin their episode steps; lut is the table, in shared memory or (LUT_GLOBAL) read through L1.
// final_state, if not null, receives the rows before the auto-reset (the many-step kernel passes null: gc_step_many
// is never fused with a final-observation buffer, and a constant null keeps the test out of its loop).  The next
// rows and episode steps come back in row0 / row1 and tout, the statistics and the bad-action bits are accumulated.
template <int RNG, bool LUT_GLOBAL>
__device__ __forceinline__ void grid_word(const GridParams &gp, const StepIO &io, const uint32_t *lut, int8_t *final_state,
                                          uint32_t e0, int rem, uint64_t gid0, uint32_t step_counter, uint32_t s0w, uint32_t s1w, uint32_t a0w,
                                          uint32_t a1w, const int (&tin)[kEPT], uint32_t &st_count, uint32_t &st_trunc,
                                          uint32_t &st_reward, uint32_t &bad_bits, uint32_t &row0, uint32_t &row1,
                                          int (&tout)[kEPT])
{
    const uint32_t ld = static_cast<uint32_t>(io.ld);
    // Table index (code_0 + 20 code_1) * 25 + a_0 + 5 a_1 of the envs (0, 2) and (1, 3) in the two 16-bit
    // lanes of a word.  Codes are masked to 5 bits and actions to 3 bits, which bounds the index by
    // kGridLutAlloc: out-of-range inputs (never produced by the kernels) read padding, not foreign memory.
    const uint32_t s0m = s0w & 0x1F1F1F1Fu, s1m = s1w & 0x1F1F1F1Fu;
    const uint32_t actw = (a0w & 0x07070707u) + (a1w & 0x07070707u) * 5u;
    const uint32_t i02 = ((s0m & 0x00FF00FFu) + 20u * (s1m & 0x00FF00FFu)) * 25u + (actw & 0x00FF00FFu);
    const uint32_t i13 = (((s0m >> 8) & 0x00FF00FFu) + 20u * ((s1m >> 8) & 0x00FF00FFu)) * 25u + ((actw >> 8) & 0x00FF00FFu);
    uint32_t ent[kEPT];
    if (LUT_GLOBAL) {
        ent[0] = __ldg(lut + (i02 & 0xFFFFu)); ent[1] = __ldg(lut + (i13 & 0xFFFFu));
        ent[2] = __ldg(lut + (i02 >> 16)); ent[3] = __ldg(lut + (i13 >> 16));
    } else {
        ent[0] = lut[i02 & 0xFFFFu]; ent[1] = lut[i13 & 0xFFFFu];
        ent[2] = lut[i02 >> 16]; ent[3] = lut[i13 >> 16];
    }
    if (RNG == GC_RNG_PHILOX) {
        // Seed dispersal (grid_world.py:160-162): unless both jurisdictions were barren, one uniform
        // draw; below dispersal_prob the 2x2 bits and the jurisdiction index are drawn as well.  The
        // trigger words of the four envs of a thread are the four words of ONE Philox block (keyed by
        // global env id / 4) whenever they share the RNG counter, which they always do unless
        // episodic counters have drifted apart.
        uint32_t trig[kEPT];
        const uint64_t grp = gid0 >> 2;
        const bool same_t = !io.episodic || (tin[0] == tin[1] && tin[1] == tin[2] && tin[2] == tin[3]);
        if (same_t) {
            const uint32_t ctr = io.episodic ? static_cast<uint32_t>(tin[0]) : step_counter;
            philox4x32_10(static_cast<uint32_t>(grp), static_cast<uint32_t>(grp >> 32), ctr, 0u, io.round_key, trig);
        } else {
#pragma unroll 1
            for (int e = 0; e < kEPT; ++e) {
                uint32_t w[4];
                philox4x32_10(static_cast<uint32_t>(grp), static_cast<uint32_t>(grp >> 32),
                              static_cast<uint32_t>(tin[e]), 0u, io.round_key, w);
                trig[e] = w[e];
            }
        }
        // One test for the four envs (the event has probability 0.01 per env-step), then per env: the
        // drawn 2x2 bits (times tree_positions) replace jurisdiction k's trees (:162); reward and the
        // side-effect bits of the entry are redone from the packed tree masks (byte 0 / byte 1).
        // Given the trigger (word < p * 2^32) the low bits of the word are uniform up to 2^-25: they
        // serve as the three binary draws that matter, b00 = bit 0, b10 = bit 1, k = bit 2.
        const uint32_t thr = gp.dispersal_thr_m1;
        if (gp.dispersal_thr_nz && (trig[0] <= thr || trig[1] <= thr || trig[2] <= thr || trig[3] <= thr)) {
#pragma unroll
            for (int e = 0; e < kEPT; ++e) {
                uint32_t x = ent[e];
                const uint32_t w = trig[e];
                if (w <= thr && ((x >> 18) & 3u) < 2u) {
                    const uint32_t Nk = ((w >> 1) & 1u) | ((w & 1u) << 1);
                    const uint32_t sh = (w & 4u) << 1;                               // 8 k
                    x = (x & ~(3u << sh)) | (Nk << sh);
                    const uint32_t Tp = (byte_of(s0w, e) & 3u) | ((byte_of(s1w, e) & 3u) << 8);
                    const uint32_t Np = x & 0x0303u;
                    const uint32_t rew = __popc(Tp & ~Np);
                    const uint32_t se1 = (Np & 3u) ? 1u : 0u, se0 = (se1 && (Np & 0x0300u)) ? 1u : 0u;
                    ent[e] = (x & ~((3u << 16) | (3u << 20))) | (rew << 16) | (se0 << 20) | (se1 << 21);
                }
            }
        }
    } else {
#pragma unroll
        for (int e = 0; e < kEPT; ++e) {
            const uint32_t nb = (ent[e] >> 18) & 3u;
            const bool valid = e < rem;
            const double *u = io.replay + (valid ? static_cast<size_t>(e0 + e) * 6 : 0);
            if (nb < 2u && valid && u[0] < gp.dispersal_prob) {
                const uint32_t b00 = static_cast<uint32_t>(u[1] * 2.0), b10 = static_cast<uint32_t>(u[3] * 2.0);
                const uint32_t k = static_cast<uint32_t>(u[5] * 2.0);
                const uint32_t T0 = byte_of(s0w, e) & 3u, T1 = byte_of(s1w, e) & 3u;
                uint32_t nc0 = ent[e] & 0xFFu, nc1 = (ent[e] >> 8) & 0xFFu;
                const uint32_t Nk = b10 | (b00 << 1);
                if (k == 0u) nc0 = (nc0 & ~3u) | Nk; else nc1 = (nc1 & ~3u) | Nk;
                const uint32_t N0 = nc0 & 3u, N1 = nc1 & 3u;
                const uint32_t rew = __popc(T0 & ~N0) + __popc(T1 & ~N1);
                const uint32_t se0 = (N0 > 0u && N1 > 0u) ? 1u : 0u, se1 = (N0 > 0u) ? 1u : 0u;
                ent[e] = nc0 | (nc1 << 8) | (rew << 16) | (nb << 18) | (se0 << 20) | (se1 << 21) |
                         (ent[e] & (1u << 22));
            }
        }
    }
    // Everything below works on the four envs at once (byte lanes).  misc byte of an entry:
    // bits 0-1 reward, 2-3 barren jurisdictions, 4 / 5 side effects [0][0] / [0][1] 'safe', 6 bad action.
    const uint32_t m01 = prmt(ent[0], ent[1], 0x0062), m23 = prmt(ent[2], ent[3], 0x0062);
    const uint32_t miscw = prmt(m01, m23, 0x5410);
    const uint32_t vbytes = valid_bytes(rem);
    bad_bits |= miscw & vbytes;
    const uint32_t rew_w = miscw & 0x03030303u, count_w = (miscw >> 2) & 0x03030303u;
    const uint32_t se0w = (miscw >> 4) & 0x01010101u, se1w = (miscw >> 5) & 0x01010101u;
    const uint32_t u = prmt(ent[0], ent[1], 0x5140), v = prmt(ent[2], ent[3], 0x5140);
    row0 = prmt(u, v, 0x5410); row1 = prmt(u, v, 0x7632);                  // next codes, byte 0 / byte 1
    uint32_t trunc_w = 0;
#pragma unroll
    for (int e = 0; e < kEPT; ++e) tout[e] = tin[e] + 1;
    if (final_state) {                                                   // final observation: before the auto-reset
        st_stream_u32(final_state + e0, row0);
        st_stream_u32(final_state + (ld + e0), row1);
    }
    if (io.max_episode_steps > 0) {
#pragma unroll
        for (int e = 0; e < kEPT; ++e) {
            const bool tr = tout[e] >= io.max_episode_steps;
            tout[e] = tr ? 0 : tout[e];
            trunc_w |= (tr ? 1u : 0u) << (8 * e);
        }
        const uint32_t gone = trunc_w * 0xFFu;                               // byte mask of the envs that reset
        row0 = (row0 & ~gone) | (0x0F0F0F0Fu & gone);                       // reset codes 15 / 18: grid_world.py:238-259
        row1 = (row1 & ~gone) | (0x12121212u & gone);
    }
    float rout[kEPT];
#pragma unroll
    // reward byte -> float without a conversion: the byte becomes the low mantissa byte of 2^23 (one PRMT),
    // minus 2^23 (one FADD on the FMA pipe, which has room; the ALU pipe is what bounds this kernel)
    for (int e = 0; e < kEPT; ++e) rout[e] = __uint_as_float(prmt(rew_w, 0x4B000000u, 0x7540u + e)) - 8388608.0f;
    const uint32_t x02 = (row0 & 0x00FF00FFu) + 20u * (row1 & 0x00FF00FFu);             // code_0 + 20 code_1
    const uint32_t x13 = ((row0 >> 8) & 0x00FF00FFu) + 20u * ((row1 >> 8) & 0x00FF00FFu);
    st_count = add_bytes(count_w & vbytes, st_count);
    st_trunc = add_bytes(trunc_w & vbytes, st_trunc);
    st_reward = add_bytes(rew_w & vbytes, st_reward);
    st_stream_u32(io.state + e0, row0);
    st_stream_u32(io.state + (ld + e0), row1);
    if (io.se_row) {
        st_stream_u32(io.se_row + e0, se0w);
        st_stream_u32(io.se_row + (ld + e0), se1w);
    }
    st_stream_v4(io.t + e0, make_int4(tout[0], tout[1], tout[2], tout[3]));
    st_stream_v4(io.reward + e0, make_int4(__float_as_int(rout[0]), __float_as_int(rout[1]),
                                           __float_as_int(rout[2]), __float_as_int(rout[3])));
    st_stream_v4(io.index + e0, make_int4(x02 & 0xFFFFu, x13 & 0xFFFFu, x02 >> 16, x13 >> 16));
    st_stream_u32(io.terminated + e0, 0u);
    st_stream_u32(io.truncated + e0, trunc_w);
    st_stream_u32(io.unsafe + e0, 0u);                          // never 'unsafe': grid_world.py:174-175
    st_stream_u32(io.count + e0, count_w);
}

template <int RNG, bool LUT_GLOBAL>
__global__ void __launch_bounds__(kGridThreads, kGridMinBlocks)
grid_step_kernel(const __grid_constant__ GridParams gp, const __grid_constant__ StepIO io)
{
    extern __shared__ __align__(16) uint32_t s_lut[];          // kGridLutAlloc entries, the first 10,000 staged (unless LUT_GLOBAL)
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;
    // Element indexes are 32-bit (gc_create bounds n_cells * ld by 2^31): an address is then ONE IMAD.WIDE.U32 on
    // the FMA pipe instead of an IADD3 / IADD3.X pair on the ALU pipe, which is the pipe that bounds this kernel
    // (14 addresses per iteration; profiles/r02_kernel_cfg5.md: math_pipe_throttle 2.0).
    const uint32_t ld = static_cast<uint32_t>(io.ld);
    // Work partition: plain grid-stride loop.  (Round 2 tried contiguous per-block chunks of equal length --
    // a launch of 1.7 waves such as 2^20 envs leaves some SMs with 4 and some with 3 block-iterations under
    // grid-stride -- and measured it SLOWER on the same box: config 3 7.58 against 7.26 us per step, config 5
    // 0.812 against 0.870 of the HBM roofline; 296 separate streams lose the DRAM page locality of one sweep.)
    const uint32_t w_lo = blockIdx.x * kGridThreads, e_end = static_cast<uint32_t>(io.end);
    const uint32_t stride = gridDim.x * kGridThreads * kEPT;
    // The inputs of the NEXT 4-env word are requested before the current one is computed: a thread only
    // reads 32 bytes per word, so without the prefetch too few bytes are in flight per SM to cover the
    // HBM latency (ncu: long-scoreboard stalls dominate at 40 % occupancy).  The first word's inputs are
    // requested before the table is staged, so that the two latencies overlap.
    uint32_t e0 = static_cast<uint32_t>(io.begin) + (w_lo + threadIdx.x) * kEPT;
    // the immutable table is requested first (possibly while the previous step kernel of the stream is
    // still running: gc_device.cuh, programmatic dependent launch), then the first word's inputs, then
    // the table is stored to shared memory, so that the two latencies overlap
    constexpr int LUT_VEC = GC_GRID_LUT_ENTRIES / 4, LUT_PER_THREAD = (LUT_VEC + kGridThreads - 1) / kGridThreads;
    uint4 lut_reg[LUT_GLOBAL ? 1 : LUT_PER_THREAD];
    if (!LUT_GLOBAL) {
        const uint4 *src = reinterpret_cast<const uint4 *>(gp.lut);
#pragma unroll
        for (int k = 0; k < LUT_PER_THREAD; ++k) {
            const int i = threadIdx.x + k * kGridThreads;
            if (i < LUT_VEC) lut_reg[k] = src[i];
        }
    }
    // (Round 2 tried a `prefetch.global.L1` sweep over the table here for the LUT_GLOBAL variant, to take the L2
    // round trip of the first lookups off the critical path: 7.22 against 7.08 us per step at 2^20 envs on the
    // same box -- the 1,250 prefetches per block cost more than the misses they save; removed.)
    pdl_launch_dependents();
    pdl_wait();
    uint32_t p_s0 = 0, p_s1 = 0, p_a0 = 0, p_a1 = 0;
    int4 p_t = make_int4(0, 0, 0, 0);
    if (e0 < e_end) {
        p_s0 = ld_stream_u32(io.state + e0); p_s1 = ld_stream_u32(io.state + (ld + e0));
        p_a0 = ld_stream_u32(io.actions + e0); p_a1 = ld_stream_u32(io.actions + (ld + e0));
        p_t = ld_stream_v4(io.t + e0);
    }
    step_counter_read(io, &s_ctr);
    if (!LUT_GLOBAL) {
        uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
#pragma unroll
        for (int k = 0; k < LUT_PER_THREAD; ++k) {
            const int i = threadIdx.x + k * kGridThreads;
            if (i < LUT_VEC) dst[i] = lut_reg[k];
        }
    }
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    __syncthreads();

    const uint32_t step_counter = step_counter_arrive(io, &s_ctr);
    uint32_t st_count = 0, st_trunc = 0, st_reward = 0, bad_bits = 0;
    for (; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;
        const uint32_t s0w = p_s0, s1w = p_s1, a0w = p_a0, a1w = p_a1;
        const int tin[kEPT] = {p_t.x, p_t.y, p_t.z, p_t.w};
        if (e0 + stride < e_end) {
            const uint32_t en = e0 + stride;
            p_s0 = ld_stream_u32(io.state + en); p_s1 = ld_stream_u32(io.state + (ld + en));
            p_a0 = ld_stream_u32(io.actions + en); p_a1 = ld_stream_u32(io.actions + (ld + en));
            p_t = ld_stream_v4(io.t + en);
        }
        uint32_t row0, row1;
        int tout[kEPT];
        grid_word<RNG, LUT_GLOBAL>(gp, io, LUT_GLOBAL ? gp.lut : s_lut, io.final_state, e0, rem, gid0, step_counter, s0w, s1w, a0w, a1w, tin,
                                   st_count, st_trunc, st_reward, bad_bits, row0, row1, tout);
    }
    if (bad_bits & 0x40404040u) atomicOr(io.status, 1ull);
    if (io.stats)
        block_flush_stats_grid(st_count, st_trunc, st_reward, static_cast<unsigned long long>(io.end - io.begin), s_stats, io.stats);
    step_counter_finish(io, &s_ctr);
}

// ---------------------------------------------------------------------------------------------
// gc_step_many in ONE launch for small grid-world shards (gc_api.cu: many_fusable; see cell_pair_many_kernel in
// gc_cell_fast.cu): the thread that owns four envs runs their n_steps bound steps back to back -- codes and
// episode steps in registers, the actions of step k + 1 requested before step k is computed, the table staged
// once -- and writes every per-step output at every step as the separate launches do.  The step itself is the
// grid_word of grid_step_kernel's Philox path (same counters: global step of the launch + k), so the results are
// bit-identical to n_steps launches (tests/test_gpu_many.py).
__global__ void __launch_bounds__(kGridThreads, kGridMinBlocks)
grid_many_kernel(const __grid_constant__ GridParams gp, const __grid_constant__ ManyIO mio)
{
    const StepIO &io = mio.io;
    extern __shared__ __align__(16) uint32_t s_lut[];          // kGridLutAlloc entries (the padding included)
    __shared__ unsigned long long s_stats[5];
    __shared__ StepCounterShared s_ctr;
    const uint32_t ld = static_cast<uint32_t>(io.ld);
    const uint32_t e_end = static_cast<uint32_t>(io.end), stride = gridDim.x * kGridThreads * kEPT;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(gp.lut);
        uint4 *dst = reinterpret_cast<uint4 *>(s_lut);
        for (int i = threadIdx.x; i < kGridLutAlloc / 4; i += kGridThreads) dst[i] = src[i];
    }
    if (threadIdx.x < 5) s_stats[threadIdx.x] = 0;
    pdl_launch_dependents();
    pdl_wait();
    step_counter_read(io, &s_ctr);
    __syncthreads();
    const uint32_t step0 = step_counter_arrive(io, &s_ctr);
    uint32_t st_count = 0, st_trunc = 0, st_reward = 0, bad_bits = 0;
#pragma unroll 1
    for (uint32_t e0 = static_cast<uint32_t>(io.begin) + (blockIdx.x * kGridThreads + threadIdx.x) * kEPT; e0 < e_end; e0 += stride) {
        const int rem = static_cast<int>(e_end - e0 < kEPT ? e_end - e0 : kEPT);
        const uint64_t gid0 = static_cast<uint64_t>(io.env_id_offset) + e0;
        uint32_t s0w = ld_stream_u32(io.state + e0), s1w = ld_stream_u32(io.state + (ld + e0));
        uint32_t n_a0 = ld_stream_u32(mio.tape[0] + e0), n_a1 = ld_stream_u32(mio.tape[0] + (ld + e0));
        const int4 t4 = ld_stream_v4(io.t + e0);
        int tin[kEPT] = {t4.x, t4.y, t4.z, t4.w};
        int slot = 0;
#pragma unroll 1
        for (int k = 0; k < mio.n_steps; ++k) {
            const uint32_t a0w = n_a0, a1w = n_a1;
            slot = slot + 1 == mio.n_tape ? 0 : slot + 1;
            if (k + 1 < mio.n_steps) {
                const int8_t *const nxt = mio.tape[slot];
                n_a0 = ld_stream_u32(nxt + e0); n_a1 = ld_stream_u32(nxt + (ld + e0));
            }
            uint32_t row0, row1;
            int tout[kEPT];
            grid_word<GC_RNG_PHILOX, false>(gp, io, s_lut, nullptr, e0, rem, gid0, step0 + static_cast<uint32_t>(k), s0w, s1w, a0w, a1w, tin,
                                            st_count, st_trunc, st_reward, bad_bits, row0, row1, tout);
            s0w = row0; s1w = row1;
#pragma unroll
            for (int e = 0; e < kEPT; ++e) tin[e] = tout[e];
        }
    }
    if (bad_bits & 0x40404040u) atomicOr(io.status, 1ull);
    if (io.stats)
        block_flush_stats_grid(st_count, st_trunc, st_reward,
                               static_cast<unsigned long long>(io.end - io.begin) * static_cast<unsigned long long>(mio.n_steps),
                               s_stats, io.stats);
    step_counter_finish(io, &s_ctr, static_cast<uint32_t>(mio.n_steps));
}

}  // namespace

template <auto Kernel>
int grid_blocks(int64_t n, int n_sm, int smem_bytes, cudaError_t *err)
{
    // per device: the opt-in to more than 48 KB of dynamic shared memory is a per-device function attribute
    static int per_sm_dev[kMaxDevices] = {};
    const int slot = current_device_slot();
    int per_sm = per_sm_dev[slot];
    if (per_sm == 0 || slot == kMaxDevices - 1) {
        *err = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kGridSmemBytes);
        if (*err != cudaSuccess) return 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, Kernel, kGridThreads, smem_bytes) != cudaSuccess || per_sm < 1)
            per_sm = 1;
        per_sm_dev[slot] = per_sm;
    }
    // one wave of resident blocks: more waves (shorter grid-stride loops, blocks out of phase) measured 0.868 (1 wave),
    // 0.784 (2), 0.663 (4) of the config-5 roofline; the per-block fixed cost outweighs the de-phasing
    // (profiles/r01_tuning_log.md)
    const int64_t need = (n + kGridThreads * kEPT - 1) / (kGridThreads * kEPT);
    const int64_t cap = static_cast<int64_t>(n_sm) * per_sm;
    return static_cast<int>(need < cap ? (need < 1 ? 1 : need) : cap);
}

template <int RNG>
cudaError_t launch_grid(const GridParams &gp, const StepIO &io, int n_sm, cudaStream_t st)
{
    const int64_t n = io.end - io.begin;
    cudaError_t err = cudaSuccess;
    // words per thread if the table-staging kernel's one wave of blocks were launched
    const int64_t wave = static_cast<int64_t>(n_sm) * kGridMinBlocks * kGridThreads * kEPT;
    if (n <= wave * kGridSmallIters) {
        const int g = grid_blocks<grid_step_kernel<RNG, true>>(n, n_sm, 0, &err);
        if (err != cudaSuccess) return err;
        return launch_step_kernel(grid_step_kernel<RNG, true>, g, kGridThreads, 0, st, gp, io);
    } else {
        const int g = grid_blocks<grid_step_kernel<RNG, false>>(n, n_sm, kGridSmemBytes, &err);
        if (err != cudaSuccess) return err;
        return launch_step_kernel(grid_step_kernel<RNG, false>, g, kGridThreads, kGridSmemBytes, st, gp, io);
    }
    return cudaGetLastError();
}

cudaError_t gc_launch_grid_step(const GridParams &gp, const StepIO &io, int rng_mode, int n_sm, cudaStream_t st)
{
    return rng_mode == GC_RNG_REPLAY ? launch_grid<GC_RNG_REPLAY>(gp, io, n_sm, st)
                                     : launch_grid<GC_RNG_PHILOX>(gp, io, n_sm, st);
}

cudaError_t gc_launch_grid_many(const GridParams &gp, const ManyIO &mio, int n_sm, cudaStream_t st)
{
    cudaError_t err = cudaSuccess;
    const int g = grid_blocks<grid_many_kernel>(mio.io.end - mio.io.begin, n_sm, kGridSmemBytes, &err);
    if (err != cudaSuccess) return err;
    return launch_step_kernel(grid_many_kernel, g, kGridThreads, kGridSmemBytes, st, gp, mio);
}
