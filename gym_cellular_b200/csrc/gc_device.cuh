// Device-side helpers shared by the kernel translation units.
#pragma once
#include "gc_internal.h"
#include <cstdlib>
#include <utility>

namespace {

constexpr int kThreads = 256;
constexpr int kEPT = 4;
// Block size of the many-step kernels for shards that do not fill every SM with 256-thread blocks (65,536 envs =
// 64 of them): such a shard is spread over more SMs, since its steps are bound by the dependent-instruction latency
// of its warps (config 2, same box: 99-106 G env-steps/s with 256-thread blocks, 117-140 with 128, 132 with 64;
// packed 113-122 / 117-120 / 127-128).
constexpr int kManySmallThreads = 64;

// ---------------------------------------------------------------------------------------------
// Philox4x32-10, counter based: word w of env e at step t = philox(key=seed, ctr=(e_lo,e_hi,t,w/4))[w%4].
// rk = the ten round keys (k0 + r*W0, k1 + r*W1), warp-uniform (StepIO::round_key): a round is two
// 32x32->64 multiplies and two three-input XORs.
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              const uint32_t (&rk)[20], uint32_t (&out)[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = static_cast<unsigned long long>(0xD2511F53u) * c0;
        const unsigned long long p1 = static_cast<unsigned long long>(0xCD9E8D57u) * c2;
        c0 = static_cast<uint32_t>(p1 >> 32) ^ c1 ^ rk[2 * r];
        c1 = static_cast<uint32_t>(p1);
        c2 = static_cast<uint32_t>(p0 >> 32) ^ c3 ^ rk[2 * r + 1];
        c3 = static_cast<uint32_t>(p0);
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { return __byte_perm(a, b, sel); }

// ---------------------------------------------------------------------------------------------
// Noise draws of a WIDE env (more than GC_NARROW_CELLS cells; cells3resetVdeadlock.py:35-41 scaled up).
// One Philox block serves EIGHT cells: 16-bit half h = c % 8 of the block philox(env, t, c / 8) (half h = the
// low (h even) or high (h odd) half of word h / 2) is the TOP half of cell c's 32-bit draw.  With
// threshold = k16 * 2^16 + r16 (= ceil(p * 2^32)) the draw fires iff
//     half < k16,  or  half == k16 and low16 < r16,
// low16 = word 0 >> 16 of the block philox(env, t, GC_NOISE_LOW_STREAM + c), computed only on a tie (2^-16 per
// cell).  P(fire) = k16 / 2^16 + r16 / 2^32 = threshold / 2^32 exactly, as for the 32-bit draws of narrow envs;
// the oracle always forms the full 32-bit value (top half << 16 | low16) and compares u = value * 2^-32 < p.
// The compares run two at a time (SWAR): for x, k in one 16-bit lane, H = 0x8000, L = 0x7FFF,
//     d = (x | H) - (k & L)     bit 15 of d  <=>  (x & L) >= (k & L)   (no borrow between the lanes)
//     x < k  <=>  (~x15 & k15) | (~(x15 ^ k15) & ~d15)
// and the two result bits of a word are gathered with one multiply (bits 15, 31 -> 30, 31).
// Returns bit c = the draw of cell c fired, for c < 8 * NB (NB Philox blocks).

// The rare part, kept out of line so that its registers do not weigh on the callers: some half of this env ties with
// the threshold's top half, so its draws are formed again block by block, with the low halves of the tied ones.
// The round keys are rebuilt from the seed (k + r * W) instead of being read through a pointer: a warp that gets
// here holds up its whole block, so the path is short even though it is rare (once per ~120 warp iterations).
__device__ __forceinline__ void philox4x32_10_seeded(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned long long p0 = static_cast<unsigned long long>(0xD2511F53u) * c[0];
        const unsigned long long p1 = static_cast<unsigned long long>(0xCD9E8D57u) * c[2];
        c[0] = static_cast<uint32_t>(p1 >> 32) ^ c[1] ^ k0;
        c[1] = static_cast<uint32_t>(p1);
        c[2] = static_cast<uint32_t>(p0 >> 32) ^ c[3] ^ k1;
        c[3] = static_cast<uint32_t>(p0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

__device__ __noinline__ uint32_t noise_fire_with_ties(int n_blocks, uint32_t k16, uint32_t r16, uint32_t gid_lo, uint32_t gid_hi,
                                                      uint32_t ctr, uint32_t seed_lo, uint32_t seed_hi)
{
    uint32_t fire = 0, ties = 0;
#pragma unroll 1
    for (int b = 0; b < n_blocks; ++b) {
        uint32_t w[4] = {gid_lo, gid_hi, ctr, static_cast<uint32_t>(b)};
        philox4x32_10_seeded(w, seed_lo, seed_hi);
#pragma unroll
        for (int h = 0; h < 8; ++h) {
            const uint32_t half = (h & 1) ? w[h >> 1] >> 16 : w[h >> 1] & 0xFFFFu;
            if (half < k16) fire |= (1u << h) << (8 * b);
            if (half == k16) ties |= (1u << h) << (8 * b);
        }
    }
    while (ties) {
        const uint32_t c = static_cast<uint32_t>(__ffs(static_cast<int>(ties))) - 1u;
        ties &= ties - 1u;
        uint32_t lo[4] = {gid_lo, gid_hi, ctr, GC_NOISE_LOW_STREAM + c};
        philox4x32_10_seeded(lo, seed_lo, seed_hi);
        if ((lo[0] >> 16) < r16) fire |= 1u << c;
    }
    return fire;
}

// Ties are detected once per env, not per word: the lane-wise minimum of (half ^ k16) over the block's eight halves
// (two VIMNMX3.U16x2 per block) has a zero lane iff some half equals k16.  Measured against the per-word
// equality masks of the first form: 294 -> 284 us per step at 16 cells x 4 levels x 2^24 envs (int8 layout),
// 207 -> 197 us packed.  Forms that moved the compares onto the FMA pipe (an IMAD for d, one 64-bit multiply-add
// as the gather, a three-input compare per value of k16's top bit) were measured slower and are not kept
// (profiles/r02_tuning_log.md).
template <int NB>
__device__ __forceinline__ uint32_t fire_bits_wide(const CellTables &tab, uint32_t gid_lo, uint32_t gid_hi, uint32_t ctr,
                                                   const uint32_t (&rk)[20])
{
    constexpr uint32_t H = 0x80008000u, L = 0x7FFF7FFFu, GATHER = 0x00008001u;
    uint32_t zmin = 0xFFFFFFFFu, fire = 0;
#pragma unroll
    for (int b = NB - 1; b >= 0; --b) {
        uint32_t w[4];
        philox4x32_10(gid_lo, gid_hi, ctr, static_cast<uint32_t>(b), rk, w);
#pragma unroll
        for (int i = 3; i >= 0; --i) {
            const uint32_t x = w[i];
            const uint32_t d = (x | H) - tab.noise_kk15;
            const uint32_t lt = ~((x & d) | ((x | d) & ~tab.noise_kmask)) & H;
            fire = __funnelshift_l(lt * GATHER, fire, 2);
        }
        zmin = __vimin3_u16x2(zmin, w[0] ^ tab.noise_kk, w[1] ^ tab.noise_kk);
        zmin = __vimin3_u16x2(zmin, w[2] ^ tab.noise_kk, w[3] ^ tab.noise_kk);
    }
    if (~(((zmin & L) + L) | zmin) & H)               // rare (2^-16 per cell): a half ties with the threshold's top half
        fire = noise_fire_with_ties(NB, tab.noise_kk & 0xFFFFu, tab.noise_r16, gid_lo, gid_hi, ctr, rk[0], rk[1]);
    return fire;
}

// byte e of w, zero-extended
__device__ __forceinline__ uint32_t byte_of(uint32_t w, int e)
{
#ifdef GC_BYTE_OF_PRMT
    return __byte_perm(w, 0u, 0x4440u + static_cast<uint32_t>(e));   // one PRMT (bytes 4.. = the zero operand)
#else
    return (w >> (8 * e)) & 0xFFu;
#endif
}

// streaming accesses: every byte is used once, keep it out of L1
__device__ __forceinline__ uint32_t ld_stream_u32(const void *p)
{
    return __ldcs(reinterpret_cast<const unsigned int *>(p));
}
__device__ __forceinline__ void st_stream_u32(void *p, uint32_t v)
{
    __stcs(reinterpret_cast<unsigned int *>(p), v);
}
__device__ __forceinline__ int4 ld_stream_v4(const void *p) { return __ldcs(reinterpret_cast<const int4 *>(p)); }
__device__ __forceinline__ void st_stream_v4(void *p, int4 v) { __stcs(reinterpret_cast<int4 *>(p), v); }

// Per-thread statistics, reduced once per block at kernel exit: REDUX.SUM over the warp, one shared-memory
// atomic per warp, one global atomic per block and statistic.
struct ThreadStats {
    uint32_t steps, unsafe, count, truncated;     // per thread and launch: < 2^32
    long long reward_q24;
};

// Global step of the launch: device-resident when the launch covers the whole shard (so that a captured
// CUDA graph advances its RNG counter on every replay), else the value the host passed.
template <class IO>
__device__ __forceinline__ uint32_t launch_step_counter(const IO &io)
{
    // (not a ?: of a volatile and a plain lvalue: that makes the parameter read itself volatile and
    // sends it through a generic-address load of the kernel parameter block)
    uint32_t v = io.rng_counter;
    if (io.step_ctr != nullptr) v = *reinterpret_cast<const volatile uint32_t *>(io.step_ctr);
    return v;
}

// Called by every thread at kernel exit: the last block to arrive advances the device step counter.
// Every thread read the counter at kernel entry, before its block's arrival, so no block can observe
// the incremented value within the same launch.
__device__ __forceinline__ void tick_step_counter(const uint32_t *step_ctr, uint32_t *done_ctr, uint32_t inc)
{
    if (done_ctr == nullptr) return;         // read-only counter: a chunk of a chunked pass (the caller ticks)
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t arrived = atomicAdd(done_ctr, 1u);
        if (arrived == gridDim.x - 1) {
            *done_ctr = 0u;
            *const_cast<uint32_t *>(step_ctr) = *reinterpret_cast<const volatile uint32_t *>(step_ctr) + inc;
        }
    }
}

template <class IO>
__device__ __forceinline__ void tick_step_counter(const IO &io) { tick_step_counter(io.step_ctr, io.done_ctr, 1u); }

// The same protocol with the arrival moved to the START of the kernel, so that no atomic round trip and
// no barrier sit on the kernel's tail (they are ~1 us of a launch-bound 4 us step):
//   step_counter_read    before the block's first __syncthreads: thread 0 copies the counter to shared
//                        memory (the store needs the loaded value, so the load has completed at the barrier)
//   step_counter_arrive  after that barrier: thread 0 arrives; every thread gets the step from shared memory
//   step_counter_finish  at kernel exit: the block that arrived last advances the counter by the launch's steps.
// Every block has read the counter before it arrives, so when the last arrival is known nobody of this
// launch reads the counter any more; the next launch starts after this one has completed.
struct StepCounterShared { uint32_t step, arrived; };

template <class IO>
__device__ __forceinline__ void step_counter_read(const IO &io, StepCounterShared *s)
{
    if (threadIdx.x == 0) s->step = launch_step_counter(io);
}

template <class IO>
__device__ __forceinline__ uint32_t step_counter_arrive(const IO &io, StepCounterShared *s)
{
    if (threadIdx.x == 0 && io.done_ctr != nullptr) s->arrived = atomicAdd(io.done_ctr, 1u);
    return s->step;
}

template <class IO>
__device__ __forceinline__ void step_counter_finish(const IO &io, const StepCounterShared *s, uint32_t n_steps = 1u)
{
    if (threadIdx.x == 0 && io.done_ctr != nullptr && s->arrived == gridDim.x - 1) {
        *io.done_ctr = 0u;
        *const_cast<uint32_t *>(io.step_ctr) = s->step + n_steps;
    }
}

// log2(1 + r) of the `nonlinear` rewards (np.log2(1 + .), cells3states3actions3.py:47-49) to ~4e-7
// relative: for -1/2 <= r <= 1 (always, for the reference's 2- and 3-cell envs) 2 atanh(s) / ln 2 with
// s = r / (2 + r), |s| <= 1/3, as a degree-6 polynomial in s^2 with 2 / ln 2 folded into the
// coefficients (10 FMA-pipe instructions and one MUFU.RCP instead of the ~25 of log1pf); log1pf beyond.
__device__ __forceinline__ float log2_1p_small(float r)
{
    float s;
    asm("div.approx.ftz.f32 %0, %1, %2;" : "=f"(s) : "f"(r), "f"(2.0f + r));
    const float z = s * s;
    constexpr float k = 2.88539008177792681f;                // 2 / ln 2
    float p = k / 13.0f;
    p = fmaf(p, z, k / 11.0f);
    p = fmaf(p, z, k / 9.0f);
    p = fmaf(p, z, k / 7.0f);
    p = fmaf(p, z, k / 5.0f);
    p = fmaf(p, z, k / 3.0f);
    p = fmaf(p, z, k);
    return s * p;
}

__device__ __forceinline__ float log2_1p(float r)
{
    if (r >= -0.5f && r <= 1.0f) return log2_1p_small(r);
    return log1pf(r) * 1.44269504088896341f;
}

// The same for the four envs of a thread: one range test (two FMNMX trees) guards the polynomial path
// of all four, so the common case carries no per-env branch.  A word with some sum outside [-1/2, 1] takes
// log2_1p env by env, so that every env's reward is a function of its own sum (the one the generic kernel
// computes), whatever the three other envs of its word hold.
__device__ __forceinline__ void log2_1p_x4(int enabled, const float (&r)[4], float (&out)[4])
{
    if (!enabled) {
#pragma unroll
        for (int e = 0; e < 4; ++e) out[e] = r[e];
        return;
    }
    const float hi = fmaxf(fmaxf(r[0], r[1]), fmaxf(r[2], r[3])), lo = fminf(fminf(r[0], r[1]), fminf(r[2], r[3]));
    if (lo >= -0.5f && hi <= 1.0f) {
#pragma unroll
        for (int e = 0; e < 4; ++e) out[e] = log2_1p_small(r[e]);
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) out[e] = log2_1p(r[e]);
    }
}

// byte mask of the envs of a 4-env word that lie inside the launch range (rem = envs left, >= 1)
__device__ __forceinline__ uint32_t valid_bytes(int rem) { return rem >= 4 ? 0xFFFFFFFFu : ((1u << (8 * rem)) - 1u); }

// sum of the four bytes of w added to acc (one IDP.4A)
__device__ __forceinline__ uint32_t add_bytes(uint32_t w, uint32_t acc) { return __dp4a(w, 0x01010101u, acc); }

// Sum of a 64-bit value over the warp with three REDUX.SUM instead of ten shuffles: the two 16-bit
// halves of the low word cannot overflow 32 bits over 32 lanes, and the high words add modulo 2^32,
// which is what their place in a 64-bit sum (modulo 2^64, signed or not) requires.
__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v)
{
    const uint32_t lo = static_cast<uint32_t>(v), hi = static_cast<uint32_t>(v >> 32);
    const uint32_t a = __reduce_add_sync(0xffffffffu, lo & 0xFFFFu);
    const uint32_t b = __reduce_add_sync(0xffffffffu, lo >> 16);
    const uint32_t c = __reduce_add_sync(0xffffffffu, hi);
    return static_cast<unsigned long long>(a) + (static_cast<unsigned long long>(b) << 16) +
           (static_cast<unsigned long long>(c) << 32);
}

__device__ __forceinline__ unsigned long long warp_sum(uint32_t v)
{
    const uint32_t a = __reduce_add_sync(0xffffffffu, v & 0xFFFFu);
    const uint32_t b = __reduce_add_sync(0xffffffffu, v >> 16);
    return static_cast<unsigned long long>(a) + (static_cast<unsigned long long>(b) << 16);
}

__device__ __forceinline__ void block_flush_stats(const ThreadStats &ts, unsigned long long *s_stats,
                                                  unsigned long long *g_stats)
{
    // s_stats zeroed before the main loop (with a __syncthreads in between)
    const unsigned long long w[5] = {warp_sum(ts.steps), warp_sum(ts.unsafe), warp_sum(ts.count), warp_sum(ts.truncated),
                                     warp_sum(static_cast<unsigned long long>(ts.reward_q24))};
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int i = 0; i < 5; ++i)
            if (w[i]) atomicAdd(&s_stats[i], w[i]);
    }
    __syncthreads();
    if (threadIdx.x < 5 && s_stats[threadIdx.x]) atomicAdd(&g_stats[threadIdx.x], s_stats[threadIdx.x]);
}

// Grid world: 'unsafe' is constant 0 (grid_world.py:174-175), the rewards are small integers (a 32-bit sum per
// thread), and the env-step count of a launch is known before it runs: 6 REDUX instead of 11 at the tail of a
// kernel that lasts 7 us at 2^20 envs.
__device__ __forceinline__ void block_flush_stats_grid(uint32_t count, uint32_t truncated, uint32_t reward,
                                                       unsigned long long launch_steps, unsigned long long *s_stats,
                                                       unsigned long long *g_stats)
{
    const unsigned long long w[3] = {warp_sum(count), warp_sum(truncated), warp_sum(reward) << 24};
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int i = 0; i < 3; ++i)
            if (w[i]) atomicAdd(&s_stats[2 + i], w[i]);
    }
    __syncthreads();
    if (threadIdx.x >= 2 && threadIdx.x < 5 && s_stats[threadIdx.x]) atomicAdd(&g_stats[threadIdx.x], s_stats[threadIdx.x]);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&g_stats[0], launch_steps);
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch: consecutive step kernels of a stream (or of a captured graph) are
// launched with cudaLaunchAttributeProgrammaticStreamSerialization, so that kernel N+1 becomes resident
// while kernel N drains and overlaps its launch latency and table loads with N's tail.  Everything that
// N may still be writing (state, t, step counter, statistics) is touched only after pdl_wait(), which
// returns once all preceding kernels of the stream have completed and flushed; only the immutable
// tables are read before it.  Both instructions are no-ops in a launch without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Per-device one-time kernel setup.  cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the
// CURRENT device only; a process driving several GPUs (one handle per device) must repeat it on each.
// Returns the slot of the current device in a per-kernel table (devices beyond the table share the last
// slot and are set up on every call).
constexpr int kMaxDevices = 64;
inline int current_device_slot()
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
    return dev < kMaxDevices ? dev : kMaxDevices - 1;
}

inline bool pdl_enabled()
{
    static const bool on = [] { const char *v = std::getenv("GC_B200_PDL"); return !(v && v[0] == '0'); }();
    return on;
}

template <typename... KArgs, typename... Args>
cudaError_t launch_step_kernel(void (*kernel)(KArgs...), int grid, int threads, size_t smem, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(grid));
    cfg.blockDim = dim3(static_cast<unsigned>(threads));
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---------------------------------------------------------------------------------------------
// Launch geometry: GC_OVERSUB waves of resident blocks (SM count x occupancy), grid-stride inside.
#ifndef GC_OVERSUB
#define GC_OVERSUB 1
#endif
template <auto Kernel, int THREADS = kThreads>
int grid_for(int64_t n_envs, int n_sm)
{
    const auto kernel = Kernel;
    static int per_sm = 0;               // one static per kernel instantiation: query the occupancy once
    if (per_sm == 0 &&
        (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, THREADS, 0) != cudaSuccess || per_sm < 1))
        per_sm = 1;
    const int64_t need = (n_envs + THREADS * kEPT - 1) / (THREADS * kEPT);
    const int64_t cap = static_cast<int64_t>(n_sm) * per_sm * GC_OVERSUB;
    return static_cast<int>(need < cap ? (need < 1 ? 1 : need) : cap);
}

}  // namespace
