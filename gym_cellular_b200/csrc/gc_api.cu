// C ABI of libgymcellular_b200.so (include/gym_cellular_b200.h).  No C++ exceptions cross the
// boundary: every entry point returns a gc_status and records a thread-local message.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <memory>
#include <new>

#include <nvtx3/nvToolsExt.h>

#include "gc_internal.h"

namespace {

thread_local char g_err[512] = "";

// NVTX range around every entry point (a profiler timeline shows the host side of each call; without a
// tool attached a push/pop is a null function-pointer test)
struct NvtxRange {
    explicit NvtxRange(const char *name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
#define GC_NVTX(name) NvtxRange nvtx_range_(name)

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define GC_CUDA(call)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail(GC_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),   \
                        __FILE__, __LINE__);                                                  \
    } while (0)

constexpr int kHostStreams = 3;
constexpr int kManyGraphs = 4;
constexpr int kManyGraphSteps = 16;   // kernels per captured graph: whole passes over the slot list, at least this many steps

// Entry points run on the handle's device but leave the caller's current device untouched (a torch
// process may be driving several GPUs).
class DeviceGuard {
public:
    explicit DeviceGuard(int device) : prev_(-1), err_(cudaSuccess)
    {
        err_ = cudaGetDevice(&prev_);
        if (err_ == cudaSuccess && prev_ != device) err_ = cudaSetDevice(device); else prev_ = -1;
    }
    ~DeviceGuard() { if (prev_ >= 0) cudaSetDevice(prev_); }
    cudaError_t error() const { return err_; }
private:
    int prev_;
    cudaError_t err_;
};

#define GC_ON_DEVICE(dev)                                                                      \
    DeviceGuard guard_(dev);                                                                   \
    if (guard_.error() != cudaSuccess)                                                         \
        return fail(GC_ERR_CUDA, "cannot switch to device %d: %s", (dev), cudaGetErrorString(guard_.error()))

// x * 2^-32 < p  <=>  x < ceil(p * 2^32)   (p * 2^32 is exact in double: a power-of-two scaling)
unsigned long long threshold_of(double p)
{
    if (!(p > 0.0)) return 0ull;
    if (p >= 1.0) return 1ull << 32;
    return static_cast<unsigned long long>(std::ceil(p * 4294967296.0));
}

}  // namespace

struct gc_env {
    gc_config cfg;
    CellTables tab;
    GridParams grid;
    bool tables_set;
    int n_sm;
    int64_t global_step;
    int64_t launches;
    unsigned long long *d_status;   // [0] status bits; the same allocation holds the step words:
    uint32_t *d_step;               // device-resident global step (RNG counter of non-episodic envs)
    uint32_t *d_done;               // block-arrival counter of the step kernels
    uint2 *d_pair_lut;            // fast-path table (GC_PAIR_LUT_ENTRIES), device memory owned by the handle
    uint2 *d_packed_lut;          // the same rules in the packed layout's index order (gc_cell_packed.cu)
    uint2 *d_pair8_lut;           // 5..8 levels (gc_cell_pair8.cu): GC_PAIR8_ENTRIES entries
    bool pair8_ok;
    int8_t *final_state;          // gc_set_final_obs: optional extra output of every int8-layout step
    bool fast_ok;
    StepIO bound[GC_MAX_BINDINGS];  // gc_bind_step slots
    PackedIO bound_packed[GC_MAX_BINDINGS];   // gc_bind_step_packed slots
    int bound_set[GC_MAX_BINDINGS]; // 0 empty, 1 int8 layout, 2 packed layout
    cudaStream_t hstream[kHostStreams];
    cudaEvent_t hevent[kHostStreams];
    bool host_ready;
    // gc_step_many: instantiated CUDA graphs of one pass over a slot list (launch-bound batch sizes)
    struct ManyGraph { int32_t slots[GC_MAX_BINDINGS]; int32_t n_slots, n_steps; cudaGraphExec_t exec; } many[kManyGraphs];
    int n_many;
};

namespace {

int check_env(const gc_env *env)
{
    if (!env) return fail(GC_ERR_INVALID, "env is NULL");
    return GC_OK;
}

int check_range(const gc_env *env, int64_t begin, int64_t count)
{
    const int64_t n = env->cfg.n_envs;
    if (begin < 0 || count < 0 || begin + count > n)
        return fail(GC_ERR_INVALID, "env range [%lld, %lld) outside [0, %lld)", (long long)begin,
                    (long long)(begin + count), (long long)n);
    if (begin % 16 != 0)
        return fail(GC_ERR_INVALID, "env_begin must be a multiple of 16");
    if ((begin + count) % 16 != 0 && begin + count != n)
        return fail(GC_ERR_INVALID, "env range must end on a multiple of 16 or at n_envs");
    return GC_OK;
}

StepIO make_io(const gc_env *env, int64_t begin, int64_t count, const int8_t *actions, int8_t *state,
               int32_t *t, float *reward, uint32_t *index, uint8_t *terminated, uint8_t *truncated,
               uint8_t *unsafe, uint8_t *count_out, int8_t *se_row, const double *replay, int64_t *stats)
{
    StepIO io;
    io.actions = actions; io.state = state; io.t = t; io.reward = reward; io.index = index;
    io.terminated = terminated; io.truncated = truncated; io.unsafe = unsafe; io.count = count_out;
    io.se_row = se_row; io.replay = replay;
    io.final_state = env->final_state;
    io.stats = reinterpret_cast<unsigned long long *>(stats);
    io.status = env->d_status;
    io.begin = begin; io.end = begin + count; io.ld = env->cfg.ld;
    io.env_id_offset = env->cfg.env_id_offset;
    io.seed_lo = static_cast<uint32_t>(env->cfg.seed);
    io.seed_hi = static_cast<uint32_t>(env->cfg.seed >> 32);
    for (int r = 0; r < 10; ++r) {
        io.round_key[2 * r] = io.seed_lo + static_cast<uint32_t>(r) * 0x9E3779B9u;
        io.round_key[2 * r + 1] = io.seed_hi + static_cast<uint32_t>(r) * 0xBB67AE85u;
    }
    io.rng_counter = static_cast<uint32_t>(env->global_step);
    // The global step (RNG counter of the non-episodic kinds) is read from DEVICE memory by every launch, so
    // CUDA-graph replays, pre-bound launches and host-path chunks all see the same truth.  A launch over the
    // whole shard also advances it (done_ctr: last block to finish); a chunk of a chunked pass only reads it
    // and the caller ticks it once after the last chunk (tick_global_step).
    io.step_ctr = env->d_step;
    io.done_ctr = nullptr;
    io.episodic = (env->cfg.flags & GC_F_RNG_EPISODIC) ? 1 : 0;
    io.max_episode_steps = env->cfg.max_episode_steps;
    return io;
}

PackedIO make_packed_io(const gc_env *env, int64_t begin, int64_t count, const uint32_t *actions, uint32_t *state,
                        int32_t *t, float *reward, uint32_t *index, uint8_t *flags, uint32_t *final_state,
                        uint32_t *se_row, int64_t *stats)
{
    PackedIO io;
    io.actions = actions; io.state = state; io.t = t; io.reward = reward; io.index = index; io.flags = flags;
    io.final_state = final_state; io.se_row = se_row;
    io.stats = reinterpret_cast<unsigned long long *>(stats);
    io.status = env->d_status;
    io.begin = begin; io.end = begin + count; io.ld = env->cfg.ld;
    io.env_id_offset = env->cfg.env_id_offset;
    const uint32_t lo = static_cast<uint32_t>(env->cfg.seed), hi = static_cast<uint32_t>(env->cfg.seed >> 32);
    for (int r = 0; r < 10; ++r) {
        io.round_key[2 * r] = lo + static_cast<uint32_t>(r) * 0x9E3779B9u;
        io.round_key[2 * r + 1] = hi + static_cast<uint32_t>(r) * 0xBB67AE85u;
    }
    io.rng_counter = static_cast<uint32_t>(env->global_step);
    io.step_ctr = env->d_step;
    io.done_ctr = nullptr;
    io.episodic = (env->cfg.flags & GC_F_RNG_EPISODIC) ? 1 : 0;
    io.max_episode_steps = env->cfg.max_episode_steps;
    return io;
}

int check_packed(const gc_env *env)
{
    if (env->cfg.kind != GC_KIND_CELLULAR || !env->fast_ok)
        return fail(GC_ERR_INVALID, "the packed layout covers the cellular family with n_states, n_actions <= 4 "
                                    "(and equal side-effect tables for the cells j >= 2)");
    return GC_OK;
}

int launch_packed(gc_env *env, const PackedIO &io, cudaStream_t st)
{
    if (io.end <= io.begin) return GC_OK;
    const bool draws = (env->cfg.flags & GC_F_NOISE) && env->tab.noise_thr_nz;
    cudaError_t e = gc_launch_cell_packed_step(env->tab, io, env->d_packed_lut, draws, env->n_sm, st);
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "packed step kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    return GC_OK;
}

// cached gc_step_many graphs hold the pointer sets of the bindings they were captured from
void drop_many_graphs(gc_env *env)
{
    for (int i = 0; i < env->n_many; ++i)
        if (env->many[i].exec) cudaGraphExecDestroy(env->many[i].exec);
    env->n_many = 0;
}

// A host-path call that fails after it queued copies must not return while they still write the caller's buffers.
struct HostDrain {
    gc_env *env;
    bool done = false;
    ~HostDrain()
    {
        if (done) return;
        for (int i = 0; i < kHostStreams; ++i) cudaStreamSynchronize(env->hstream[i]);
        cudaGetLastError();
    }
};

int host_streams(gc_env *env)
{
    if (!env->host_ready) {
        for (int i = 0; i < kHostStreams; ++i) {
            GC_CUDA(cudaStreamCreateWithFlags(&env->hstream[i], cudaStreamNonBlocking));
            GC_CUDA(cudaEventCreateWithFlags(&env->hevent[i], cudaEventDisableTiming));
        }
        env->host_ready = true;
    }
    return GC_OK;
}

// advances the device-resident global step after the last chunk of a chunked pass (stream-ordered)
int tick_global_step(gc_env *env, cudaStream_t st)
{
    cudaError_t e = gc_launch_tick(env->d_step, 1u, st);
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "step-counter kernel launch failed: %s", cudaGetErrorString(e));
    env->global_step += 1;
    return GC_OK;
}

int launch_step(gc_env *env, const StepIO &io, cudaStream_t st)
{
    if (io.end <= io.begin) return GC_OK;
    cudaError_t e;
    if (env->cfg.kind == GC_KIND_CELLULAR) {
        // noise with probability 0 never fires: the deterministic kernels then do the same job
        const bool draws = (env->cfg.flags & GC_F_NOISE) && env->tab.noise_thr_nz;
        const int mode = io.replay ? GC_RNG_REPLAY : (draws ? GC_RNG_PHILOX : GC_RNG_NONE);
        if (env->fast_ok)
            e = gc_launch_cell_pair_step(env->tab, io, env->d_pair_lut, mode, env->n_sm, st);
        else if (env->pair8_ok && mode != GC_RNG_REPLAY)
            e = gc_launch_cell_pair8_step(env->tab, io, env->d_pair8_lut, mode, env->n_sm, st);
        else
            e = gc_launch_cell_step(env->tab, io, mode, env->n_sm, st);
    } else {
        e = gc_launch_grid_step(env->grid, io, io.replay ? GC_RNG_REPLAY : GC_RNG_PHILOX, env->n_sm, st);
    }
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "step kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    return GC_OK;
}

}  // namespace

extern "C" {

int gc_abi_version(void) { return GC_ABI_VERSION; }

const char *gc_last_error(void) { return g_err; }

int gc_create(const gc_config *cfg, gc_env **out)
{
    GC_NVTX("gc_create");
    if (!cfg || !out) return fail(GC_ERR_INVALID, "cfg/out is NULL");
    if (cfg->struct_size != sizeof(gc_config))
        return fail(GC_ERR_INVALID, "gc_config.struct_size %u != %zu (ABI mismatch)", cfg->struct_size, sizeof(gc_config));
    if (cfg->n_envs < 1) return fail(GC_ERR_INVALID, "n_envs must be >= 1");
    if (cfg->ld < cfg->n_envs || cfg->ld % 16 != 0)
        return fail(GC_ERR_INVALID, "ld must be a multiple of 16 and >= n_envs");
    if (cfg->max_episode_steps < 0) return fail(GC_ERR_INVALID, "max_episode_steps must be >= 0");
    // the kernels index their arrays with 32-bit element offsets (one IMAD.WIDE per address)
    if (cfg->n_cells >= 1 && cfg->ld > (int64_t(1) << 31) / cfg->n_cells)
        return fail(GC_ERR_INVALID, "n_cells * ld must not exceed 2^31 (%d cells: at most %lld envs per handle)", cfg->n_cells,
                    (long long)((int64_t(1) << 31) / cfg->n_cells));
    if (cfg->env_id_offset < 0 || cfg->env_id_offset % 4 != 0)
        return fail(GC_ERR_INVALID, "env_id_offset must be a non-negative multiple of 4");
    // probabilities, not thresholds: NaN or a value outside [0, 1] is a caller's mistake, never "never" or "always"
    if (!(cfg->noise_prob >= 0.0 && cfg->noise_prob <= 1.0))
        return fail(GC_ERR_INVALID, "noise_prob must lie in [0, 1] (got %g)", cfg->noise_prob);
    if (!(cfg->dispersal_prob >= 0.0 && cfg->dispersal_prob <= 1.0))
        return fail(GC_ERR_INVALID, "dispersal_prob must lie in [0, 1] (got %g)", cfg->dispersal_prob);
    if (cfg->kind == GC_KIND_CELLULAR) {
        if (cfg->n_cells < 1 || cfg->n_cells > GC_MAX_CELLS)
            return fail(GC_ERR_INVALID, "n_cells must be in 1..%d", GC_MAX_CELLS);
        if (cfg->n_states < 2 || cfg->n_states > GC_MAX_LEVELS || cfg->n_actions < 1 || cfg->n_actions > GC_MAX_LEVELS)
            return fail(GC_ERR_INVALID, "n_states must be in 2..%d and n_actions in 1..%d", GC_MAX_LEVELS, GC_MAX_LEVELS);
        if (cfg->n_cells * std::log2((double)cfg->n_states) > 32.0 + 1e-9)
            return fail(GC_ERR_INVALID, "n_states^n_cells does not fit the 32-bit tabular index");
    } else if (cfg->kind == GC_KIND_GRIDWORLD) {
        if (cfg->n_cells != 2 || cfg->n_states != 20 || cfg->n_actions != 5)
            return fail(GC_ERR_INVALID, "grid world is 2 jurisdictions x 20 codes x 5 actions");
    } else {
        return fail(GC_ERR_INVALID, "unknown kind %d", cfg->kind);
    }
    int n_dev = 0;
    GC_CUDA(cudaGetDeviceCount(&n_dev));
    if (cfg->device < 0 || cfg->device >= n_dev)
        return fail(GC_ERR_INVALID, "device %d not in [0, %d)", cfg->device, n_dev);
    GC_ON_DEVICE(cfg->device);
    int n_sm = 0;
    GC_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, cfg->device));
    gc_env *env = new (std::nothrow) gc_env();
    if (!env) return fail(GC_ERR_INVALID, "out of host memory");
    std::memset(env, 0, sizeof(*env));
    env->cfg = *cfg;
    env->n_sm = n_sm;
    env->grid.dispersal_thr = threshold_of(cfg->dispersal_prob);
    env->grid.dispersal_thr_nz = env->grid.dispersal_thr != 0ull;
    env->grid.dispersal_thr_m1 = env->grid.dispersal_thr_nz ? static_cast<uint32_t>(env->grid.dispersal_thr - 1ull) : 0u;
    env->grid.dispersal_prob = cfg->dispersal_prob;
    env->tables_set = (cfg->kind == GC_KIND_GRIDWORLD);
    cudaError_t e = cudaMalloc(&env->d_status, 2 * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMemset(env->d_status, 0, 2 * sizeof(unsigned long long));
    if (e == cudaSuccess) {
        env->d_step = reinterpret_cast<uint32_t *>(env->d_status + 1);
        env->d_done = env->d_step + 1;
    }
    if (e == cudaSuccess && cfg->kind == GC_KIND_GRIDWORLD) {
        std::unique_ptr<uint32_t[]> lut(new (std::nothrow) uint32_t[GC_GRID_LUT_ENTRIES]);
        uint32_t *d_lut = nullptr;
        if (!lut) e = cudaErrorMemoryAllocation;
        if (e == cudaSuccess) {
            gc_build_grid_lut(lut.get());
            e = cudaMalloc(&d_lut, GC_GRID_LUT_ALLOC * sizeof(uint32_t));
        }
        if (e == cudaSuccess) e = cudaMemset(d_lut, 0, GC_GRID_LUT_ALLOC * sizeof(uint32_t));
        if (e == cudaSuccess) e = cudaMemcpy(d_lut, lut.get(), GC_GRID_LUT_ENTRIES * sizeof(uint32_t), cudaMemcpyHostToDevice);
        env->grid.lut = d_lut;
    }
    if (e != cudaSuccess) {
        if (env->d_status) cudaFree(env->d_status);
        if (env->grid.lut) cudaFree(const_cast<uint32_t *>(env->grid.lut));
        delete env;
        return fail(GC_ERR_CUDA, "device table allocation failed: %s", cudaGetErrorString(e));
    }
    *out = env;
    return GC_OK;
}

int gc_destroy(gc_env *env)
{
    if (!env) return GC_OK;
    DeviceGuard guard_(env->cfg.device);
    drop_many_graphs(env);
    if (env->host_ready)
        for (int i = 0; i < kHostStreams; ++i) {
            cudaStreamDestroy(env->hstream[i]);
            cudaEventDestroy(env->hevent[i]);
        }
    if (env->d_status) cudaFree(env->d_status);
    if (env->d_pair_lut) cudaFree(env->d_pair_lut);
    if (env->d_packed_lut) cudaFree(env->d_packed_lut);
    if (env->d_pair8_lut) cudaFree(env->d_pair8_lut);
    if (env->grid.lut) cudaFree(const_cast<uint32_t *>(env->grid.lut));
    delete env;
    return GC_OK;
}

int gc_set_tables(gc_env *env, const gc_cell_tables *t)
{
    GC_NVTX("gc_set_tables");
    if (int rc = check_env(env)) return rc;
    if (env->cfg.kind != GC_KIND_CELLULAR) return fail(GC_ERR_INVALID, "tables apply to the cellular family only");
    if (!t || !t->move || !t->reward || !t->side_effects || !t->counted || !t->initial_state)
        return fail(GC_ERR_INVALID, "move, reward, side_effects, counted and initial_state are required");
    const int C = env->cfg.n_cells, S = env->cfg.n_states, A = env->cfg.n_actions;
    const bool noise = (env->cfg.flags & GC_F_NOISE) != 0;
    if (noise && (!t->noisy || !t->draws)) return fail(GC_ERR_INVALID, "GC_F_NOISE needs the noisy and draws tables");
    // built aside and committed at the end: a rejected call leaves the handle's previous tables in force
    CellTables tab;
    std::memset(&tab, 0, sizeof(tab));
    for (int s = 0; s < S; ++s)
        for (int a = 0; a < A; ++a) {
            const int mv = t->move[s * A + a];
            const int nz = t->noisy ? t->noisy[s * A + a] : mv;
            const int dr = (noise && t->draws) ? (t->draws[s * A + a] != 0) : 0;
            if (mv < 0 || mv >= S || nz < 0 || nz >= S)
                return fail(GC_ERR_INVALID, "move/noisy[%d][%d] outside [0, %d)", s, a, S);
            tab.sa[s * GC_LVL_PAD + a] = (uint32_t)mv | ((uint32_t)nz << 4) | ((uint32_t)dr << 8);
            if (!std::isfinite(t->reward[s * A + a]) || (t->reward_noisy && !std::isfinite(t->reward_noisy[s * A + a])))
                return fail(GC_ERR_INVALID, "reward/reward_noisy[%d][%d] is not finite", s, a);
            tab.reward[s * GC_LVL_PAD + a] = t->reward[s * A + a];
            tab.reward_noisy[s * GC_LVL_PAD + a] = (t->reward_noisy ? t->reward_noisy : t->reward)[s * A + a];
        }
    {
        // The reward statistic adds round(reward * 2^24) as a 32-bit integer per env-step, so every step's reward
        // must stay below 128 in magnitude.  A step's cell sum lies in [C lo, C hi] for the smallest and largest
        // table entry, and the float32 sum may pass that by half an ulp (< 2^-18 below 128) per addition.
        double lo = t->reward[0], hi = t->reward[0];
        for (int i = 0; i < S * A; ++i)
            for (const float *r : {t->reward, t->reward_noisy})
                if (r) { lo = std::min(lo, (double)r[i]); hi = std::max(hi, (double)r[i]); }
        const double slack = C * std::ldexp(1.0, -18);
        double bound = std::max(std::fabs(C * lo), std::fabs(C * hi)) + slack;
        if (env->cfg.flags & GC_F_REWARD_LOG2)
            bound = 1.0 + C * lo - slack > 0.0
                        ? std::max(std::fabs(std::log2(1.0 + C * lo - slack)), std::fabs(std::log2(1.0 + C * hi + slack)))
                        : HUGE_VAL;
        if (!(bound < 128.0))
            return fail(GC_ERR_INVALID, "rewards reach %g in magnitude per step (n_cells x the largest |reward|%s): the "
                        "reward statistic holds |reward| < 128", bound,
                        (env->cfg.flags & GC_F_REWARD_LOG2) ? ", under log2(1 + .)" : "");
    }
    for (int j = 0; j < C; ++j)
        for (int s0 = 0; s0 < S; ++s0)
            for (int sp = 0; sp < S; ++sp) {
                const int code = t->side_effects[(j * S + s0) * S + sp];
                if (code < 0 || code > 2) return fail(GC_ERR_INVALID, "side_effects code %d not in {0,1,2}", code);
                tab.se[j][s0 * GC_LVL_PAD + sp] = (uint8_t)code;
            }
    // place values of the tabular index: uniform radix n_states, or the per-cell level counts of a ragged
    // state space (generalized_space_transformations.py:1-12 takes one space per cell)
    bool ragged = false;
    if (t->radix) {
        double bits = 0.0;
        for (int c = 0; c < C; ++c) {
            if (t->radix[c] < 1 || t->radix[c] > S) return fail(GC_ERR_INVALID, "radix[%d] = %d not in 1..n_states", c, t->radix[c]);
            bits += std::log2((double)t->radix[c]);
            ragged = ragged || t->radix[c] != S;
        }
        if (bits > 32.0 + 1e-9) return fail(GC_ERR_INVALID, "the ragged state space does not fit the 32-bit tabular index");
    }
    uint32_t place = 1, init_index = 0;
    for (int c = 0; c < C; ++c) {
        const int lv = t->initial_state[c];
        const int radix_c = t->radix ? t->radix[c] : S;
        if (lv < 0 || lv >= radix_c) return fail(GC_ERR_INVALID, "initial_state[%d] outside [0, %d)", c, radix_c);
        tab.place[c] = place;
        tab.init[c] = (int8_t)lv;
        init_index += (uint32_t)lv * place;
        place *= (uint32_t)radix_c;
    }
    tab.init_index = init_index;
    for (int s = 0; s < S; ++s) if (t->counted[s]) tab.counted_mask |= 1u << s;
    tab.n_cells = C; tab.n_states = S; tab.n_actions = A;
    tab.reward_log2 = (env->cfg.flags & GC_F_REWARD_LOG2) ? 1 : 0;
    tab.noise_thr = threshold_of(env->cfg.noise_prob);
    tab.noise_prob = env->cfg.noise_prob;

    tab.noise_thr_nz = tab.noise_thr != 0ull;
    tab.noise_thr_m1 = tab.noise_thr_nz ? static_cast<uint32_t>(tab.noise_thr - 1ull) : 0u;
    {
        // threshold = k16 * 2^16 + r16; a threshold of 2^32 (p >= 1) is k16 = 65535, r16 = 2^16: a half below
        // 65535 fires, 65535 ties and the tie always fires
        uint32_t k16 = static_cast<uint32_t>(tab.noise_thr >> 16), r16 = static_cast<uint32_t>(tab.noise_thr & 0xFFFFull);
        if (k16 > 65535u) { k16 = 65535u; r16 = 1u << 16; }
        tab.noise_kk15 = (k16 & 0x7FFFu) * 0x00010001u;
        tab.noise_kmask = (k16 & 0x8000u) ? 0xFFFFFFFFu : 0u;
        tab.noise_kk = k16 * 0x00010001u;
        tab.noise_r16 = r16;
    }

    // ---- fast path: pair table (gc_cell_fast.cu) -------------------------------------------------
    // (a ragged index needs per-cell place values: generic kernel)
    bool fast_ok = S <= 4 && A <= 4 && !ragged && !(env->cfg.flags & GC_F_GENERIC_KERNEL);
    for (int j = 3; j < C && fast_ok; ++j)
        if (std::memcmp(t->side_effects + (size_t)j * S * S, t->side_effects + (size_t)2 * S * S, (size_t)S * S) != 0)
            fast_ok = false;
    // the device copies below are synchronous (pageable source), i.e. ordered after every step launched before
    // this call on any blocking stream; kernels still in flight on non-blocking streams must be waited for by
    // the caller (include/gym_cellular_b200.h)
    if (fast_ok) {
        uint2 lut[GC_PAIR_LUT_ENTRIES];                       // 8.4 KB, on the stack: handles may be set up concurrently
        gc_build_pair_lut(t, C, S, A, noise, lut, &tab.unsafe_rows);
        uint32_t p4 = 1;
        for (int i = 0; i < 4; ++i) { tab.place4[i] = p4; p4 *= (uint32_t)S; }
        GC_ON_DEVICE(env->cfg.device);
        if (!env->d_pair_lut) GC_CUDA(cudaMalloc(&env->d_pair_lut, sizeof(lut)));
        GC_CUDA(cudaMemcpy(env->d_pair_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
        gc_build_packed_lut(t, C, S, A, noise, lut);
        tab.init_packed = 0;
        for (int c = 0; c < C; ++c) tab.init_packed |= (uint32_t)(tab.init[c] & 3) << (2 * c);
        if (!env->d_packed_lut) GC_CUDA(cudaMalloc(&env->d_packed_lut, sizeof(lut)));
        GC_CUDA(cudaMemcpy(env->d_packed_lut, lut, sizeof(lut), cudaMemcpyHostToDevice));
    }
    // ---- 5..8 levels: 3-bit pair table, single-cell table with the fire bit (gc_cell_pair8.cu) -----------
    bool pair8_ok = !fast_ok && S <= 8 && A <= 8 && !ragged && !(env->cfg.flags & GC_F_GENERIC_KERNEL);
    for (int j = 3; j < C && pair8_ok; ++j)
        if (std::memcmp(t->side_effects + (size_t)j * S * S, t->side_effects + (size_t)2 * S * S, (size_t)S * S) != 0)
            pair8_ok = false;
    if (pair8_ok) {
        std::unique_ptr<uint2[]> lut8(new (std::nothrow) uint2[GC_PAIR8_ENTRIES]);
        if (!lut8) return fail(GC_ERR_INVALID, "out of host memory");
        gc_build_pair8_lut(t, C, S, A, noise, lut8.get(), &tab.unsafe_rows8, &tab.unsafe01_rows8);
        GC_ON_DEVICE(env->cfg.device);
        if (!env->d_pair8_lut) GC_CUDA(cudaMalloc(&env->d_pair8_lut, GC_PAIR8_ENTRIES * sizeof(uint2)));
        GC_CUDA(cudaMemcpy(env->d_pair8_lut, lut8.get(), GC_PAIR8_ENTRIES * sizeof(uint2), cudaMemcpyHostToDevice));
    }
    drop_many_graphs(env);                     // captured kernel nodes carry the tables by value
    env->tab = tab;
    env->fast_ok = fast_ok;
    env->pair8_ok = pair8_ok;
    env->tables_set = true;
    return GC_OK;
}

int gc_set_final_obs(gc_env *env, int8_t *final_state)
{
    if (int rc = check_env(env)) return rc;
    env->final_state = final_state;
    drop_many_graphs(env);
    for (int i = 0; i < GC_MAX_BINDINGS; ++i)
        if (env->bound_set[i] == 1) env->bound[i].final_state = final_state;
    return GC_OK;
}

int gc_set_global_step(gc_env *env, int64_t step)
{
    if (int rc = check_env(env)) return rc;
    env->global_step = step;
    const uint32_t v = static_cast<uint32_t>(step);
    GC_ON_DEVICE(env->cfg.device);
    GC_CUDA(cudaMemcpy(env->d_step, &v, sizeof(v), cudaMemcpyHostToDevice));   // synchronous: rare, control path
    // a copy from pageable memory may return before its DMA has landed: wait for it, so that a kernel queued next on
    // a non-blocking stream reads the new value
    GC_CUDA(cudaStreamSynchronize(cudaStreamLegacy));
    return GC_OK;
}

// Host mirror of the step counter.  Replaying a captured CUDA graph advances only the device word;
// gc_sync_global_step reads it back.
int64_t gc_get_global_step(const gc_env *env) { return env ? env->global_step : -1; }

int gc_sync_global_step(gc_env *env, void *stream)
{
    if (int rc = check_env(env)) return rc;
    GC_ON_DEVICE(env->cfg.device);
    uint32_t v = 0;
    GC_CUDA(cudaMemcpyAsync(&v, env->d_step, sizeof(v), cudaMemcpyDeviceToHost, static_cast<cudaStream_t>(stream)));
    GC_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    env->global_step = (env->global_step & ~0xFFFFFFFFll) | v;
    return GC_OK;
}

int64_t gc_launch_count(const gc_env *env) { return env ? env->launches : -1; }

int gc_reset(gc_env *env, const uint8_t *mask, int8_t *state, int32_t *t, uint32_t *index, void *stream)
{
    GC_NVTX("gc_reset");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (!state || !t) return fail(GC_ERR_INVALID, "state/t is NULL");
    GC_ON_DEVICE(env->cfg.device);
    int8_t init[GC_MAX_CELLS] = {0};
    uint32_t init_index;
    if (env->cfg.kind == GC_KIND_GRIDWORLD) {
        init[0] = 15; init[1] = 18; init_index = 15 + 20 * 18;     // grid_world.py:238-259
    } else {
        std::memcpy(init, env->tab.init, sizeof(init));
        init_index = env->tab.init_index;
    }
    // whole words are written, so cover the padded length
    const int64_t n_pad = (env->cfg.n_envs + 3) / 4 * 4;
    cudaError_t e = gc_launch_reset(env->cfg.n_cells, init, init_index, mask, state, t, index, n_pad,
                                    env->cfg.ld, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "reset kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    return GC_OK;
}

int gc_step(gc_env *env, int64_t env_begin, int64_t env_count, const int8_t *actions, int8_t *state,
            int32_t *t, float *reward, uint32_t *index, uint8_t *terminated, uint8_t *truncated,
            uint8_t *unsafe, uint8_t *count, int8_t *se_row, const double *replay_u, int64_t *stats,
            void *stream)
{
    GC_NVTX("gc_step");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (!actions || !state || !t || !reward || !index || !terminated || !truncated || !unsafe || !count)
        return fail(GC_ERR_INVALID, "a required device pointer is NULL");
    if (int rc = check_range(env, env_begin, env_count)) return rc;
    GC_ON_DEVICE(env->cfg.device);
    StepIO io = make_io(env, env_begin, env_count, actions, state, t, reward, index, terminated,
                        truncated, unsafe, count, se_row, replay_u, stats);
    const bool full = env_begin == 0 && env_count == env->cfg.n_envs;
    if (full) io.done_ctr = env->d_done;     // whole shard in one launch: the kernel itself advances the step
    if (int rc = launch_step(env, io, static_cast<cudaStream_t>(stream))) return rc;
    if (full) {
        env->global_step += 1;
    } else if (env_begin + env_count == env->cfg.n_envs) {                 // last chunk of a chunked pass
        if (int rc = tick_global_step(env, static_cast<cudaStream_t>(stream))) return rc;
    }
    return GC_OK;
}

int gc_bind_step(gc_env *env, int32_t slot, const int8_t *actions, int8_t *state, int32_t *t, float *reward,
                 uint32_t *index, uint8_t *terminated, uint8_t *truncated, uint8_t *unsafe, uint8_t *count,
                 int8_t *se_row, int64_t *stats)
{
    if (int rc = check_env(env)) return rc;
    if (slot < 0 || slot >= GC_MAX_BINDINGS) return fail(GC_ERR_INVALID, "slot must be in [0, %d)", GC_MAX_BINDINGS);
    if (!actions || !state || !t || !reward || !index || !terminated || !truncated || !unsafe || !count)
        return fail(GC_ERR_INVALID, "a required device pointer is NULL");
    env->bound[slot] = make_io(env, 0, env->cfg.n_envs, actions, state, t, reward, index, terminated, truncated,
                               unsafe, count, se_row, nullptr, stats);
    env->bound[slot].done_ctr = env->d_done;
    env->bound_set[slot] = 1;
    drop_many_graphs(env);
    return GC_OK;
}

namespace {
int launch_bound(gc_env *env, int32_t slot, cudaStream_t st)
{
    if (slot < 0 || slot >= GC_MAX_BINDINGS || !env->bound_set[slot])
        return fail(GC_ERR_INVALID, "no binding in slot %d", slot);
    // a packed binding outlives the tables it was checked against: the packed LUT is rebuilt only for tables that
    // admit the layout, so the slot is refused while the current ones do not
    if (env->bound_set[slot] == 2)
        if (int rc = check_packed(env)) return rc;
    if (int rc = env->bound_set[slot] == 2 ? launch_packed(env, env->bound_packed[slot], st)
                                           : launch_step(env, env->bound[slot], st))
        return rc;
    env->global_step += 1;
    return GC_OK;
}
}  // namespace

int gc_step_bound(gc_env *env, int32_t slot, void *stream)
{
    if (!env) return fail(GC_ERR_INVALID, "gc_step_bound: env is NULL");
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    GC_ON_DEVICE(env->cfg.device);
    return launch_bound(env, slot, static_cast<cudaStream_t>(stream));
}

namespace {
// The instantiated graph of one pass over `slots` (one kernel node per bound step, chained by the programmatic
// dependency edges the launches carry), captured on a stream of the handle; NULL if it cannot be built.
const gc_env::ManyGraph *many_graph(gc_env *env, const int32_t *slots, int32_t n_slots)
{
    for (int i = 0; i < env->n_many; ++i)
        if (env->many[i].n_slots == n_slots && std::memcmp(env->many[i].slots, slots, n_slots * sizeof(int32_t)) == 0)
            return &env->many[i];
    if (n_slots > GC_MAX_BINDINGS || host_streams(env) != GC_OK) return nullptr;
    if (env->n_many == kManyGraphs) drop_many_graphs(env);
    // several passes per graph: the gap between two graph launches (~2-3 us on the device) is paid once per
    // kManyGraphSteps kernels instead of once per n_slots
    static const int graph_steps = [] {
        const char *v = std::getenv("GC_B200_STEP_MANY_GRAPH_STEPS");
        const int k = v ? std::atoi(v) : 0;
        return k > 0 ? k : kManyGraphSteps;
    }();
    const int32_t passes = (graph_steps + n_slots - 1) / n_slots;
    cudaStream_t cap = env->hstream[0];
    const int64_t launches = env->launches, step = env->global_step;      // capturing executes nothing
    if (cudaStreamBeginCapture(cap, cudaStreamCaptureModeRelaxed) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    int rc = GC_OK;
    for (int32_t p = 0; p < passes && rc == GC_OK; ++p)
        for (int32_t i = 0; i < n_slots && rc == GC_OK; ++i) rc = launch_bound(env, slots[i], cap);
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamEndCapture(cap, &graph);
    env->launches = launches; env->global_step = step;
    cudaGraphExec_t exec = nullptr;
    if (rc == GC_OK && e == cudaSuccess && graph) e = cudaGraphInstantiate(&exec, graph, 0);
    if (graph) cudaGraphDestroy(graph);
    if (rc != GC_OK || e != cudaSuccess || !exec) { cudaGetLastError(); return nullptr; }
    gc_env::ManyGraph &m = env->many[env->n_many++];
    std::memcpy(m.slots, slots, n_slots * sizeof(int32_t));
    m.n_slots = n_slots;
    m.n_steps = passes * n_slots;
    m.exec = exec;
    return &m;
}

// Graph replay pays off where the HOST call per kernel is the bound: short kernels.  Measured (same box, 2000
// steps): 65,536 envs 15.0 -> 20.7 G env-steps/s, 2^20 grid-world envs 147.5 -> 149.0 G; with 4M-env kernels
// (40 us each) the full dependency at every graph boundary costs more than the host calls saved (0.878 -> 0.857
// of the roofline), so larger shards keep plain launches.
constexpr int64_t kManyGraphMaxEnvs = 1 << 21;

bool many_graphs_enabled(const gc_env *env)
{
    static const bool on = [] { const char *v = std::getenv("GC_B200_STEP_MANY_GRAPH"); return !(v && v[0] == '0'); }();
    return on && env->cfg.n_envs <= kManyGraphMaxEnvs;
}

// Small shards whose bound slots differ ONLY in their action buffers (the usual ring of action buffers around one
// set of in-place state / output tensors) run all their steps in one launch: state in registers between the steps,
// every per-step output written as the separate launches write it (gc_cell_fast.cu: cell_pair_many_kernel).
// GC_B200_STEP_MANY_FUSED=0 switches it off (the cached graph of chained launches is used instead).
bool many_fusable(const gc_env *env, const int32_t *slots, int32_t n_slots)
{
    const char *v = std::getenv("GC_B200_STEP_MANY_FUSED");          // read at every call: benches measure both ways
    if ((v && v[0] == '0') || env->cfg.n_envs > kManyGraphMaxEnvs || env->final_state) return false;
    if (env->cfg.kind == GC_KIND_CELLULAR) {
        if (!env->fast_ok || env->cfg.n_cells > GC_MANY_MAX_CELLS) return false;
    }
    const int layout = env->bound_set[slots[0]];             // 1: int8 bindings, 2: packed bindings
    for (int32_t i = 0; i < n_slots; ++i)
        if (env->bound_set[slots[i]] != layout) return false;
    if (layout == 2) {
        if (env->cfg.kind != GC_KIND_CELLULAR) return false;
        const PackedIO &a = env->bound_packed[slots[0]];
        for (int32_t i = 1; i < n_slots; ++i) {
            const PackedIO &b = env->bound_packed[slots[i]];
            if (a.state != b.state || a.t != b.t || a.reward != b.reward || a.index != b.index || a.flags != b.flags ||
                a.se_row != b.se_row || a.stats != b.stats || a.final_state != b.final_state)
                return false;
        }
        return a.final_state == nullptr;
    }
    const StepIO &a = env->bound[slots[0]];
    for (int32_t i = 1; i < n_slots; ++i) {
        const StepIO &b = env->bound[slots[i]];
        if (a.state != b.state || a.t != b.t || a.reward != b.reward || a.index != b.index || a.terminated != b.terminated ||
            a.truncated != b.truncated || a.unsafe != b.unsafe || a.count != b.count || a.se_row != b.se_row ||
            a.stats != b.stats || a.final_state != b.final_state)
            return false;
    }
    return a.final_state == nullptr && a.replay == nullptr;
}

constexpr int32_t kManyFusedMaxSteps = 4096;       // steps per launch

int launch_many_fused(gc_env *env, const int32_t *slots, int32_t n_slots, int32_t first, int32_t n_steps, cudaStream_t st)
{
    const bool draws = (env->cfg.flags & GC_F_NOISE) && env->tab.noise_thr_nz;
    if (env->bound_set[slots[0]] == 2) {
        PackedManyIO pio;
        pio.io = env->bound_packed[slots[0]];
        for (int32_t i = 0; i < GC_MAX_BINDINGS; ++i)
            pio.tape[i] = i < n_slots ? env->bound_packed[slots[(first + i) % n_slots]].actions : nullptr;
        pio.n_tape = n_slots;
        pio.n_steps = n_steps;
        const cudaError_t e = gc_launch_cell_packed_many(env->tab, pio, env->d_packed_lut, draws, env->n_sm, st);
        if (e != cudaSuccess) return fail(GC_ERR_CUDA, "many-step kernel launch failed: %s", cudaGetErrorString(e));
        env->launches += 1;
        env->global_step += n_steps;
        return GC_OK;
    }
    ManyIO mio;
    mio.io = env->bound[slots[0]];
    for (int32_t i = 0; i < n_slots; ++i) mio.tape[i] = env->bound[slots[(first + i) % n_slots]].actions;
    for (int32_t i = n_slots; i < GC_MAX_BINDINGS; ++i) mio.tape[i] = nullptr;
    mio.n_tape = n_slots;
    mio.n_steps = n_steps;
    const cudaError_t e = env->cfg.kind == GC_KIND_CELLULAR
        ? gc_launch_cell_pair_many(env->tab, mio, env->d_pair_lut, draws ? GC_RNG_PHILOX : GC_RNG_NONE, env->n_sm, st)
        : gc_launch_grid_many(env->grid, mio, env->n_sm, st);
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "many-step kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    env->global_step += n_steps;
    return GC_OK;
}
}  // namespace

int gc_prepare_step_many(gc_env *env, const int32_t *slots, int32_t n_slots)
{
    if (!env || !slots || n_slots < 1) return fail(GC_ERR_INVALID, "gc_prepare_step_many: bad arguments");
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    for (int32_t i = 0; i < n_slots; ++i) {
        if (slots[i] < 0 || slots[i] >= GC_MAX_BINDINGS || !env->bound_set[slots[i]])
            return fail(GC_ERR_INVALID, "no binding in slot %d", slots[i]);
        if (env->bound_set[slots[i]] == 2)
            if (int rc = check_packed(env)) return rc;
    }
    GC_ON_DEVICE(env->cfg.device);
    if (n_slots <= GC_MAX_BINDINGS && many_fusable(env, slots, n_slots)) return GC_OK;     // one launch for all steps: no graph needed
    if (many_graphs_enabled(env) && n_slots >= 2) many_graph(env, slots, n_slots);   // best effort: plain launches otherwise
    return GC_OK;
}

int gc_step_many(gc_env *env, const int32_t *slots, int32_t n_slots, int32_t n_steps, void *stream)
{
    GC_NVTX("gc_step_many");
    if (!env || !slots || n_slots < 1 || n_steps < 0) return fail(GC_ERR_INVALID, "gc_step_many: bad arguments");
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    GC_ON_DEVICE(env->cfg.device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int32_t done = 0;
    // every slot is checked before the first step runs: a list the handle cannot step in full is refused whole
    for (int32_t i = 0; i < n_slots; ++i) {
        if (slots[i] < 0 || slots[i] >= GC_MAX_BINDINGS || !env->bound_set[slots[i]])
            return fail(GC_ERR_INVALID, "no binding in slot %d", slots[i]);
        if (env->bound_set[slots[i]] == 2)
            if (int rc = check_packed(env)) return rc;
    }
    // Small shards with one set of in-place buffers: all steps in one launch (many_fusable)
    if (n_steps >= 2 && n_slots <= GC_MAX_BINDINGS && many_fusable(env, slots, n_slots)) {
        for (; done < n_steps;) {
            const int32_t k = n_steps - done < kManyFusedMaxSteps ? n_steps - done : kManyFusedMaxSteps;
            if (int rc = launch_many_fused(env, slots, n_slots, done % n_slots, k, st)) return rc;
            done += k;
        }
        return GC_OK;
    }
    // Launch-bound batch sizes: whole passes over the slot list are replayed from a cached CUDA graph (one host
    // call per n_slots kernels instead of one per kernel; the RNG step counter lives in device memory, so every
    // replay draws fresh numbers).  Not while the caller's stream is itself being captured.
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    if (many_graphs_enabled(env) && n_slots >= 2 && n_steps >= 2 * n_slots &&
        cudaStreamIsCapturing(st, &capturing) == cudaSuccess && capturing == cudaStreamCaptureStatusNone) {
        if (const gc_env::ManyGraph *m = many_graph(env, slots, n_slots)) {
            for (; done + m->n_steps <= n_steps; done += m->n_steps) {
                GC_CUDA(cudaGraphLaunch(m->exec, st));
                env->launches += m->n_steps;
                env->global_step += m->n_steps;
            }
        }
    }
    for (int32_t i = done; i < n_steps; ++i)
        if (int rc = launch_bound(env, slots[i % n_slots], st)) return rc;
    return GC_OK;
}

int gc_step_host(gc_env *env, const int8_t *h_actions, int8_t *h_state, float *h_reward,
                 uint32_t *h_index, uint8_t *h_terminated, uint8_t *h_truncated, uint8_t *h_unsafe,
                 uint8_t *h_count, int8_t *h_se_row, int8_t *d_actions, int8_t *d_state, int32_t *d_t,
                 float *d_reward, uint32_t *d_index, uint8_t *d_terminated, uint8_t *d_truncated,
                 uint8_t *d_unsafe, uint8_t *d_count, int8_t *d_se_row, int64_t *d_stats,
                 int64_t chunk_envs)
{
    GC_NVTX("gc_step_host");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (!h_actions || !d_actions || !d_state || !d_t || !d_reward || !d_index || !d_terminated ||
        !d_truncated || !d_unsafe || !d_count)
        return fail(GC_ERR_INVALID, "a required pointer is NULL");
    if (h_se_row && !d_se_row) return fail(GC_ERR_INVALID, "h_se_row needs d_se_row");
    GC_ON_DEVICE(env->cfg.device);
    if (int rc = host_streams(env)) return rc;
    const int64_t n = env->cfg.n_envs, ld = env->cfg.ld;
    const int C = env->cfg.n_cells;
    if (chunk_envs <= 0) chunk_envs = 1 << 20;
    chunk_envs = (chunk_envs + 15) / 16 * 16;
    HostDrain drain{env};
    int k = 0;
    for (int64_t b = 0; b < n; b += chunk_envs, ++k) {
        const int64_t cnt = (b + chunk_envs < n) ? chunk_envs : (n - b);
        const int64_t cnt_pad = (cnt + 3) / 4 * 4;      // whole words; ld padding makes this safe
        cudaStream_t st = env->hstream[k % kHostStreams];
        GC_CUDA(cudaMemcpy2DAsync(d_actions + b, ld, h_actions + b, ld, cnt_pad, C, cudaMemcpyHostToDevice, st));
        const StepIO io = make_io(env, b, cnt, d_actions, d_state, d_t, d_reward, d_index, d_terminated,
                                  d_truncated, d_unsafe, d_count, d_se_row, nullptr, d_stats);
        if (int rc = launch_step(env, io, st)) return rc;
        if (h_state) GC_CUDA(cudaMemcpy2DAsync(h_state + b, ld, d_state + b, ld, cnt, C, cudaMemcpyDeviceToHost, st));
        if (h_reward) GC_CUDA(cudaMemcpyAsync(h_reward + b, d_reward + b, cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (h_index) GC_CUDA(cudaMemcpyAsync(h_index + b, d_index + b, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (h_terminated) GC_CUDA(cudaMemcpyAsync(h_terminated + b, d_terminated + b, cnt, cudaMemcpyDeviceToHost, st));
        if (h_truncated) GC_CUDA(cudaMemcpyAsync(h_truncated + b, d_truncated + b, cnt, cudaMemcpyDeviceToHost, st));
        if (h_unsafe) GC_CUDA(cudaMemcpyAsync(h_unsafe + b, d_unsafe + b, cnt, cudaMemcpyDeviceToHost, st));
        if (h_count) GC_CUDA(cudaMemcpyAsync(h_count + b, d_count + b, cnt, cudaMemcpyDeviceToHost, st));
        if (h_se_row)
            GC_CUDA(cudaMemcpy2DAsync(h_se_row + b, ld, d_se_row + b, ld, cnt, C, cudaMemcpyDeviceToHost, st));
    }
    for (int i = 0; i < kHostStreams && i < k; ++i) GC_CUDA(cudaStreamSynchronize(env->hstream[i]));
    // every chunk read the device-resident global step; advance it once, after all of them
    if (int rc = tick_global_step(env, env->hstream[0])) return rc;
    GC_CUDA(cudaStreamSynchronize(env->hstream[0]));
    drain.done = true;
    return GC_OK;
}

namespace {

// RolloutIO of a whole-shard gc_rollout / gc_collect launch (the record and epsilon fields stay zero)
RolloutIO make_rollout_io(const gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, int8_t *state,
                          int32_t *t, uint32_t *index, int64_t *stats)
{
    RolloutIO io;
    std::memset(&io, 0, sizeof(io));
    io.state = state; io.t = t; io.index = index; io.policy = policy;
    io.stats = reinterpret_cast<unsigned long long *>(stats);
    io.status = env->d_status;
    io.n = env->cfg.n_envs; io.ld = env->cfg.ld; io.env_id_offset = env->cfg.env_id_offset;
    const uint32_t lo = static_cast<uint32_t>(env->cfg.seed), hi = static_cast<uint32_t>(env->cfg.seed >> 32);
    for (int r = 0; r < 10; ++r) {
        io.round_key[2 * r] = lo + static_cast<uint32_t>(r) * 0x9E3779B9u;
        io.round_key[2 * r + 1] = hi + static_cast<uint32_t>(r) * 0xBB67AE85u;
    }
    io.step_ctr = env->d_step; io.done_ctr = env->d_done;
    io.episodic = (env->cfg.flags & GC_F_RNG_EPISODIC) ? 1 : 0;
    io.max_episode_steps = env->cfg.max_episode_steps;
    io.n_steps = n_steps; io.policy_kind = policy_kind;
    return io;
}

bool misaligned(const void *p) { return p && (reinterpret_cast<uintptr_t>(p) & 15u) != 0; }

// argument checks shared by gc_collect and gc_collect_counts, so that both reject the same calls (out = the record or
// the count struct)
int check_collect_args(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
                       const int8_t *state, const int32_t *t, const uint32_t *index, const void *out)
{
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (!state || !t || !index || !out) return fail(GC_ERR_INVALID, "a required pointer is NULL");
    if (n_steps < 1) return fail(GC_ERR_INVALID, "n_steps must be >= 1");
    if (policy_kind != GC_POLICY_RANDOM && policy_kind != GC_POLICY_TABLE) return fail(GC_ERR_INVALID, "unknown policy kind");
    if (policy_kind == GC_POLICY_TABLE && !policy) return fail(GC_ERR_INVALID, "GC_POLICY_TABLE needs a policy table");
    if (!(epsilon >= 0.0 && epsilon <= 1.0)) return fail(GC_ERR_INVALID, "epsilon must lie in [0, 1] (got %g)", epsilon);
    if (policy_kind == GC_POLICY_RANDOM && epsilon != 0.0)
        return fail(GC_ERR_INVALID, "epsilon applies to GC_POLICY_TABLE only (GC_POLICY_RANDOM needs epsilon 0)");
    return GC_OK;
}

// RolloutIO of a gc_collect / gc_collect_counts launch: the rollout's, plus the epsilon-greedy fields
RolloutIO make_collect_io(const gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
                          int8_t *state, int32_t *t, uint32_t *index, int64_t *stats)
{
    RolloutIO io = make_rollout_io(env, n_steps, policy_kind, policy, state, t, index, stats);
    unsigned long long joint = 1;
    for (int c = 0; c < env->cfg.n_cells; ++c) joint *= static_cast<unsigned long long>(env->cfg.n_actions);
    io.joint_actions = joint;
    const unsigned long long thr = threshold_of(epsilon);
    io.explore_thr_nz = thr != 0 ? 1u : 0u;
    io.explore_thr_m1 = static_cast<uint32_t>(thr - 1);
    return io;
}

}  // namespace

int gc_rollout(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, int8_t *state,
               int32_t *t, uint32_t *index, float *ret, int32_t *n_unsafe, int64_t *stats, void *stream)
{
    GC_NVTX("gc_rollout");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (!state || !t || !index || !ret || !n_unsafe) return fail(GC_ERR_INVALID, "a required device pointer is NULL");
    if (n_steps < 1) return fail(GC_ERR_INVALID, "n_steps must be >= 1");
    if (policy_kind != GC_POLICY_RANDOM && policy_kind != GC_POLICY_TABLE) return fail(GC_ERR_INVALID, "unknown policy kind");
    if (policy_kind == GC_POLICY_TABLE && !policy) return fail(GC_ERR_INVALID, "GC_POLICY_TABLE needs a policy table");
    if (env->cfg.kind == GC_KIND_CELLULAR && !env->fast_ok)
        return fail(GC_ERR_INVALID, "gc_rollout supports the cellular family with n_states, n_actions <= 4 only");
    GC_ON_DEVICE(env->cfg.device);
    RolloutIO io = make_rollout_io(env, n_steps, policy_kind, policy, state, t, index, stats);
    io.ret = ret; io.n_unsafe = n_unsafe;
    cudaError_t e;
    if (env->cfg.kind == GC_KIND_CELLULAR)
        e = gc_launch_cell_rollout(env->tab, io, env->d_pair_lut, (env->cfg.flags & GC_F_NOISE) != 0, env->n_sm,
                                   static_cast<cudaStream_t>(stream));
    else
        e = gc_launch_grid_rollout(env->grid, io, env->n_sm, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "rollout kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    env->global_step += n_steps;
    return GC_OK;
}


int gc_collect(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
               int8_t *state, int32_t *t, uint32_t *index, const gc_record *record, int64_t *stats, void *stream)
{
    GC_NVTX("gc_collect");
    if (int rc = check_collect_args(env, n_steps, policy_kind, policy, epsilon, state, t, index, record)) return rc;
    if (record->struct_size != sizeof(gc_record))
        return fail(GC_ERR_INVALID, "record->struct_size %u != sizeof(gc_record) %zu", record->struct_size, sizeof(gc_record));
    if (misaligned(record->obs) || misaligned(record->action) || misaligned(record->reward) || misaligned(record->flags) ||
        misaligned(record->next_obs))
        return fail(GC_ERR_INVALID, "record pointers must be 16-byte aligned");
    if (env->cfg.kind == GC_KIND_CELLULAR && !env->fast_ok)
        return fail(GC_ERR_INVALID, "gc_collect supports the cellular family with n_states, n_actions <= 4 only");
    GC_ON_DEVICE(env->cfg.device);
    RolloutIO io = make_collect_io(env, n_steps, policy_kind, policy, epsilon, state, t, index, stats);
    io.rec_obs = record->obs; io.rec_action = record->action; io.rec_reward = record->reward;
    io.rec_flags = record->flags; io.rec_next_obs = record->next_obs;
    cudaError_t e;
    if (env->cfg.kind == GC_KIND_CELLULAR)
        e = gc_launch_cell_collect(env->tab, io, env->d_pair_lut, (env->cfg.flags & GC_F_NOISE) != 0, env->n_sm,
                                   static_cast<cudaStream_t>(stream));
    else
        e = gc_launch_grid_collect(env->grid, io, env->n_sm, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "collect kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    env->global_step += n_steps;
    return GC_OK;
}

int gc_collect_counts(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
                      int8_t *state, int32_t *t, uint32_t *index, const gc_counts *counts, int64_t *stats, void *stream)
{
    GC_NVTX("gc_collect_counts");
    if (int rc = check_collect_args(env, n_steps, policy_kind, policy, epsilon, state, t, index, counts)) return rc;
    if (counts->struct_size != sizeof(gc_counts))
        return fail(GC_ERR_INVALID, "counts->struct_size %u != sizeof(gc_counts) %zu", counts->struct_size, sizeof(gc_counts));
    const void *ptrs[5] = {counts->visits, counts->next, counts->reward_q24, counts->unsafe, counts->cell_next};
    bool any = false;
    for (const void *p : ptrs) {
        if (p && (reinterpret_cast<uintptr_t>(p) & 7u) != 0) return fail(GC_ERR_INVALID, "count pointers must be 8-byte aligned");
        any = any || p;
    }
    if (!any) return fail(GC_ERR_INVALID, "every count pointer is NULL: nothing to count");
    const bool cellular = env->cfg.kind == GC_KIND_CELLULAR;
    if (!cellular && counts->cell_next) return fail(GC_ERR_INVALID, "cell_next counts the cellular family only, not grid world");
    if (cellular && !env->fast_ok)
        return fail(GC_ERR_INVALID, "gc_collect_counts supports the cellular family with n_states, n_actions <= 4 only");
    // joint table sizes, saturated above the 2^31-entry limit (indices are 32-bit in the kernels)
    constexpr unsigned long long kJointLimit = 1ull << 31;
    auto sat_mul = [](unsigned long long a, unsigned long long b) { return a > kJointLimit || b > kJointLimit || a * b > kJointLimit ? kJointLimit + 1 : a * b; };
    unsigned long long nS = 400, nA = 25;
    if (cellular) {
        nS = nA = 1;
        for (int c = 0; c < env->cfg.n_cells; ++c) {
            nS = sat_mul(nS, static_cast<unsigned long long>(env->cfg.n_states));
            nA = sat_mul(nA, static_cast<unsigned long long>(env->cfg.n_actions));
        }
    }
    const unsigned long long n_sa = sat_mul(nS, nA), n_sas = sat_mul(n_sa, nS);
    if ((counts->visits || counts->reward_q24 || counts->unsafe) && n_sa > kJointLimit)
        return fail(GC_ERR_INVALID, "the joint (state, action) tables would have more than 2^31 entries: count cell_next only");
    if (counts->next && n_sas > kJointLimit)
        return fail(GC_ERR_INVALID, "the joint 'next' table would have more than 2^31 entries");
    GC_ON_DEVICE(env->cfg.device);
    RolloutIO io = make_collect_io(env, n_steps, policy_kind, policy, epsilon, state, t, index, stats);
    CountIO cnt;
    cnt.visits = reinterpret_cast<unsigned long long *>(counts->visits);
    cnt.next = reinterpret_cast<unsigned long long *>(counts->next);
    cnt.reward_q24 = reinterpret_cast<unsigned long long *>(counts->reward_q24);
    cnt.unsafe = reinterpret_cast<unsigned long long *>(counts->unsafe);
    cnt.cell_next = reinterpret_cast<unsigned long long *>(counts->cell_next);
    cnt.n_states = static_cast<uint32_t>(nS);          // used only when a joint table fits, i.e. nS, nA <= 2^31
    cnt.n_actions = static_cast<uint32_t>(nA);
    cudaError_t e;
    if (cellular)
        e = gc_launch_cell_count(env->tab, io, cnt, env->d_pair_lut, (env->cfg.flags & GC_F_NOISE) != 0, env->n_sm,
                                 static_cast<cudaStream_t>(stream));
    else
        e = gc_launch_grid_count(env->grid, io, cnt, env->n_sm, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "count kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    env->global_step += n_steps;
    return GC_OK;
}

int gc_poll_status(gc_env *env, void *stream)
{
    GC_NVTX("gc_poll_status");
    if (int rc = check_env(env)) return rc;
    GC_ON_DEVICE(env->cfg.device);
    unsigned long long word = 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    GC_CUDA(cudaMemcpyAsync(&word, env->d_status, sizeof(word), cudaMemcpyDeviceToHost, st));
    GC_CUDA(cudaStreamSynchronize(st));
    if (word) {
        GC_CUDA(cudaMemsetAsync(env->d_status, 0, sizeof(word), st));
        return fail(GC_ERR_ACTION, "'position': a grid-world action named no go-to position in any jurisdiction");
    }
    return GC_OK;
}

int gc_encode(int device, int64_t n, int64_t ld, int32_t n_cells, int32_t radix, const int8_t *cells,
              uint32_t *index, void *stream)
{
    if (!cells || !index || n < 0 || ld < n || ld % 16 != 0 || n_cells < 1 || radix < 1)
        return fail(GC_ERR_INVALID, "gc_encode: bad arguments");
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_encode((n + 3) / 4 * 4, ld, n_cells, (uint32_t)radix, cells, index,
                                     static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "encode kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

int gc_decode(int device, int64_t n, int64_t ld, int32_t n_cells, int32_t radix, const uint32_t *index,
              int8_t *cells, void *stream)
{
    if (!cells || !index || n < 0 || ld < n || ld % 16 != 0 || n_cells < 1 || radix < 1)
        return fail(GC_ERR_INVALID, "gc_decode: bad arguments");
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_decode((n + 3) / 4 * 4, ld, n_cells, (uint32_t)radix, index, cells,
                                     static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "decode kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

namespace {
// radix / min: host arrays of n_cells entries; the product of the radices must fit the 32-bit index
int check_mixed(const char *who, int64_t n, int64_t ld, int32_t n_cells, const int32_t *radix, const int32_t *min)
{
    if (n < 0 || ld < n || ld % 16 != 0 || n_cells < 1 || n_cells > GC_MAX_CELLS || !radix)
        return fail(GC_ERR_INVALID, "%s: bad arguments", who);
    double bits = 0.0;
    for (int c = 0; c < n_cells; ++c) {
        if (radix[c] < 1 || radix[c] > 256) return fail(GC_ERR_INVALID, "%s: radix[%d] = %d not in 1..256", who, c, radix[c]);
        const int lo = min ? min[c] : 0;
        if (lo < -128 || lo + radix[c] - 1 > 127)
            return fail(GC_ERR_INVALID, "%s: cell %d spans [%d, %d], outside int8", who, c, lo, lo + radix[c] - 1);
        bits += std::log2((double)radix[c]);
    }
    if (bits > 32.0 + 1e-9) return fail(GC_ERR_INVALID, "%s: the space does not fit the 32-bit tabular index", who);
    return GC_OK;
}
}  // namespace

int gc_encode_mixed(int device, int64_t n, int64_t ld, int32_t n_cells, const int32_t *radix, const int32_t *min,
                    const int8_t *cells, uint32_t *index, void *stream)
{
    GC_NVTX("gc_encode_mixed");
    if (!cells || !index) return fail(GC_ERR_INVALID, "gc_encode_mixed: cells/index is NULL");
    if (int rc = check_mixed("gc_encode_mixed", n, ld, n_cells, radix, min)) return rc;
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_encode_mixed((n + 3) / 4 * 4, ld, n_cells, radix, min, cells, index, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "encode kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

int gc_decode_mixed(int device, int64_t n, int64_t ld, int32_t n_cells, const int32_t *radix, const int32_t *min,
                    const uint32_t *index, int8_t *cells, void *stream)
{
    GC_NVTX("gc_decode_mixed");
    if (!cells || !index) return fail(GC_ERR_INVALID, "gc_decode_mixed: cells/index is NULL");
    if (int rc = check_mixed("gc_decode_mixed", n, ld, n_cells, radix, min)) return rc;
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_decode_mixed((n + 3) / 4 * 4, ld, n_cells, radix, min, index, cells, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "decode kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

// ---- packed layout (include/gym_cellular_b200.h: "Packed layout") ---------------------------------

int gc_reset_packed(gc_env *env, const uint8_t *mask, uint32_t *state, int32_t *t, uint32_t *index, void *stream)
{
    GC_NVTX("gc_reset_packed");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (int rc = check_packed(env)) return rc;
    if (!state || !t) return fail(GC_ERR_INVALID, "state/t is NULL");
    GC_ON_DEVICE(env->cfg.device);
    cudaError_t e = gc_launch_reset_packed(env->tab.init_packed, env->tab.init_index, mask, state, t, index,
                                           env->cfg.n_envs, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "reset kernel launch failed: %s", cudaGetErrorString(e));
    env->launches += 1;
    return GC_OK;
}

int gc_step_packed(gc_env *env, int64_t env_begin, int64_t env_count, const uint32_t *actions, uint32_t *state,
                   int32_t *t, float *reward, uint32_t *index, uint8_t *flags, uint32_t *final_state,
                   uint32_t *se_row, int64_t *stats, void *stream)
{
    GC_NVTX("gc_step_packed");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (int rc = check_packed(env)) return rc;
    if (!actions || !state || !t || !reward || !flags) return fail(GC_ERR_INVALID, "a required device pointer is NULL");
    if (int rc = check_range(env, env_begin, env_count)) return rc;
    GC_ON_DEVICE(env->cfg.device);
    PackedIO io = make_packed_io(env, env_begin, env_count, actions, state, t, reward, index, flags, final_state,
                                 se_row, stats);
    const bool full = env_begin == 0 && env_count == env->cfg.n_envs;
    if (full) io.done_ctr = env->d_done;
    if (int rc = launch_packed(env, io, static_cast<cudaStream_t>(stream))) return rc;
    if (full) {
        env->global_step += 1;
    } else if (env_begin + env_count == env->cfg.n_envs) {
        if (int rc = tick_global_step(env, static_cast<cudaStream_t>(stream))) return rc;
    }
    return GC_OK;
}

int gc_bind_step_packed(gc_env *env, int32_t slot, const uint32_t *actions, uint32_t *state, int32_t *t,
                        float *reward, uint32_t *index, uint8_t *flags, uint32_t *final_state, uint32_t *se_row,
                        int64_t *stats)
{
    if (int rc = check_env(env)) return rc;
    if (int rc = check_packed(env)) return rc;
    if (slot < 0 || slot >= GC_MAX_BINDINGS) return fail(GC_ERR_INVALID, "slot must be in [0, %d)", GC_MAX_BINDINGS);
    if (!actions || !state || !t || !reward || !flags) return fail(GC_ERR_INVALID, "a required device pointer is NULL");
    env->bound_packed[slot] = make_packed_io(env, 0, env->cfg.n_envs, actions, state, t, reward, index, flags,
                                             final_state, se_row, stats);
    env->bound_packed[slot].done_ctr = env->d_done;
    env->bound_set[slot] = 2;
    drop_many_graphs(env);
    return GC_OK;
}

int gc_step_host_packed(gc_env *env, const uint32_t *h_actions, uint32_t *h_state, float *h_reward,
                        uint32_t *h_index, uint8_t *h_flags, uint32_t *d_actions, uint32_t *d_state, int32_t *d_t,
                        float *d_reward, uint32_t *d_index, uint8_t *d_flags, int64_t *d_stats, int64_t chunk_envs)
{
    GC_NVTX("gc_step_host_packed");
    if (int rc = check_env(env)) return rc;
    if (!env->tables_set) return fail(GC_ERR_STATE, "gc_set_tables has not been called");
    if (int rc = check_packed(env)) return rc;
    if (!h_actions || !d_actions || !d_state || !d_t || !d_reward || !d_flags)
        return fail(GC_ERR_INVALID, "a required pointer is NULL");
    if (h_index && !d_index) return fail(GC_ERR_INVALID, "h_index needs d_index");
    GC_ON_DEVICE(env->cfg.device);
    if (int rc = host_streams(env)) return rc;
    const int64_t n = env->cfg.n_envs;
    if (chunk_envs <= 0) chunk_envs = 1 << 20;
    chunk_envs = (chunk_envs + 15) / 16 * 16;
    HostDrain drain{env};
    int k = 0;
    for (int64_t b = 0; b < n; b += chunk_envs, ++k) {
        const int64_t cnt = (b + chunk_envs < n) ? chunk_envs : (n - b);
        cudaStream_t st = env->hstream[k % kHostStreams];
        GC_CUDA(cudaMemcpyAsync(d_actions + b, h_actions + b, cnt * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        const PackedIO io = make_packed_io(env, b, cnt, d_actions, d_state, d_t, d_reward, d_index, d_flags,
                                           nullptr, nullptr, d_stats);
        if (int rc = launch_packed(env, io, st)) return rc;
        if (h_state) GC_CUDA(cudaMemcpyAsync(h_state + b, d_state + b, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (h_reward) GC_CUDA(cudaMemcpyAsync(h_reward + b, d_reward + b, cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
        if (h_index) GC_CUDA(cudaMemcpyAsync(h_index + b, d_index + b, cnt * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (h_flags) GC_CUDA(cudaMemcpyAsync(h_flags + b, d_flags + b, cnt, cudaMemcpyDeviceToHost, st));
    }
    for (int i = 0; i < kHostStreams && i < k; ++i) GC_CUDA(cudaStreamSynchronize(env->hstream[i]));
    if (int rc = tick_global_step(env, env->hstream[0])) return rc;
    GC_CUDA(cudaStreamSynchronize(env->hstream[0]));
    drain.done = true;
    return GC_OK;
}

int gc_pack_cells(int device, int64_t n, int64_t ld, int32_t n_cells, const int8_t *cells, uint32_t *packed, void *stream)
{
    if (!cells || !packed || n < 0 || ld < n || ld % 16 != 0 || n_cells < 1 || n_cells > GC_MAX_CELLS)
        return fail(GC_ERR_INVALID, "gc_pack_cells: bad arguments");
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_pack((n + 3) / 4 * 4, ld, n_cells, cells, packed, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "pack kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

int gc_unpack_cells(int device, int64_t n, int64_t ld, int32_t n_cells, const uint32_t *packed, int8_t *cells, void *stream)
{
    if (!cells || !packed || n < 0 || ld < n || ld % 16 != 0 || n_cells < 1 || n_cells > GC_MAX_CELLS)
        return fail(GC_ERR_INVALID, "gc_unpack_cells: bad arguments");
    GC_ON_DEVICE(device);
    cudaError_t e = gc_launch_unpack((n + 3) / 4 * 4, ld, n_cells, packed, cells, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(GC_ERR_CUDA, "unpack kernel launch failed: %s", cudaGetErrorString(e));
    return GC_OK;
}

}  // extern "C"
