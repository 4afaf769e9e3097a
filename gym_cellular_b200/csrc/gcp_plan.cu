// libgymcellular_b200_plan.so: batched value iteration, one thread-block cluster per model, one launch per call
// (include/gym_cellular_b200_plan.h states the arithmetic).
//
// Rows across the cluster: the model's states are split over the cluster's CTAs in contiguous ranges.  Each CTA scans
// its own (s, a) rows of the dense input once, one warp per row with a ballot over the nonzeros, and compacts them
// into shared memory as (s', p) entries behind row offsets, p formed once in float64.  A CTA whose nonzeros do not fit
// reads its rows densely from global memory (L2) in every iteration instead; skipping p = 0 is exact either way, so
// both give the same bits.
//
// V across the cluster: V_{k-1} is double-buffered in every CTA's shared memory.  A warp computes one state's Q
// values, lanes over actions, reduces the maximum with the first-index rule by shuffles, and writes V_k(s) into every
// CTA's copy through distributed shared memory; one cluster barrier per iteration.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <map>
#include <mutex>
#include <tuple>

#include "gym_cellular_b200_plan.h"

namespace cg = cooperative_groups;

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

constexpr int kPlanThreads = 256;
constexpr int kPlanWarps = kPlanThreads / 32;
constexpr int kMaxCluster = 16;                        // non-portable cluster size (8 is the portable limit)
constexpr int kEntryBytes = sizeof(double) + sizeof(uint16_t);   // one compacted (p, s') entry; s' < 4096

struct PlanArgs {
    const int64_t *visits, *next, *reward_q24;         // counts input
    const double *P, *R;                               // model input
    int32_t *policy;
    double *value;
    double gamma;
    int32_t nS, nA, iters;
    int32_t rows_cap;                                  // ceil(nS / cluster size) * nA: the rows of the largest range
    int32_t entry_cap;                                 // compacted entries that fit in a CTA's shared memory
};

// Shared memory of one CTA, in this order: V[2][nS] (double), r[rows_cap] (double), row offsets[rows_cap + 1] (int32,
// padded to 8 bytes), p[entry_cap] (double), s'[entry_cap] (uint16).
__host__ __device__ inline size_t fixed_smem(int nS, int rows_cap)
{
    return (2 * static_cast<size_t>(nS) + rows_cap) * sizeof(double) + (static_cast<size_t>(rows_cap) + 2) / 2 * 8;
}

// p(s' = t | row) of the dense input; `n` is max(visits, 1) of the row (counts input).
template <bool COUNTS>
__device__ __forceinline__ double dense_p(const PlanArgs &a, int64_t row, double n, int t)
{
    const int64_t i = row * a.nS + t;
    if constexpr (COUNTS)
        return __ddiv_rn(static_cast<double>(__ldg(a.next + i)), n);
    else
        return __ldg(a.P + i);
}

template <bool COUNTS>
__device__ __forceinline__ double row_n(const PlanArgs &a, int64_t row)
{
    if constexpr (COUNTS) {
        const double v = static_cast<double>(__ldg(a.visits + row));
        return v < 1.0 ? 1.0 : v;
    } else {
        return 1.0;
    }
}

template <bool COUNTS>
__global__ void __launch_bounds__(kPlanThreads) plan_kernel(PlanArgs a)
{
    cg::cluster_group cluster = cg::this_cluster();
    const int c = static_cast<int>(cluster.num_blocks());
    const int rank = static_cast<int>(cluster.block_rank());
    const int64_t m = blockIdx.x / c;
    const int nS = a.nS, nA = a.nA;
    const int s0 = static_cast<int>(static_cast<int64_t>(rank) * nS / c);
    const int s1 = static_cast<int>(static_cast<int64_t>(rank + 1) * nS / c);
    const int rows = (s1 - s0) * nA;
    const int64_t grow0 = (m * nS + s0) * nA;          // global row of the CTA's first row
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;

    extern __shared__ __align__(16) unsigned char smem[];
    double *V = reinterpret_cast<double *>(smem);
    double *rew = V + 2 * nS;
    int32_t *off = reinterpret_cast<int32_t *>(rew + a.rows_cap);
    double *pe = reinterpret_cast<double *>(smem + fixed_smem(nS, a.rows_cap));
    uint16_t *col = reinterpret_cast<uint16_t *>(pe + a.entry_cap);

    // 1. nonzeros per row, the rewards, V_0 = +0.0
    for (int i = threadIdx.x; i < nS; i += kPlanThreads)
        V[i] = 0.0;
    for (int r = warp; r < rows; r += kPlanWarps) {
        const double n = row_n<COUNTS>(a, grow0 + r);
        int cnt = 0;
        for (int t0 = 0; t0 < nS; t0 += 32) {
            const int t = t0 + lane;
            cnt += __popc(__ballot_sync(~0u, t < nS && dense_p<COUNTS>(a, grow0 + r, n, t) != 0.0));
        }
        if (lane == 0) {
            off[r + 1] = cnt;
            if constexpr (COUNTS)
                rew[r] = __ddiv_rn(__dmul_rn(static_cast<double>(__ldg(a.reward_q24 + grow0 + r)), 0x1p-24), n);
            else
                rew[r] = __ldg(a.R + grow0 + r);
        }
    }
    __syncthreads();
    // 2. row offsets: an inclusive scan of the counts by warp 0 (at most 2^17 rows of at most 4096 entries: int32)
    if (warp == 0) {
        int carry = 0;
        for (int base = 0; base < rows; base += 32) {
            const int i = base + lane;
            int v = i < rows ? off[i + 1] : 0;
#pragma unroll
            for (int o = 1; o < 32; o *= 2) {
                const int u = __shfl_up_sync(~0u, v, o);
                if (lane >= o) v += u;
            }
            if (i < rows) off[i + 1] = v + carry;
            carry += __shfl_sync(~0u, v, 31);
        }
        if (lane == 0) off[0] = 0;
    }
    __syncthreads();
    const bool dense = off[rows] > a.entry_cap;
    // 3. compaction: entry order within a row is ascending s', as the contract sums
    if (!dense) {
        for (int r = warp; r < rows; r += kPlanWarps) {
            const double n = row_n<COUNTS>(a, grow0 + r);
            int pos = off[r];
            for (int t0 = 0; t0 < nS; t0 += 32) {
                const int t = t0 + lane;
                const double p = t < nS ? dense_p<COUNTS>(a, grow0 + r, n, t) : 0.0;
                const unsigned b = __ballot_sync(~0u, p != 0.0);
                if (p != 0.0) {
                    const int e = pos + __popc(b & ((1u << lane) - 1u));
                    pe[e] = p;
                    col[e] = static_cast<uint16_t>(t);
                }
                pos += __popc(b);
            }
        }
    }
    // Every CTA of the cluster has started and zeroed its V_0 before any CTA writes into another's shared memory.
    cluster.sync();

    // 4. the iterations.  Iteration k reads only the local buffer V[(k-1) & 1] and writes V_k into buffer k & 1 of
    // every CTA.  One barrier per iteration is enough: a CTA that has passed barrier k (and so writes buffer
    // (k+1) & 1 = (k-1) & 1 in iteration k + 1) knows that every CTA has finished iteration k, hence its reads of
    // that buffer, and every read of buffer k & 1 in iteration k + 1 comes after barrier k, hence after every write of
    // it.  The last iteration writes nothing remote, so no CTA writes into one that has exited.
    for (int k = 1; k <= a.iters; ++k) {
        const double *Vp = V + ((k - 1) & 1) * nS;
        const int nxt = (k & 1) * nS;
        const bool last = k == a.iters;
        for (int s = s0 + warp; s < s1; s += kPlanWarps) {
            const int lrow = (s - s0) * nA;
            double best = 0.0;
            int bi = nA;                                       // nA = none yet
            for (int act = lane; act < nA; act += 32) {
                const int r = lrow + act;
                double sum = 0.0;
                if (!dense) {
                    const int e1 = off[r + 1];
                    for (int e = off[r]; e < e1; ++e)
                        sum = __dadd_rn(sum, __dmul_rn(pe[e], Vp[col[e]]));
                } else {
                    const double n = row_n<COUNTS>(a, grow0 + r);
                    for (int t = 0; t < nS; ++t) {
                        const double p = dense_p<COUNTS>(a, grow0 + r, n, t);
                        if (p != 0.0)
                            sum = __dadd_rn(sum, __dmul_rn(p, Vp[t]));
                    }
                }
                const double q = __dadd_rn(rew[r], __dmul_rn(a.gamma, sum));
                if (bi == nA || q > best) {                    // strict: the first maximum of this lane's actions
                    best = q;
                    bi = act;
                }
            }
            // first maximum over the lanes: the larger value, or the smaller action of an equal one
#pragma unroll
            for (int o = 16; o > 0; o /= 2) {
                const double ob = __shfl_down_sync(~0u, best, o);
                const int oi = __shfl_down_sync(~0u, bi, o);
                if (oi < nA && (bi == nA || ob > best || (ob == best && oi < bi))) {
                    best = ob;
                    bi = oi;
                }
            }
            const double v = __shfl_sync(~0u, best, 0);
            if (!last) {
                if (lane < c)
                    cluster.map_shared_rank(V, lane)[nxt + s] = v;
            } else if (lane == 0) {
                a.policy[m * nS + s] = bi;                     // lane 0 holds action 0 at least: bi < nA
                a.value[m * nS + s] = v;
            }
        }
        if (!last)
            cluster.sync();
    }
}

// The cluster size of a shape, its launch geometry and shared memory; cached per (device, input kind, shape).
struct Geometry {
    int cluster;
    int rows_cap;
    int entry_cap;
    size_t smem;
};

Geometry geometry_for(int c, int nS, int nA, size_t budget)
{
    Geometry g;
    g.cluster = c;
    g.rows_cap = (nS + c - 1) / c * nA;
    const size_t fixed = fixed_smem(nS, g.rows_cap);
    const size_t dense_bound = static_cast<size_t>(g.rows_cap) * nS;
    const size_t room = fixed < budget ? (budget - fixed) / kEntryBytes : 0;
    g.entry_cap = static_cast<int>(dense_bound < room ? dense_bound : room);
    g.smem = fixed + static_cast<size_t>(g.entry_cap) * kEntryBytes;
    return g;
}

// The rule (shapes only, no data): the smallest cluster whose CTAs can hold every entry of their rows even if every
// entry is nonzero (nS * nA * nS / c), or 16 if none can, raised to the most CTAs that still put every cluster of the
// call on its own SMs (SMs / n_models), and at most nS.  More CTAs per model cut the rows each CTA walks per
// iteration; fewer keep the clusters of many models resident in one wave.  A size the device cannot co-schedule
// (cudaOccupancyMaxActiveClusters < 1) falls back to the next smaller one.
template <bool COUNTS>
int choose_geometry(int device, int n_models, int nS, int nA, Geometry *out)
{
    using Key = std::tuple<int, bool, int, int, int>;
    static std::mutex mu;
    static std::map<Key, Geometry> cache;
    const Key key{device, COUNTS, n_models, nS, nA};
    {
        std::lock_guard<std::mutex> lock(mu);
        auto it = cache.find(key);
        if (it != cache.end()) {
            *out = it->second;
            return GC_OK;
        }
    }
    int n_sm = 0, optin = 0;
    cudaError_t e = cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(plan_kernel<COUNTS>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(plan_kernel<COUNTS>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    if (e != cudaSuccess)
        return fail(GC_ERR_CUDA, "gcp_value_iteration: device setup: %s", cudaGetErrorString(e));
    const size_t budget = static_cast<size_t>(optin);
    int c_fit = kMaxCluster;
    for (int c = 1; c <= kMaxCluster; ++c) {
        const Geometry g = geometry_for(c, nS, nA, budget);
        if (static_cast<size_t>(g.entry_cap) == static_cast<size_t>(g.rows_cap) * nS) {
            c_fit = c;
            break;
        }
    }
    const int c_par = n_sm / n_models > 1 ? n_sm / n_models : 1;
    int c = c_fit > c_par ? c_fit : c_par;
    if (c > kMaxCluster) c = kMaxCluster;
    if (c > nS) c = nS;
    if (c > 0x7fffffff / n_models) c = 0x7fffffff / n_models;
    for (; c >= 1; --c) {
        const Geometry g = geometry_for(c, nS, nA, budget);
        if (fixed_smem(nS, g.rows_cap) > budget)
            continue;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(static_cast<unsigned>(c));
        cfg.blockDim = dim3(kPlanThreads);
        cfg.dynamicSmemBytes = g.smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = static_cast<unsigned>(c);
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, plan_kernel<COUNTS>, &cfg) != cudaSuccess) {
            (void)cudaGetLastError();                  // a size the query refuses is not an error of the call
            continue;
        }
        if (clusters >= 1) {
            std::lock_guard<std::mutex> lock(mu);
            cache[key] = g;
            *out = g;
            return GC_OK;
        }
    }
    return fail(GC_ERR_CUDA, "gcp_value_iteration: no cluster of %d x %d states x actions fits on device %d", nS, nA,
                device);
}

bool misaligned(const void *p, size_t a) { return reinterpret_cast<uintptr_t>(p) % a != 0; }

template <bool COUNTS>
int launch(int device, const gcp_model *model, double gamma, int32_t iters, int32_t *policy, double *value,
           cudaStream_t stream)
{
    Geometry g;
    const int rc = choose_geometry<COUNTS>(device, model->n_models, model->n_states, model->n_actions, &g);
    if (rc != GC_OK)
        return rc;
    PlanArgs a;
    a.visits = model->visits;
    a.next = model->next;
    a.reward_q24 = model->reward_q24;
    a.P = model->P;
    a.R = model->R;
    a.policy = policy;
    a.value = value;
    a.gamma = gamma;
    a.nS = model->n_states;
    a.nA = model->n_actions;
    a.iters = iters;
    a.rows_cap = g.rows_cap;
    a.entry_cap = g.entry_cap;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(static_cast<unsigned>(model->n_models) * static_cast<unsigned>(g.cluster));
    cfg.blockDim = dim3(kPlanThreads);
    cfg.dynamicSmemBytes = g.smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = static_cast<unsigned>(g.cluster);
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, plan_kernel<COUNTS>, a);
    if (e != cudaSuccess)
        return fail(GC_ERR_CUDA, "gcp_value_iteration: launch of %d clusters of %d: %s", model->n_models, g.cluster,
                    cudaGetErrorString(e));
    return GC_OK;
}

}  // namespace

extern "C" {

int gcp_abi_version(void) { return GCP_ABI_VERSION; }

const char *gcp_last_error(void) { return g_err; }

int gcp_value_iteration(int device, const gcp_model *model, double gamma, int32_t iters, int32_t *policy, double *value,
                        void *stream)
{
    if (!model)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: model is NULL");
    if (model->struct_size != sizeof(gcp_model))
        return fail(GC_ERR_INVALID, "model->struct_size %u != sizeof(gcp_model) %zu (ABI mismatch)", model->struct_size,
                    sizeof(gcp_model));
    if (device < 0)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: device %d < 0", device);
    const int64_t M = model->n_models, nS = model->n_states, nA = model->n_actions;
    if (M < 1 || nS < 1 || nA < 1)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: n_models %lld, n_states %lld and n_actions %lld must be >= 1",
                    (long long)M, (long long)nS, (long long)nA);
    if (nS > GCP_MAX_STATES)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: %lld states exceed the planner's limit of %d", (long long)nS,
                    GCP_MAX_STATES);
    if (nS * nA > GCP_MAX_STATE_ACTIONS)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: %lld x %lld state-action pairs exceed the planner's limit of %d",
                    (long long)nS, (long long)nA, GCP_MAX_STATE_ACTIONS);
    if (M * nS * nA * nS > (int64_t(1) << 31))
        return fail(GC_ERR_INVALID, "gcp_value_iteration: %lld models of %lld x %lld x %lld entries exceed 2^31 in all",
                    (long long)M, (long long)nS, (long long)nA, (long long)nS);
    const bool any_counts = model->visits || model->next || model->reward_q24;
    const bool any_model = model->P || model->R;
    if (any_counts == any_model)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: give either the counts (visits, next, reward_q24) or the "
                                    "model (P, R), not %s", any_counts ? "both" : "neither");
    if (any_counts && !(model->visits && model->next && model->reward_q24))
        return fail(GC_ERR_INVALID, "gcp_value_iteration: counts input needs visits, next and reward_q24 (one is NULL)");
    if (any_model && !(model->P && model->R))
        return fail(GC_ERR_INVALID, "gcp_value_iteration: model input needs P and R (one is NULL)");
    if (misaligned(model->visits, 8) || misaligned(model->next, 8) || misaligned(model->reward_q24, 8) ||
        misaligned(model->P, 8) || misaligned(model->R, 8))
        return fail(GC_ERR_INVALID, "gcp_value_iteration: input tables must be 8-byte aligned");
    if (!policy || !value)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: policy and value must not be NULL");
    if (misaligned(policy, 4) || misaligned(value, 8))
        return fail(GC_ERR_INVALID, "gcp_value_iteration: policy must be 4-byte and value 8-byte aligned");
    if (!std::isfinite(gamma) || gamma < 0.0 || gamma > 1.0)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: gamma %g must be finite and in [0, 1]", gamma);
    if (iters < 1)
        return fail(GC_ERR_INVALID, "gcp_value_iteration: iters %d must be >= 1", iters);

    int prev = -1;
    cudaError_t e = cudaGetDevice(&prev);
    if (e == cudaSuccess && prev != device) e = cudaSetDevice(device);
    if (e != cudaSuccess)
        return fail(GC_ERR_CUDA, "gcp_value_iteration: device %d: %s", device, cudaGetErrorString(e));
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rc = any_counts ? launch<true>(device, model, gamma, iters, policy, value, st)
                              : launch<false>(device, model, gamma, iters, policy, value, st);
    if (prev != device)
        cudaSetDevice(prev);
    return rc;
}

}  // extern "C"
