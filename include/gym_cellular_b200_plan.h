/*
 * gym_cellular_b200_plan.h -- C ABI of libgymcellular_b200_plan.so: batched value iteration on the device.
 *
 * The planner consumes the count format of gc_collect_counts (include/gym_cellular_b200.h), or explicit float64
 * models, and returns the greedy int32 policy tables that gc_rollout / gc_collect / gc_collect_counts take (one table,
 * or a stack for GC_POLICY_TABLE_STACK).  It needs no env handle: it is a separate library so that the env library's
 * kernels stay exactly the step, rollout and count kernels.
 *
 * Conventions are those of gym_cellular_b200.h: every function returns GC_OK or a negative gc_status, and
 * gcp_last_error() returns a thread-local message.
 *
 * Arithmetic, per model m (stated exactly; tests/_plan_reference.py restates it):
 *   counts input  n = max(visits[s][a], 1) as a double,
 *                 p(s'|s,a) = (double)next[s][a][s'] / n,  r(s,a) = ((double)reward_q24[s][a] * 2^-24) / n
 *                 (an unvisited pair has no successor and reward 0)
 *   model input   p = P[m][s][a][s'], r = R[m][s][a]
 *   V_0 = +0.0; for k = 1..iters:
 *     sum = +0.0; for s' ascending with p != 0: sum = sum + p * V_{k-1}(s')    (each * and + rounded on its own)
 *     Q_k(s,a) = r + gamma * sum
 *     pi_k(s) = the smallest a maximising Q_k(s, .),  V_k(s) = Q_k(s, pi_k(s))
 *   Skipping p = 0 changes no bit while V is finite: such a term adds +-0 to sum.
 * The outputs are pi_iters and V_iters.  Non-finite model entries give non-finite values (and a policy entry in
 * [0, nA)), never an access outside the arrays.  Nothing on the host depends on the data: a call adds no
 * synchronisation and can be captured into a CUDA graph.
 */
#ifndef GYM_CELLULAR_B200_PLAN_H
#define GYM_CELLULAR_B200_PLAN_H

#include "gym_cellular_b200.h"      /* gc_status */

#ifdef __cplusplus
extern "C" {
#endif

#define GCP_ABI_VERSION 1
#define GCP_MAX_STATES 4096             /* nS of one model                                               */
#define GCP_MAX_STATE_ACTIONS 131072    /* nS * nA of one model (2^17)                                   */

/* The models of one call, all of one shape: n_models x nS states x nA actions, contiguous, model-major.  Exactly one
 * input kind is given, the other's pointers are NULL:
 *   counts  visits, reward_q24 [n_models][nS][nA] and next [n_models][nS][nA][nS], int64, 8-byte aligned (the joint
 *           tables of gc_counts, grouped or not)
 *   model   P [n_models][nS][nA][nS] and R [n_models][nS][nA], float64, 8-byte aligned
 * n_models * nS * nA * nS is at most 2^31. */
typedef struct {
    uint32_t struct_size;          /* sizeof(gcp_model), for ABI evolution */
    int32_t n_models;
    int32_t n_states;
    int32_t n_actions;
    const int64_t *visits;
    const int64_t *next;
    const int64_t *reward_q24;
    const double *P;
    const double *R;
} gcp_model;

int         gcp_abi_version(void);
const char *gcp_last_error(void);

/* Value iteration of every model of `model`, `iters` iterations with discount `gamma` (finite, in [0, 1]), in one
 * kernel launch on `stream` (a cudaStream_t; NULL = the legacy default stream) of device `device`.  Writes policy
 * int32 [n_models][nS] (4-byte aligned) and value float64 [n_models][nS] (8-byte aligned), device arrays.  Every
 * argument is validated before any CUDA call: GC_ERR_INVALID with a message for NULLs, misalignment, sizes beyond
 * the limits above, gamma and iters < 1; GC_ERR_CUDA if the launch fails. */
int gcp_value_iteration(int device, const gcp_model *model, double gamma, int32_t iters, int32_t *policy, double *value,
                        void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GYM_CELLULAR_B200_PLAN_H */
