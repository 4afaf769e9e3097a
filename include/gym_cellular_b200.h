/*
 * gym_cellular_b200.h -- C ABI of libgymcellular_b200.so: the batched, B200-native (sm_100a)
 * environment step of gym-cellular.
 *
 * What this boundary replaces.  The reference has no FFI: its hot path is the Python method
 * `Env.step(action)` / `Env.reset()` of each environment class plus the tabular codec that agents
 * call on every observation.  Each entry point below cites the reference code it stands in for
 * (paths relative to the reference checkout):
 *
 *   gc_step    <- Cells3States3Actions3Env.step   gym_cellular/envs/cells3states3actions3.py:116-125
 *                 (transition_func :133-154, reward funcs :9-49, side_effects_func :157-212)
 *                 Cells2Rest3Env.step             gym_cellular/envs/cells2rest3.py:103-112
 *                 Cells3ResetVDeadlockEnv.step    gym_cellular/envs/cells3resetVdeadlock.py:148-157
 *                 (reset/add_noise/deadlock :35-68)
 *                 GridWorldEnv.step               gym_cellular/envs/grid_world.py:107-116
 *                 (transition_func :119-165, reward_func :30-39, side_effects_func :168-179)
 *                 + PriorKnowledge.tabularize of the returned state (cells3states3actions3.py:281-284,
 *                   grid_world.py:397-405)
 *   gc_reset   <- *.reset                         cells3states3actions3.py:99-113, grid_world.py:97-104
 *   gc_encode  <- generalized_cellular2tabular    gym_cellular/envs/utils/generalized_space_transformations.py:1-12
 *   gc_decode  <- generalized_tabular2cellular    gym_cellular/envs/utils/generalized_space_transformations.py:15-23
 *   gc_encode_mixed / gc_decode_mixed <- the same two functions with a per-cell space list (arbitrary
 *                 minimum and length per cell), as the reference defines them
 *   gc_step_packed / gc_step_host_packed <- the same step() in the packed layout (one 32-bit word per
 *                 env for the joint state, one for the joint action: "Packed layout" below)
 *   gc_step_host <- the same step() seen from a host caller (numpy in, numpy out): H2D of the
 *                 actions, the kernel, D2H of observation/reward/flags, pipelined in chunks.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no C++/torch types.  Every function returns 0 on
 *     success or a negative gc_status; gc_last_error() returns a thread-local message.
 *   - The CALLER owns every device buffer (torch tensors on the Python side, handed over as
 *     data_ptr()).  The library never allocates or frees per-step memory; a handle owns only its
 *     constant tables, a few streams/events for gc_step_host and one 64-bit device status word.
 *   - Batch layout: structure of arrays, cell-major.  `state` and `actions` are int8 [n_cells][ld]
 *     (element (c, e) at c*ld + e); per-env vectors have ld elements.  ld is the row stride,
 *     ld >= n_envs, ld % 16 == 0, all base pointers 16-byte aligned: kernels use vector accesses
 *     and may read/write the padding envs [n_envs, ld).
 *   - All calls are asynchronous on the given stream (`stream` is a cudaStream_t passed as
 *     void*; NULL = the legacy default stream).  gc_step never synchronises.
 *   - One host thread per handle at a time; handles are independent (one per GPU per rank).
 */
#ifndef GYM_CELLULAR_B200_H
#define GYM_CELLULAR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GC_ABI_VERSION 2

typedef struct gc_env gc_env;

typedef enum {
    GC_OK = 0,
    GC_ERR_INVALID = -1,      /* bad argument / unsupported shape */
    GC_ERR_CUDA = -2,         /* a CUDA runtime call failed (message has the CUDA error string) */
    GC_ERR_STATE = -3,        /* tables not set, handle destroyed, ... */
    GC_ERR_ACTION = -4        /* gc_poll_status: an env received an action the reference raises on */
} gc_status;

/* Environment families.  GC_KIND_CELLULAR is the table-driven per-cell MDP that covers the
 * polarisation family (Cells3States3Actions3, Cells2Rest3, Cells3ResetVDeadlock and the scaled
 * 16-cell x 4-state variant): every cell moves by the same [S][A] tables. */
#define GC_KIND_CELLULAR  0
#define GC_KIND_GRIDWORLD 1

/* gc_config.flags */
#define GC_F_NOISE        1u  /* stochastic cell transitions: Philox draw where the table says so  */
#define GC_F_RNG_EPISODIC 4u  /* RNG counter = episode step (the reference re-seeds in reset(),
                                 cells3resetVdeadlock.py:131); otherwise the handle's global step  */
#define GC_F_REWARD_LOG2  16u /* reward = log2(1 + sum) (`nonlinear`, cells3states3actions3.py:47-49) */
#define GC_F_GENERIC_KERNEL 32u /* always use the generic per-cell kernel, never the pair-table fast path (tests) */

#define GC_MAX_CELLS   16
#define GC_MAX_LEVELS  8      /* intracellular states / actions per cell */
#define GC_N_STATS     8

/* indices into the int64 statistics vector accumulated by gc_step (device memory, caller-owned) */
#define GC_STAT_STEPS       0 /* env-steps executed                                              */
#define GC_STAT_UNSAFE      1 /* steps whose side-effects row contains 'unsafe'                  */
#define GC_STAT_COUNT       2 /* sum of polarised cells (cellular) / barren jurisdictions (grid) */
#define GC_STAT_TRUNCATED   3 /* episodes ended by the time limit                                */
#define GC_STAT_REWARD_Q24  4 /* sum of round(reward * 2^24): order-independent, exact across GPUs (each
                                 term is a 32-bit integer: gc_set_tables keeps |reward| < 128) */

typedef struct {
    uint32_t struct_size;        /* sizeof(gc_config), for ABI evolution                          */
    int32_t  kind;               /* GC_KIND_*                                                     */
    int32_t  device;             /* CUDA device ordinal                                           */
    int32_t  n_cells;            /* cellular: 1..GC_MAX_CELLS; grid world: 2                      */
    int32_t  n_states;           /* levels per cell (cellular: 2..GC_MAX_LEVELS; grid world: 20)  */
    int32_t  n_actions;          /* intracellular actions (cellular: 1..GC_MAX_LEVELS; grid: 5)   */
    int32_t  max_episode_steps;  /* 0 = never truncate (reference behaviour, __init__.py:7);
                                    > 0 = time-limit truncation with fused auto-reset             */
    uint32_t flags;              /* GC_F_*                                                        */
    int64_t  n_envs;             /* envs of this shard                                            */
    int64_t  ld;                 /* row stride, >= n_envs, multiple of 16; n_cells * ld <= 2^31
                                    (the kernels index with 32-bit element offsets)               */
    int64_t  env_id_offset;      /* global id of env 0 (multiple of 4): RNG streams are keyed by global env id */
    uint64_t seed;               /* Philox key                                                    */
    double   noise_prob;         /* cellular noise threshold (0.1, cells3resetVdeadlock.py:36), in [0, 1] */
    double   dispersal_prob;     /* grid-world seed dispersal (0.01, grid_world.py:161), in [0, 1]        */
} gc_config;

/* Tables of the cellular family (host pointers, copied into the handle).
 *   move   [S][A] int8   next level without noise          (cells3states3actions3.py:133-154)
 *   noisy  [S][A] int8   next level when the draw fires    (cells3resetVdeadlock.py:37-41)
 *   draws  [S][A] uint8  1 if (level, action) consumes a draw (cells3resetVdeadlock.py:49-60)
 *   reward [S][A] float  per-cell reward of the OLD level  (cells3states3actions3.py:9-45); finite
 *   reward_noisy [S][A] float  optional: per-cell reward when the draw fired, for rewards that depend on
 *          the NEXT level (debug/deep_exploration.py:11-16); NULL = same as `reward`; finite
 *          Bound: every step's reward must stay below 128 in magnitude.  With lo / hi the smallest / largest
 *          entry of reward and reward_noisy, gc_set_tables requires n_cells * max(|lo|, |hi|) < 128 (under
 *          GC_F_REWARD_LOG2: 1 + n_cells * lo > 0 and |log2(1 + n_cells * lo)|, |log2(1 + n_cells * hi)| < 128),
 *          with a margin of n_cells * 2^-18 for the float32 sum.
 *   side_effects [C][S][S] int8  code (0 silent, 1 safe, 2 unsafe) of row-0 entry j of the
 *          side-effects matrix as a function of (s'_0, s'_p), p = 1 for j = 0 and p = j otherwise
 *          (cells3states3actions3.py:157-212; only row 0 is ever written by the reference)
 *   counted [S] uint8    1 if a cell at that level counts towards side_effects_incidence (:159-162)
 *   initial_state [C] int8                                   (cells3states3actions3.py:238)
 */
typedef struct {
    const int8_t  *move;
    const int8_t  *noisy;
    const uint8_t *draws;
    const float   *reward;
    const int8_t  *side_effects;
    const uint8_t *counted;
    const int8_t  *initial_state;
    const float   *reward_noisy;
    const int32_t *radix;        /* optional [C]: levels of each cell for the tabular index of a ragged state
                                    space (radix[c] <= n_states; the moves must keep cell c below radix[c]);
                                    NULL = n_states for every cell */
} gc_cell_tables;

int         gc_abi_version(void);
const char *gc_last_error(void);

int gc_create(const gc_config *cfg, gc_env **out);
int gc_destroy(gc_env *env);
/* Cellular family only.  Validates everything first: a rejected call leaves the previous tables in force.  The
 * staged device tables are replaced with synchronous copies, so steps still in flight on a NON-BLOCKING stream must
 * be waited for by the caller before the tables are changed; cached gc_step_many graphs are rebuilt on their next
 * use.  Int8 bindings stay valid and step by the new tables.  Packed bindings stay in their slots but step only
 * while the tables admit the packed layout (as gc_bind_step_packed requires): under other tables gc_step_bound and
 * gc_step_many / gc_prepare_step_many on a list holding one are refused with GC_ERR_INVALID before any step runs,
 * and they step again once such tables are set. */
int gc_set_tables(gc_env *env, const gc_cell_tables *tables);

/* Final observation (gymnasium's SAME_STEP auto-reset convention; the reference never ends an episode,
 * gym_cellular/__init__.py:7, so this belongs to the time limit added here): when set, every following
 * int8-layout step of the handle (gc_step, bound steps, gc_step_host) also writes the next state BEFORE the
 * auto-reset to final_state, int8 [C][ld] device memory owned by the caller; it equals `state` wherever
 * truncated == 0.  NULL switches it off.  Not part of the 3C + 20 algorithmic bytes (+C when on). */
int gc_set_final_obs(gc_env *env, int8_t *final_state);

/* Global step counter used as the RNG counter when GC_F_RNG_EPISODIC is off.  It lives in device
 * memory: a gc_step over the whole shard reads it in the kernel and the kernel advances it, so a
 * gc_step captured into a CUDA graph keeps drawing fresh numbers on every replay.  The host keeps a
 * mirror (gc_get_global_step); after graph replays call gc_sync_global_step to refresh it.
 * gc_set_global_step is synchronous: it returns once the device word holds the new value, and it is ordered only
 * after work on blocking streams.  A kernel still queued or running on a NON-BLOCKING stream reads the counter when
 * it runs and writes it back when it ends, so the caller must wait for that stream first. */
int gc_set_global_step(gc_env *env, int64_t step);
int64_t gc_get_global_step(const gc_env *env);
int gc_sync_global_step(gc_env *env, void *stream);
/* Number of kernels this handle has launched so far (bench.py's gpu_launches). */
int64_t gc_launch_count(const gc_env *env);

/* reset(): write the initial state, t = 0 and its tabular index for every env (mask == NULL) or
 * for the envs whose mask byte is non-zero.  mask: device uint8 [ld].  index may be NULL. */
int gc_reset(gc_env *env, const uint8_t *mask, int8_t *state, int32_t *t, uint32_t *index, void *stream);

/* One env.step() for envs [env_begin, env_begin + env_count) of the shard (pass 0, n_envs for all;
 * env_begin % 16 == 0).  All pointers are device pointers to the FULL arrays.
 *   actions    int8  [C][ld]  in      cellular: level chosen per cell; grid world: go-to position
 *                                     code per jurisdiction, 0..3 = row*2+col, 4 = none (other codes are
 *                                     invalid: the kernels stay memory-safe, the result is unspecified)
 *   state      int8  [C][ld]  in/out  cellular: level per cell; grid world: the reference's own
 *                                     cellular code per jurisdiction (grid_world.py:349-359)
 *   t          int32 [ld]     in/out  episode step (data['time_step'])
 *   reward     float [ld]     out
 *   index      uint32[ld]     out     tabular index of the returned state (little-endian mixed radix)
 *   terminated uint8 [ld]     out     always 0 (cells3states3actions3.py:121)
 *   truncated  uint8 [ld]     out     1 when the time limit fired (state/t/index are then the reset ones)
 *   unsafe     uint8 [ld]     out     1 if row 0 of the side-effects matrix holds 'unsafe'
 *   count      uint8 [ld]     out     polarised cells of the next state / barren jurisdictions of the
 *                                     pre-step state (= side_effects_incidence * n_cells)
 *   se_row     int8  [C][ld]  out     optional (NULL to skip): row 0 of the side-effects matrix
 *   replay_u   double[n][slots] in    optional: replayed uniform draws instead of Philox (parity
 *                                     tests); slots = n_cells (cellular: slot c = cell c) or 6 (grid
 *                                     world: trigger, b00, b01, b10, b11, k; randint(n) = floor(u*n))
 *   stats      int64 [GC_N_STATS] in/out optional accumulators (GC_STAT_*)
 */
int gc_step(gc_env *env, int64_t env_begin, int64_t env_count, const int8_t *actions, int8_t *state,
            int32_t *t, float *reward, uint32_t *index, uint8_t *terminated, uint8_t *truncated,
            uint8_t *unsafe, uint8_t *count, int8_t *se_row, const double *replay_u, int64_t *stats,
            void *stream);

/* Pre-bound step for tight loops: gc_bind_step stores the pointer set of a full-shard gc_step in one of
 * GC_MAX_BINDINGS slots of the handle, gc_step_bound launches it (same semantics as gc_step over
 * [0, n_envs)); the foreign-function call then carries three arguments instead of sixteen. */
#define GC_MAX_BINDINGS 16
int gc_bind_step(gc_env *env, int32_t slot, const int8_t *actions, int8_t *state, int32_t *t, float *reward,
                 uint32_t *index, uint8_t *terminated, uint8_t *truncated, uint8_t *unsafe, uint8_t *count,
                 int8_t *se_row, int64_t *stats);
int gc_step_bound(gc_env *env, int32_t slot, void *stream);
/* n_steps pre-bound steps back to back in ONE foreign call: step i launches slot slots[i % n_slots]
 * (int8 or packed bindings), one kernel per step, chained with programmatic dependent launch; no host code
 * runs between them.  Whole passes over the slot list (16 steps or more per graph) are replayed from a CUDA
 * graph the handle captures once per slot list (caller's stream not being captured; GC_B200_STEP_MANY_GRAPH=0
 * in the environment switches it off): the host then pays one call per 16 kernels, which is what bounds the
 * launch-bound batch sizes (BASELINE configs 2 and 3).  Same kernels, same results, same statistics.
 * Shards above 2^21 envs always take plain launches (their kernels are long enough to hide the host calls).
 * gc_prepare_step_many builds the graph of a slot list ahead of time (no step is executed), so that the first
 * gc_step_many does not pay for the capture.
 * ONE launch for all n_steps: when the slots of the list are bindings of one layout that differ only in their action
 * buffers (one set of in-place state / output arrays, a ring of action buffers), the shard has at most 2^21 envs
 * (cellular: levels and actions <= 4, at most 8 cells; or grid world) and no final-observation buffer is set, the
 * steps run inside a single kernel: the thread that owns an env keeps its state and episode step in registers
 * from one step to the next and writes EVERY per-step output (state, t, reward, index, flags, side-effect row,
 * statistics) at every step, as the separate launches would; results are bit-identical to them.  Only the
 * launch gaps and the re-read of state and t go away (a 65,536-env step is a 3 us launch around 0.6 us of work).
 * GC_B200_STEP_MANY_FUSED=0 in the environment (read at every call) keeps the separate launches. */
int gc_step_many(gc_env *env, const int32_t *slots, int32_t n_slots, int32_t n_steps, void *stream);
int gc_prepare_step_many(gc_env *env, const int32_t *slots, int32_t n_slots);

/* The same step for a HOST caller: h_* are host buffers (pinned for full speed) in the same
 * layouts with row stride ld; d_* the caller-owned resident device arrays.  Copies the actions in,
 * steps, copies state/reward/index/flags out, pipelined over chunks on the handle's own streams;
 * returns after everything has landed in the host buffers.  Any h_* output may be NULL; the row-0
 * side-effect codes are produced only when d_se_row is given (and copied out when h_se_row is). */
int gc_step_host(gc_env *env, const int8_t *h_actions, int8_t *h_state, float *h_reward,
                 uint32_t *h_index, uint8_t *h_terminated, uint8_t *h_truncated, uint8_t *h_unsafe,
                 uint8_t *h_count, int8_t *h_se_row, int8_t *d_actions, int8_t *d_state, int32_t *d_t,
                 float *d_reward, uint32_t *d_index, uint8_t *d_terminated, uint8_t *d_truncated,
                 uint8_t *d_unsafe, uint8_t *d_count, int8_t *d_se_row, int64_t *d_stats,
                 int64_t chunk_envs);

/* ---- Packed layout -------------------------------------------------------------------------------
 * Cellular family with n_states, n_actions <= 4 (every polarisation env of the reference and the 16 x 4
 * scale-up).  The joint state and the joint action of an env are ONE uint32 each, 2 bits per cell, cell c in
 * bits 2c and 2c+1 -- for n_states == 4 the state word is the reference's tabular index itself
 * (generalized_space_transformations.py:1-12: cell 0 least significant).  Per-env outputs shrink to the
 * reward and one flag byte, so an env-step moves 25 bytes through HBM instead of 3 n_cells + 20 and 4 bytes
 * in / 9 bytes out over the host link instead of n_cells / n_cells + 10:
 *   actions     uint32 [ld]  in      joint action word
 *   state       uint32 [ld]  in/out  joint state word
 *   t           int32  [ld]  in/out  episode step
 *   reward      float  [ld]  out
 *   index       uint32 [ld]  out     optional: tabular index of the returned state (== state when n_states == 4)
 *   flags       uint8  [ld]  out     bit 0 unsafe, bit 1 truncated, bits 2-6 count (GC_FLAG_*); terminated is
 *                                    always false (cells3states3actions3.py:121) and has no bit
 *   final_state uint32 [ld]  out     optional: the next state BEFORE the time-limit auto-reset (gymnasium's
 *                                    final observation; equals `state` where truncated == 0)
 *   se_row      uint32 [ld]  out     optional: row 0 of the side-effects matrix, 2 bits per entry
 * Same semantics, same Philox draws and bit-identical results as gc_step on the int8 layout
 * (gc_pack_cells / gc_unpack_cells convert).  Replay of recorded uniforms is offered by gc_step only. */
#define GC_FLAG_UNSAFE      1u
#define GC_FLAG_TRUNCATED   2u
#define GC_FLAG_COUNT_SHIFT 2
int gc_reset_packed(gc_env *env, const uint8_t *mask, uint32_t *state, int32_t *t, uint32_t *index, void *stream);
int gc_step_packed(gc_env *env, int64_t env_begin, int64_t env_count, const uint32_t *actions, uint32_t *state,
                   int32_t *t, float *reward, uint32_t *index, uint8_t *flags, uint32_t *final_state,
                   uint32_t *se_row, int64_t *stats, void *stream);
/* Packed binding (gc_bind_step's slots): refused unless the current tables admit the packed layout; a bound slot is
 * stepped only while they still do (gc_set_tables). */
int gc_bind_step_packed(gc_env *env, int32_t slot, const uint32_t *actions, uint32_t *state, int32_t *t,
                        float *reward, uint32_t *index, uint8_t *flags, uint32_t *final_state, uint32_t *se_row,
                        int64_t *stats);
/* Host caller, packed wire format: h_actions in (4 bytes per env), h_state / h_reward / h_flags (and h_index
 * when asked for) out; chunks pipelined over the handle's streams like gc_step_host.  (final_state and se_row
 * are outputs of the device path only.) */
int gc_step_host_packed(gc_env *env, const uint32_t *h_actions, uint32_t *h_state, float *h_reward,
                        uint32_t *h_index, uint8_t *h_flags, uint32_t *d_actions, uint32_t *d_state, int32_t *d_t,
                        float *d_reward, uint32_t *d_index, uint8_t *d_flags, int64_t *d_stats, int64_t chunk_envs);
/* int8 [n_cells][ld] levels <-> packed words [ld] */
int gc_pack_cells(int device, int64_t n, int64_t ld, int32_t n_cells, const int8_t *cells, uint32_t *packed, void *stream);
int gc_unpack_cells(int device, int64_t n, int64_t ld, int32_t n_cells, const uint32_t *packed, int8_t *cells, void *stream);

/* K-step fused rollout (the caller's loop around step(): pick an action, step, accumulate).  Runs
 * n_steps consecutive steps for every env of the shard inside ONE kernel; the state stays in
 * registers, actions are generated in the kernel:
 *   GC_POLICY_RANDOM  cellular: every cell draws uniformly from its actions; grid world: the
 *                     distribution of the reference's action sampler (one jurisdiction named, uniform
 *                     position; grid_world.py:191-195).  Philox, keyed like the step's noise.
 *   GC_POLICY_TABLE   action = policy[tabular state] (device int32 [n_states^n_cells], tabular action
 *                     index): `initial_policy` as a table (cells3states3actions3.py:293-295)
 * The result is bit-identical to n_steps calls of gc_step with the same actions.  Cellular family:
 * fast path only (n_states, n_actions <= 4).  ret [ld] float: sum of the n_steps rewards;
 * n_unsafe [ld] int32: steps that reported 'unsafe'; state / t / index as in gc_step. */
#define GC_POLICY_RANDOM 0
#define GC_POLICY_TABLE  1
int gc_rollout(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, int8_t *state,
               int32_t *t, uint32_t *index, float *ret, int32_t *n_unsafe, int64_t *stats, void *stream);

/* Transition record of gc_collect: step-major arrays [n_steps][ld] (element (k, e) at k*ld + e, the handle's ld),
 * device memory owned by the caller, base pointers 16-byte aligned.  Every pointer may be NULL (not recorded). */
typedef struct {
    uint32_t  struct_size;
    uint32_t *obs;       /* tabular index of the state step k starts from (what gc_step wrote to `index` before it) */
    uint32_t *action;    /* tabular action index of the action EXECUTED at step k                                 */
    float    *reward;    /* reward of step k, the bits gc_step writes                                             */
    uint8_t  *flags;     /* GC_FLAG_UNSAFE | GC_FLAG_TRUNCATED | count << GC_FLAG_COUNT_SHIFT                      */
    uint32_t *next_obs;  /* tabular index of the successor BEFORE the time-limit auto-reset (== obs[k+1] unless truncated) */
} gc_record;

/* Experience collection: the fused rollout above (same envs, same kernel, same advance of state, t, index, global
 * step, statistics and launch count) that also writes every transition into `record`.  Policies:
 *   GC_POLICY_RANDOM  as in gc_rollout; epsilon must be 0
 *   GC_POLICY_TABLE   epsilon-greedy, epsilon in [0, 1]: env g at global step G explores iff word (g % 4) of
 *                     philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000000)) < ceil(epsilon * 2^32); the explored action is
 *                     word (g % 4) of philox(key, ((g/4)_lo, (g/4)_hi, G, 0x50000001)) mapped to the joint action
 *                     floor(word * A^C / 2^32) (cellular) or by the random policy's rule (grid world); otherwise
 *                     action = policy[obs].  G is the global step even under GC_F_RNG_EPISODIC (exploration is the
 *                     agent's, not the environment's).  epsilon = 0 draws nothing: gc_rollout's actions exactly.
 * No per-env return / unsafe count: the record holds the per-step values.  One kernel launch. */
int gc_collect(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
               int8_t *state, int32_t *t, uint32_t *index, const gc_record *record, int64_t *stats, void *stream);

/* Experience counts of gc_collect_counts: int64 device arrays owned by the caller, 8-byte aligned, each NULL = not
 * counted (but not all of them).  s is the tabular index gc_collect records as `obs`, a the executed tabular action it
 * records as `action`, s' its `next_obs`; nS = n_states^n_cells, nA = n_actions^n_cells (grid world: 400 and 25).  A
 * joint table may have at most 2^31 entries; cell_next is cellular only (C = n_cells, S = n_states, A = n_actions). */
typedef struct {
    uint32_t struct_size;
    int64_t *visits;      /* [nS][nA]       N(s, a)                                                      */
    int64_t *next;        /* [nS][nA][nS]   N(s, a, s'), s' = successor BEFORE the time-limit auto-reset   */
    int64_t *reward_q24;  /* [nS][nA]       sum of round(reward * 2^24), the term GC_STAT_REWARD_Q24 adds  */
    int64_t *unsafe;      /* [nS][nA]       steps that reported 'unsafe'                                  */
    int64_t *cell_next;   /* [C][S][A][S]   per cell c: N_c(s_c, a_c, s'_c); cellular only               */
} gc_counts;

/* Experience counts: gc_collect with the same arguments (same envs, policies, epsilon rule, Philox streams, and the
 * same advance of state, t, index, global step, statistics and launch count) that ADDS every transition to `counts`
 * instead of recording it, so that the counts equal the histogram of gc_collect's record.  Integer counts: exact,
 * independent of the order of the adds and of the sharding of the envs.  Arguments are validated before any CUDA
 * call.  One kernel launch. */
int gc_collect_counts(gc_env *env, int32_t n_steps, int32_t policy_kind, const int32_t *policy, double epsilon,
                      int8_t *state, int32_t *t, uint32_t *index, const gc_counts *counts, int64_t *stats, void *stream);

/* Reads and clears the handle's device status word (synchronises `stream`).  Returns GC_OK or
 * GC_ERR_ACTION if some env received a grid-world action without any go-to position since the
 * last poll (the reference raises KeyError('position'), grid_world.py:143). */
int gc_poll_status(gc_env *env, void *stream);

/* Standalone batched codec, uniform radix (cells int8 [n_cells][ld], index uint32 [ld]). */
int gc_encode(int device, int64_t n, int64_t ld, int32_t n_cells, int32_t radix, const int8_t *cells,
              uint32_t *index, void *stream);
int gc_decode(int device, int64_t n, int64_t ld, int32_t n_cells, int32_t radix, const uint32_t *index,
              int8_t *cells, void *stream);

/* The reference's codec with its per-cell space list (generalized_space_transformations.py:1-23): cell c
 * takes the values min[c] .. min[c] + radix[c] - 1 (radix, min: HOST arrays of n_cells entries, min may be
 * NULL = all zero); index = sum_c (cells[c] - min[c]) * prod_{k<c} radix[k].  The product of the radices
 * must fit the 32-bit index (the reference works on unbounded Python ints). */
int gc_encode_mixed(int device, int64_t n, int64_t ld, int32_t n_cells, const int32_t *radix, const int32_t *min,
                    const int8_t *cells, uint32_t *index, void *stream);
int gc_decode_mixed(int device, int64_t n, int64_t ld, int32_t n_cells, const int32_t *radix, const int32_t *min,
                    const uint32_t *index, int8_t *cells, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GYM_CELLULAR_B200_H */
