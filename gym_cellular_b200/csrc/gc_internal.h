// Internal declarations shared by the kernels (gc_kernels.cu) and the C ABI (gc_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gym_cellular_b200.h"

#define GC_LVL_PAD 8                       // tables are indexed [s * GC_LVL_PAD + a]
#define GC_TBL (GC_LVL_PAD * GC_LVL_PAD)   // 64 entries

// Cellular noise draws: envs of up to GC_NARROW_CELLS cells take one 32-bit Philox word per cell (one block
// per env); wider envs take one 16-bit half per cell (eight cells per block) plus 16 lazily drawn bits (gc_device.cuh)
#define GC_NARROW_CELLS 4
#define GC_NOISE_LOW_STREAM 0x20000000u   // Philox stream of the low 16 bits of cell c's draw: GC_NOISE_LOW_STREAM + c

// RNG source of a launch
enum { GC_RNG_NONE = 0, GC_RNG_PHILOX = 1, GC_RNG_REPLAY = 2 };

// Per-env array pointers of one step launch (device pointers to the full arrays).
struct StepIO {
    const int8_t *actions;
    int8_t       *state;
    int32_t      *t;
    float        *reward;
    uint32_t     *index;
    uint8_t      *terminated, *truncated, *unsafe, *count;
    int8_t       *se_row;       // optional
    int8_t       *final_state;  // optional, [C][ld]: next state BEFORE the time-limit auto-reset (final observation)
    const double *replay;       // optional, [n][slots]
    unsigned long long *stats;  // optional, int64[GC_N_STATS]
    unsigned long long *status; // handle-owned status word
    int64_t begin, end;         // env range of this launch (end <= n_envs)
    int64_t ld;
    int64_t env_id_offset;
    uint32_t seed_lo, seed_hi;
    uint32_t round_key[20];     // Philox round keys (k0_r, k1_r), r = 0..9: warp-uniform, precomputed on the host
    uint32_t rng_counter;       // global step (ignored when episodic); used when step_ctr == NULL
    const uint32_t *step_ctr;   // device-resident global step: read by every thread at kernel entry and
    uint32_t *done_ctr;         // advanced by the last block to finish (CUDA-graph friendly), or NULL
    int32_t  episodic;
    int32_t  max_episode_steps;
};

// gc_step_many in ONE launch (gc_cell_fast.cu: cell_pair_many_kernel; gc_grid.cu: grid_many_kernel): the bound
// steps of a handle whose slots share every buffer but the actions
struct ManyIO {
    StepIO io;                                  // the shared buffers (io.actions is not used)
    const int8_t *tape[GC_MAX_BINDINGS];        // actions of step k: tape[k % n_tape]
    int32_t n_tape, n_steps;
};
#define GC_MANY_MAX_CELLS 8

// Packed layout (gc_cell_packed.cu): ONE 32-bit word per env for the state and one for the action, 2 bits per
// cell (cell c in bits 2c, 2c+1; n_states, n_actions <= 4).  For n_states == 4 the state word IS the tabular
// index.  Per-env outputs shrink to reward + one flag byte.
struct PackedIO {
    const uint32_t *actions;    // [ld]
    uint32_t *state;            // [ld] in/out
    int32_t  *t;                // [ld] in/out
    float    *reward;           // [ld] out
    uint32_t *index;            // [ld] out, optional: tabular index of the returned state
    uint8_t  *flags;            // [ld] out: bit 0 unsafe, bit 1 truncated, bits 2-6 count
    uint32_t *final_state;      // [ld] out, optional: next state BEFORE the auto-reset (final observation)
    uint32_t *se_row;           // [ld] out, optional: row 0 of the side-effects matrix, 2 bits per entry
    unsigned long long *stats;
    unsigned long long *status;
    int64_t begin, end, ld, env_id_offset;
    uint32_t round_key[20];
    uint32_t rng_counter;
    const uint32_t *step_ctr;
    uint32_t *done_ctr;
    int32_t episodic, max_episode_steps;
};

struct PackedManyIO {                           // gc_step_many in one launch, packed bindings (gc_cell_packed.cu)
    PackedIO io;                                // the shared buffers (io.actions is not used)
    const uint32_t *tape[GC_MAX_BINDINGS];      // action words of step k: tape[k % n_tape]
    int32_t n_tape, n_steps;
};

// K-step fused rollout (gc_rollout.cu): state stays in registers for n_steps steps, actions are
// generated in the kernel (uniformly random, or from a tabular policy).
struct RolloutIO {
    int8_t       *state;
    int32_t      *t;
    uint32_t     *index;
    float        *ret;          // [ld] out: sum of the rewards of the n_steps steps
    int32_t      *n_unsafe;     // [ld] out: steps that reported 'unsafe'
    const int32_t *policy;      // GC_POLICY_TABLE(_STACK): tabular action index per tabular state, else NULL
    unsigned long long *stats;
    unsigned long long *status;
    int64_t n, ld, env_id_offset;
    uint32_t round_key[20];
    const uint32_t *step_ctr;
    uint32_t *done_ctr;
    int32_t episodic, max_episode_steps, n_steps, policy_kind;
    // gc_collect (the RECORD kernels; appended so that the fields above keep their offsets): the transition
    // record, step-major [n_steps][ld], each pointer NULL = not recorded
    uint32_t *rec_obs, *rec_action, *rec_next_obs;
    float    *rec_reward;
    uint8_t  *rec_flags;
    unsigned long long joint_actions;        // A^C (<= 2^32): an explored cellular action is floor(word * A^C / 2^32)
    uint32_t explore_thr_m1, explore_thr_nz; // the table policy explores iff thr_nz && word <= thr_m1 (P = eps)
    // GC_POLICY_TABLE_STACK (appended like the record fields): env e acts by table row table_of_env[e], clamped to
    // [0, n_tables), of policy [n_tables][table_stride]
    const int32_t *table_of_env;             // [ld], 16-byte aligned
    unsigned long long table_stride;         // nS: n_states^n_cells (grid world 400)
    uint32_t n_tables;
};

// gc_collect_counts (the COUNT rollout kernels): int64 counters the kernels add to, NULL = not counted.  A kernel
// parameter of its own, after the others, so that RolloutIO and the other kernels' parameters keep their layout.
struct CountIO {
    unsigned long long *visits;        // [nS][nA]
    unsigned long long *next;          // [nS][nA][nS]
    unsigned long long *reward_q24;    // [nS][nA], two's complement
    unsigned long long *unsafe;        // [nS][nA]
    unsigned long long *cell_next;     // [C][S][A][S], cellular only
    uint32_t n_states, n_actions;      // nS, nA of the joint tables
    // gc_collect_counts_grouped (appended): every table has a leading [n_groups] dimension and env e adds into group
    // g = min(table_of_env[e], n_groups - 1) of the policy stack's map (RolloutIO), at g times the table's size.
    // n_groups = 0: ungrouped.  n_groups times each counted table's size is at most 2^31, so the offsets are 32-bit.
    uint32_t n_groups;
    uint32_t sa_stride, cell_stride;   // nS nA (the 'next' table's group size is sa_stride * nS), C S A S
};

// Constant tables of the cellular family, passed by value as a __grid_constant__ parameter and
// staged into shared memory once per block.
struct CellTables {
    uint32_t sa[GC_TBL];             // bits 0-3 move, 4-7 noisy, 8 draws
    float    reward[GC_TBL];
    float    reward_noisy[GC_TBL];   // reward when the draw fired (== reward unless it depends on the next level)
    uint8_t  se[GC_MAX_CELLS][GC_TBL]; // [j][s0' * GC_LVL_PAD + s'_p]
    uint32_t place[GC_MAX_CELLS];    // mixed-radix place values S^c (mod 2^32)
    uint32_t place4[4];              // S^0..S^3: digits of four cells folded into one byte (fast path)
    uint32_t unsafe_rows;            // byte s0': set of levels x with SE[j>=2][s0'][x] == unsafe (fast path)
    int8_t   init[GC_MAX_CELLS];
    uint32_t init_index;
    uint32_t counted_mask;           // bit l set: level l counts towards the incidence
    int32_t  n_cells, n_states, n_actions;
    int32_t  reward_log2;
    unsigned long long noise_thr;    // draw fires iff word < noise_thr  (word*2^-32 < p)
    uint32_t noise_thr_m1;           // noise_thr - 1 (32-bit compare: fires iff thr != 0 and word <= thr - 1)
    uint32_t noise_thr_nz;
    // wide envs (more than GC_NARROW_CELLS cells): one 16-bit HALF of a Philox block per cell (eight cells per
    // block), the low 16 bits of the draw only on a tie of that half with the threshold's top half
    // (gc_device.cuh: fire_bits_wide)
    uint32_t noise_kk15;             // (k16 & 0x7FFF) * 0x00010001, k16 = top half of the threshold
    uint32_t noise_kmask;            // all ones iff k16 >= 0x8000
    uint32_t noise_kk;               // k16 * 0x00010001
    uint32_t noise_r16;              // low half of the threshold: on a tie the draw fires iff its low 16 bits < r16
    double   noise_prob;             // for the replay path (compares doubles like the reference)
    // packed layout (gc_cell_packed.cu)
    uint32_t init_packed;            // initial state, 2 bits per cell
    // 5..8 levels (gc_cell_pair8.cu): byte s0' = set of levels x with SE[j >= 2][s0'][x] == unsafe
    unsigned long long unsafe_rows8;
    // stochastic variant: bit 8 s0' + s1' = entry 0 or 1 of row 0 of the side-effects matrix is 'unsafe' for (s0', s1')
    unsigned long long unsafe01_rows8;
};

struct GridParams {
    unsigned long long dispersal_thr;
    uint32_t dispersal_thr_m1, dispersal_thr_nz;
    double dispersal_prob;
    const uint32_t *lut;             // GC_GRID_LUT_ENTRIES transition entries, device memory (handle-owned)
};

// Grid-world transition table: entry index = (code_0 + 20 * code_1) * 25 + (a_0 + 5 * a_1)
#define GC_GRID_LUT_ENTRIES (400 * 25)
// largest index the kernels' masked inputs (5-bit codes, 3-bit actions) can form, (31 + 20 * 31) * 25 + 7 + 5 * 7,
// rounded up: the device table and its shared-memory copy are this long (zero padding beyond the 10,000
// entries), so that out-of-range inputs -- never produced by the kernels -- read padding, not foreign memory
#define GC_GRID_LUT_ALLOC (((31 + 20 * 31) * 25 + 42 + 1 + 3) / 4 * 4)
// entry layout: byte 0 next code_0, byte 1 next code_1, bits 16-17 reward (trees that died),
// bits 18-19 barren jurisdictions before the step, bit 20 / 21 row-0 side effects [0][0] / [0][1]
// == 'safe', bit 22 the action names no position although an agent exists (reference: KeyError)
void gc_build_grid_lut(uint32_t *lut);
void gc_build_pair_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut,
                       uint32_t *unsafe_rows);

cudaError_t gc_launch_cell_step(const CellTables &tab, const StepIO &io, int rng_mode, int n_sm,
                                cudaStream_t stream);
// fast path (S, A <= 4): lut = 1024 pair entries [fire_d][fire_c][s_c | a_c<<2 | s_d<<4 | a_d<<6] followed
// by 32 single-cell entries [fire][s | a<<2], device memory
#define GC_PAIR_LUT_PAIRS 1024
#define GC_PAIR_LUT_ENTRIES (GC_PAIR_LUT_PAIRS + 32)
cudaError_t gc_launch_cell_pair_step(const CellTables &tab, const StepIO &io, const uint2 *lut, int rng_mode,
                                     int n_sm, cudaStream_t stream);
cudaError_t gc_launch_grid_many(const GridParams &gp, const ManyIO &mio, int n_sm, cudaStream_t stream);
cudaError_t gc_launch_cell_pair_many(const CellTables &tab, const ManyIO &mio, const uint2 *lut, int rng_mode, int n_sm,
                                     cudaStream_t stream);
// 5..8 levels / actions (gc_cell_pair8.cu): 4096 pair entries [a_d][s_d][a_c][s_c] (3-bit digits, no noise)
// followed by 128 single-cell entries [fire][a][s]
#define GC_PAIR8_PAIRS 4096
#define GC_PAIR8_ENTRIES (GC_PAIR8_PAIRS + 128)
void gc_build_pair8_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut, unsigned long long *unsafe_rows8,
                        unsigned long long *unsafe01_rows8);
cudaError_t gc_launch_cell_pair8_step(const CellTables &tab, const StepIO &io, const uint2 *lut, int rng_mode, int n_sm,
                                      cudaStream_t stream);
// packed layout: lut = GC_PAIR_LUT_ENTRIES entries in the packed index order (gc_build_packed_lut)
void gc_build_packed_lut(const gc_cell_tables *t, int C, int S, int A, bool noise, uint2 *lut);
cudaError_t gc_launch_cell_packed_step(const CellTables &tab, const PackedIO &io, const uint2 *lut, bool noise,
                                       int n_sm, cudaStream_t stream);
cudaError_t gc_launch_cell_packed_many(const CellTables &tab, const PackedManyIO &mio, const uint2 *lut, bool noise, int n_sm,
                                       cudaStream_t stream);
cudaError_t gc_launch_reset_packed(uint32_t init_packed, uint32_t init_index, const uint8_t *mask, uint32_t *state,
                                   int32_t *t, uint32_t *index, int64_t n, cudaStream_t stream);
cudaError_t gc_launch_pack(int64_t n, int64_t ld, int n_cells, const int8_t *cells, uint32_t *packed, cudaStream_t stream);
cudaError_t gc_launch_unpack(int64_t n, int64_t ld, int n_cells, const uint32_t *packed, int8_t *cells, cudaStream_t stream);
cudaError_t gc_launch_cell_rollout(const CellTables &tab, const RolloutIO &io, const uint2 *lut, bool noise,
                                   int n_sm, cudaStream_t stream);
cudaError_t gc_launch_grid_rollout(const GridParams &gp, const RolloutIO &io, int n_sm, cudaStream_t stream);
// the same kernels writing the transition record, table policy epsilon-greedy (gc_collect)
cudaError_t gc_launch_cell_collect(const CellTables &tab, const RolloutIO &io, const uint2 *lut, bool noise,
                                   int n_sm, cudaStream_t stream);
cudaError_t gc_launch_grid_collect(const GridParams &gp, const RolloutIO &io, int n_sm, cudaStream_t stream);
// the same kernels adding every transition to the counters of `cnt` (gc_collect_counts)
cudaError_t gc_launch_cell_count(const CellTables &tab, const RolloutIO &io, const CountIO &cnt, const uint2 *lut,
                                 bool noise, int n_sm, cudaStream_t stream);
cudaError_t gc_launch_grid_count(const GridParams &gp, const RolloutIO &io, const CountIO &cnt, int n_sm, cudaStream_t stream);
cudaError_t gc_launch_grid_step(const GridParams &gp, const StepIO &io, int rng_mode, int n_sm,
                                cudaStream_t stream);
cudaError_t gc_launch_reset(int n_cells, const int8_t *init, uint32_t init_index, const uint8_t *mask,
                            int8_t *state, int32_t *t, uint32_t *index, int64_t n, int64_t ld,
                            cudaStream_t stream);
cudaError_t gc_launch_encode_mixed(int64_t n, int64_t ld, int n_cells, const int32_t *radix, const int32_t *min,
                                   const int8_t *cells, uint32_t *index, cudaStream_t stream);
cudaError_t gc_launch_decode_mixed(int64_t n, int64_t ld, int n_cells, const int32_t *radix, const int32_t *min,
                                   const uint32_t *index, int8_t *cells, cudaStream_t stream);
cudaError_t gc_launch_tick(uint32_t *d_step, uint32_t inc, cudaStream_t stream);
cudaError_t gc_launch_encode(int64_t n, int64_t ld, int n_cells, uint32_t radix, const int8_t *cells,
                             uint32_t *index, cudaStream_t stream);
cudaError_t gc_launch_decode(int64_t n, int64_t ld, int n_cells, uint32_t radix, const uint32_t *index,
                             int8_t *cells, cudaStream_t stream);
