/*
 * dpb200.h — C ABI of the B200-native policy-iteration engine (libdpb200.so).
 *
 * This is the drop-in boundary for the hot path of
 * nicoRomeroCuruchet/DynamicProgramming, src/cuda_policy_iteration.py.  The
 * reference has no FFI of its own (its plugin boundary is a Python ABC plus a
 * CUDA source string handed to cupy.RawModule); every entry point below cites
 * the reference method (file:line, relative to the reference root) it replaces.
 * A Python host binds these with ctypes (dynamicprogramming_b200/_ffi.py);
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every function returns an int status: PI_OK (0) or a PI_ERR_* class;
 *     pi_last_error() returns a thread-local message (incl. the NVRTC log).
 *   - plain pointers and sizes only; host buffers are caller-owned; the engine
 *     owns all device memory, its stream, graphs and (multi-GPU) communicator.
 *   - one caller thread per engine handle (same as the reference object).
 *   - there is NO CPU fallback: without a CUDA device pi_create fails.
 */
#ifndef DPB200_H
#define DPB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PI_MAX_DIMS 6
#define PI_ABI_VERSION 1

enum {
    PI_OK = 0,
    PI_ERR_INVALID = 1,   /* bad argument / wrong call order              */
    PI_ERR_CUDA = 2,      /* CUDA runtime / driver failure                */
    PI_ERR_COMPILE = 3,   /* NVRTC rejected the dynamics source           */
    PI_ERR_COMM = 4,      /* NCCL failure                                 */
    PI_ERR_NO_DEVICE = 5  /* no usable CUDA device                        */
};

/* Row sentinels stored in the base-index word of a transition row. */
#define PI_ROW_TERMINATED (-1) /* step_dynamics set *terminated: sum w*V := 0   */
#define PI_ROW_ABSORBING (-2)  /* state is in the terminal mask: new_V := V     */

typedef struct pi_engine pi_engine;

/* Regular grid. Replaces bins_space + _precompute_grid_metadata
 * (src/cuda_policy_iteration.py:81-109, :480-514, :894-937): dim 0 is the
 * slowest, dim n_dims-1 has stride 1; lo/hi are the float32 min/max of each
 * axis; axes[d] points to shape[d] float32 node coordinates (bit-identical to
 * the columns of the reference's states_space). */
typedef struct pi_grid {
    int32_t n_dims;
    int32_t shape[PI_MAX_DIMS];
    float lo[PI_MAX_DIMS];
    float hi[PI_MAX_DIMS];
    const float* axes[PI_MAX_DIMS];
} pi_grid;

/* Mirrors CudaPIConfig (src/cuda_policy_iteration.py:36-43) plus the
 * hard-coded SYNC_INTERVAL = 25 of policy_evaluation (:303). */
typedef struct pi_config {
    float gamma;
    float theta;
    int32_t max_eval_iter;
    int32_t max_pi_iter;
    int32_t log_interval;
    int32_t sync_interval; /* 0 -> 25 */
} pi_config;

/* State-range sharding over the GPUs of one box (new; the reference is
 * single-GPU).  Rank r owns flat states [r*N/world, (r+1)*N/world). */
typedef struct pi_shard {
    int32_t rank;
    int32_t world_size;
    uint8_t nccl_id[128]; /* ncclUniqueId bytes from rank 0; ignored if world_size==1 */
} pi_shard;

typedef struct pi_stats {
    int32_t pi_iterations;    /* outer iterations executed                      */
    int32_t converged;        /* 1 if the policy became stable                  */
    int64_t eval_sweeps;      /* total evaluation sweeps                        */
    float last_delta;         /* last residual read at a sync point             */
    int64_t last_changed;     /* states whose action changed in the last improve*/
    double build_ms;          /* device time of the transition-table build      */
    double eval_ms;           /* device time inside evaluation sweeps           */
    double improve_ms;        /* device time inside improvement passes          */
} pi_stats;

/* Log callback: level 0=debug 1=info 2=success 3=warning (loguru levels used
 * by the reference, src/cuda_policy_iteration.py:106,:328-335,:360-368). */
typedef void (*pi_log_fn)(int level, const char* msg, void* user);

const char* pi_last_error(void);
int pi_abi_version(void);

/* Number of visible CUDA devices (0 when there is no driver). */
int pi_device_count(void);

/* Run-time compiles (the plugin's table builder, the grid-specialised sweeps) are cached on disk as
 * cubins keyed by NVRTC version + options + source text: $DPB200_CACHE_DIR, else
 * $XDG_CACHE_HOME/dpb200, else ~/.cache/dpb200; DPB200_CACHE=off disables.  Counters of this
 * process: NVRTC compilations actually run / compilations answered from the cache. */
int pi_nvrtc_counters(int64_t* compiles, int64_t* cache_hits);

/* Compile-only check of a plugin's dynamics source against the table-builder
 * template (NVRTC, sm_100a); needs no GPU.  Errors carry the NVRTC log — the
 * analogue of cupy's CompileException at src/cuda_policy_iteration.py:289. */
int pi_compile_check(const char* dynamics_src, int32_t n_dims, int64_t* cubin_bytes);
/* The same compile, checked for the recompute-mode kernels of the builder program (pi_improve_recompute,
 * pi_policy_rows; see pi_table_mode); needs no GPU.  Errors carry the NVRTC log. */
int pi_recompute_compile_check(const char* dynamics_src, int32_t n_dims, int64_t* cubin_bytes);

/* ncclGetUniqueId for pi_shard.nccl_id: rank 0 calls it and ships the 128 bytes
 * to the other ranks through its own process group (torch.distributed). */
int pi_nccl_unique_id(uint8_t out[128]);

/* __init__ + _allocate_tensors_and_compile (src/cuda_policy_iteration.py:65-91,
 * :142-175, :288-296).  `dynamics_src` is the string returned by the plugin's
 * _dynamics_cuda_src() (:113-125, :518-530, :941-954); it is compiled by NVRTC
 * (default options, like cupy.RawModule) into the transition-table builder.
 * policy := 0, V := 0.  `shard` may be NULL (single GPU).
 *
 * Table mode (N7), read from DPB200_TABLE = auto | full | recompute here (any other value: PI_ERR_INVALID) and kept
 * for the engine's life, pi_retrain and pooled reuse included:
 *   full       the all-action table (A rows per state) is allocated and built once; the improvement pass reads it.
 *   recompute  no table is allocated: wherever the table was read (improvement, policy rows, pi_expand_rows, the
 *              sharded exchange plan) the rows are recomputed on the device by the builder's own code.  Results are
 *              bit-identical to full mode; only memory and time differ.
 *   auto       full when the table plus the engine's other buffers plus a fixed reserve fit the free device
 *              memory (cudaMemGetInfo) and the table's allocation succeeds, else recompute.  Each rank of a sharded
 *              engine decides for its own slice. */
int pi_create(const pi_grid* grid, const float* actions, int32_t n_actions,
              const pi_config* config, const char* dynamics_src, int32_t device,
              const pi_shard* shard, pi_engine** out);

void pi_destroy(pi_engine* e);

int pi_set_log(pi_engine* e, pi_log_fn fn, void* user);

/* Terminal mask + initial value: d_terminal_mask, V[mask] = value, new_V = V
 * (src/cuda_policy_iteration.py:156-161).  `mask` has n_states bytes (global). */
int pi_set_terminal(pi_engine* e, const uint8_t* mask, float value);

/* V[mask] = value on both buffers without touching the terminal mask — the
 * overhead-crane goal initialisation (runners/overhead_crane_cuda.py:193-206). */
int pi_set_values(pi_engine* e, const uint8_t* mask, float value);

/* The same on ONE buffer: which = 0 -> d_value_function, 1 -> d_new_value_function.  What a
 * boolean-mask store `self.d_value_function[d_mask] = value` of a reference subclass does
 * (runners/overhead_crane_cuda.py:201-202); `mask` is in reference order, n_states bytes. */
int pi_set_values_buffer(pi_engine* e, int32_t which, const uint8_t* mask, float value);

/* Transition-table build (new stage; arithmetic oracle = step_dynamics +
 * get_barycentric_{2,4,6}d, src/cuda_policy_iteration.py:183-210, :580-614,
 * :1007-1042).  One compact row per (state, action): base flat index,
 * n_dims interpolation fractions, reward.  Must follow pi_set_terminal.  Recompute mode: only the rows of the
 * current policy are built (pi_stats.build_ms is their device time). */
int pi_build_table(pi_engine* e);

/* N4 — a persistent engine across autoresearch trials (runners/trial_runner.sh:33-60 starts a new Python process per trial;
 * only the dynamics / reward text of runners/double_cartpole_swingup_cuda.py changes between trials).  pi_retrain puts
 * the engine back into its freshly constructed state — V := 0, policy := 0, the given terminal mask / value (NULL: none) —
 * and rebuilds the transition table, recompiling the builder only when `dynamics_src` differs from the text it was built
 * from (*recompiled).  Everything that does not depend on the dynamics is kept: CUDA context, buffers, storage order,
 * the JIT-compiled sweep kernels, CUDA graphs, the NCCL communicator and the peer mappings.  Equivalent to
 * pi_destroy + pi_create + pi_set_terminal + pi_build_table for the same grid, bit for bit.  The table mode is kept;
 * in recompute mode only the policy-0 rows are rebuilt. */
int pi_retrain(pi_engine* e, const char* dynamics_src, const uint8_t* terminal_mask, float terminal_value, int32_t* recompiled);

/* policy_evaluation() (src/cuda_policy_iteration.py:300-336): Jacobi sweeps,
 * residual read every sync_interval sweeps, returns at the first sync sweep
 * with delta < theta.  *delta = value the reference would return; *sweeps =
 * number of sweeps executed. */
int pi_evaluate(pi_engine* e, float* delta, int32_t* sweeps);

/* policy_improvement() (src/cuda_policy_iteration.py:338-355): greedy argmax,
 * strict '>' from -1e30f so the lowest action index wins ties; *stable = 1 iff
 * no state changed its action.  Recompute mode: every (state, action) row is recomputed from the dynamics in this
 * pass, with the same result; pi_stats.improve_ms includes that work. */
int pi_improve(pi_engine* e, int32_t* stable, int64_t* n_changed);

/* run() (src/cuda_policy_iteration.py:357-370) without the final D2H. */
int pi_run(pi_engine* e, pi_stats* stats);

/* _pull_tensors_from_gpu (src/cuda_policy_iteration.py:372-388): global V and
 * policy (n_states each) to host.  Multi-GPU: collective, every rank gets all. */
int pi_copy_results(pi_engine* e, float* value_function, int32_t* policy);

/* This rank's slice only (internal states [pi_local_begin, pi_local_end), in the
 * engine's storage order, see pi_layout); no collective. */
int pi_copy_local_results(pi_engine* e, float* value_function_local, int32_t* policy_local);

/* Host <-> device hand-off used by the end-to-end evaluation call and tests. */
int pi_upload_policy(pi_engine* e, const int32_t* policy);     /* n_states  */
int pi_upload_values(pi_engine* e, const float* value_function); /* n_states */
/* This rank's slice of the policy only, in the engine's storage order (the layout
 * pi_copy_local_results returns): n_local int32; no collective, no full-grid staging. */
int pi_upload_policy_local(pi_engine* e, const int32_t* policy_local);

/* Exactly `n_sweeps` evaluation sweeps with no convergence test (steady-state
 * timing); *delta = residual of the last sweep, *device_ms = CUDA-event time. */
int pi_sweeps(pi_engine* e, int32_t n_sweeps, float* delta, float* device_ms);

/* Expand compact rows into the reference's 2^D corner form for parity checks:
 * for `count` states starting at global state `s_begin` (must lie in this
 * rank's range) and action `action`, writes idx[count][C], w[count][C],
 * reward[count], terminated[count] exactly as step_dynamics +
 * get_barycentric_Nd would produce them (corner c, bit d <-> dim d for
 * D=4,6; the 2-D corner order of :201-209 for D=2).  Any output may be NULL.  Recompute mode: the action's rows of
 * this rank's slice are recomputed into a temporary buffer first (same bits as the table). */
int pi_expand_rows(pi_engine* e, int32_t action, int64_t s_begin, int64_t count,
                   int32_t* idx, float* w, float* reward, uint8_t* terminated);

/* Raw device pointers for torch/__cuda_array_interface__ hand-off
 * (d_value_function, d_policy, ... of the reference object). */
int pi_device_ptrs(pi_engine* e, void** value_function, void** new_value_function,
                   void** policy, void** terminal_mask);

/* Internal storage order (DESIGN.md §3).  The engine may store states with a
 * different dimension fastest than the reference does (chosen by a build-time
 * probe of gather coalescing; DPB200_FAST_DIM=ref|auto|<dim> overrides).  Every
 * host-facing call above takes and returns REFERENCE order; only the raw
 * device pointers and pi_copy_local_results expose the internal order.
 * perm[k] = logical dimension stored at position k (0 = slowest);
 * probe_lines[d] = measured 128-byte lines per warp gather with d fastest. */
int pi_layout(const pi_engine* e, int32_t* fast_dim, int32_t perm[PI_MAX_DIMS],
              double probe_lines[PI_MAX_DIMS]);

/* Geometry queries. */
int64_t pi_n_states(const pi_engine* e);
int64_t pi_local_begin(const pi_engine* e);
int64_t pi_local_end(const pi_engine* e);
/* Device bytes of the all-action table plus the policy's rows; 0 in recompute mode (no table). */
int64_t pi_table_bytes(const pi_engine* e);
/* 0 = full table, 1 = recompute (see pi_create). */
int32_t pi_table_mode(const pi_engine* e);
/* Number of kernel launches issued by this engine so far (bench bookkeeping). */
int64_t pi_launch_count(const pi_engine* e);
/* Last-stage device timings in ms (build, eval, improve).  Recompute mode: build_ms is the device time of the current
 * policy's rows, improve_ms includes recomputing every row. */
int pi_get_stats(const pi_engine* e, pi_stats* stats);

/* Evaluation-sweep kernel selection (new; no reference counterpart).  At pi_build_table the
 * engine times its scalar gather sweep against the x-line sweep (csrc/xline_sweep_src.cuh:
 * K consecutive states of the fast-stored dimension per thread, vector window loads, packed
 * fp32 arithmetic, tile-ordered rows; JIT-compiled with the grid geometry as constants) on
 * the freshly built rows and keeps the faster one; both produce bit-identical V.
 * DPB200_XLINE = off | auto | [force:]K,LV,PF,warps,minb[,roll]:T0,T1,..[;more] overrides.
 * pi_eval_kernel_info returns 1 (x-line) / 0 (scalar), a description and the probe timings. */
int pi_eval_kernel_info(const pi_engine* e, char* buf, int32_t buf_len, double* ms_scalar, double* ms_selected);
/* Compile-only check of a JIT sweep for a synthetic bins^n_dims grid; needs no GPU.
 * cfg: an x-line configuration, or "pair:<threads>,<minb>" for the packed-pair sweep. */
int pi_xline_compile_check(int32_t n_dims, int32_t bins, const char* cfg, int64_t* cubin_bytes);
/* Test hook: x-line sweep `cfg` vs the scalar sweep on the current rows and V (bitwise
 * comparison + timings); info = {registers, grid, block, tiles}; engine state unchanged. */
int pi_debug_xline(pi_engine* e, const char* cfg, int32_t iters, float* ms_xline, float* ms_scalar,
                   int64_t* mismatches, double* window_fraction, int32_t* info);

/* Test hook for the plane-staged sweep (csrc/plane_sweep_src.cuh: V read from shared memory, V-planes staged by TMA
 * bulk copies after a per-policy plan, csrc/plane_plan.cuh): compiles configuration `cfg` = "NS,L,minb,lv,pack"
 * (slots, state-planes per chunk, CTAs per SM, lean weight-tree levels; pack: 0 one state per thread, 1 the same with a
 * packed f32x2 weight tree, 2 item mode = two states per thread, regular pairs share loads; NS / L 0 = default),
 * plans the current rows, runs it and the engine's currently selected kernel `iters` times on the current rows and V
 * and counts differing words (must be 0).  stats = {plane loads, late loads, cells per state-plane, fraction of states
 * not staged, regular pairs per state-plane, items outside their bank-aligned lane, single states on the pair path (item mode)} — SEVEN doubles; info = {registers, grid, block, shared-memory
 * bytes, slots, chunk}.  Engine state unchanged. */
int pi_debug_plane(pi_engine* e, const char* cfg, int32_t iters, float* ms_plane, float* ms_base, int64_t* mismatches,
                   double* stats, int32_t* info);

/* Test hook: as pi_debug_plane, with the plan stitched for the chunk rotation `rot` (-1: the engine's own, 0 on one GPU),
 * and the schedule and plan it ran.  sched = {state-planes, chunks, grid, rotation, slots, slot pitch in floats, outer
 * corners per cell, bytes per plan record} — EIGHT int32; chunk_begin (>= chunks + 1 entries, or null) = first state-plane
 * of every chunk and the end; records (or null) = the plan records of every local state-plane, as the sweep reads them.
 * CTA b of the sweep takes the chunks (b + rot) mod chunks, (b + grid + rot) mod chunks, ... */
int pi_debug_plane_schedule(pi_engine* e, const char* cfg, int32_t rot, int32_t iters, int64_t* mismatches, double* stats,
                            int32_t* sched, int32_t* chunk_begin, int64_t chunk_cap, void* records, int64_t record_cap);

/* Test hook for the JIT sweeps of csrc/pair_sweep_src.cuh (grid strides as immediates): compiles the
 * configuration (threads per block, blocks per SM, lean weight-tree levels 1..3, gathers per explicitly
 * scheduled group or 0, single = 1: one state per thread / 0: two states per thread with packed f32x2
 * math), runs it and the scalar sweep `iters` times on the current rows and V, and counts differing words
 * of the result (must be 0). */
int pi_debug_pair(pi_engine* e, int32_t threads, int32_t minb, int32_t lv, int32_t group, int32_t single, int32_t iters,
                  float* ms_pair, float* ms_scalar, int64_t* mismatches, int32_t* regs);

/* N2: batched policy lookup with get_optimal_action semantics — action(p) = sum_c lambda_c(p) *
 * action_space[policy[idx_c(p)]] (utils/barycentric.py:76-108; weights and indices as
 * get_barycentric_weights_and_indices computes them, :11-73, in the arithmetic numba gives
 * them: float32 step / cell, float64 t and weight products, corner_bits order).  One CUDA thread
 * per query point; used by closed-loop rollouts (every runner's evaluate(), e.g.
 * runners/pendulum_cuda.py:161-166) to query thousands of states per call.
 * points: n_points x n_dims float32 (host); out: n_points float32 (host). */
int pi_lookup_actions(pi_engine* e, const float* points, int64_t n_points, float* out);

/* N6: warm start from another grid's value function (new; the reference has no counterpart — every run of it starts
 * from V = 0, policy = 0, src/cuda_policy_iteration.py:142-175).  Enables solving at a coarse --bins first (the
 * autoresearch loop trains and scores at --bins 12, runners/trial_runner.sh) and starting the fine solve from that V.
 * For every state of this rank's slice that is not absorbing (terminal mask), both V buffers get the source value
 * function interpolated at the state's node (grid->axes bits) with the arithmetic of pi_lookup_actions: the node is
 * clamped to the source box, the source grid is taken as uniform from source->lo / hi / shape (source->axes is not
 * used), float64 fractions and weight products, corner_bits order, float32 sum in ascending corner order.  Absorbing
 * states keep the value they hold (pi_set_terminal / pi_set_values).  `source_values` has prod(source->shape) floats in
 * reference order.  *device_ms (may be NULL) = CUDA-event time of the prolongation kernel.  Sharded engines: collective;
 * every rank computes its slice and the full V is all-gathered.  PI_ERR_INVALID for a null pointer, a different n_dims,
 * a source shape[d] < 2, lo[d] >= hi[d] or a call before pi_build_table; the engine stays usable.
 * The policy is not touched: pi_improve afterwards makes it greedy with respect to the prolonged V (and re-compacts the
 * rows, re-plans and reselects the sweep kernel); its `stable` / n_changed then compare with the policy held before the
 * warm start, not with a converged one, and mean nothing for convergence. */
int pi_prolong_values(pi_engine* e, const pi_grid* source, const float* source_values, float* device_ms);

/* The same lookup for a SAVED policy (Cls.load(path), src/cuda_policy_iteration.py:411-432;
 * runners/hybrid_double_cartpole.py:35-43): the policy table (reference order, n_states int32)
 * and the action values are uploaded once, queries are batched.  grid->axes is not used. */
typedef struct pi_lookup pi_lookup;
int pi_lookup_create(const pi_grid* grid, const int32_t* policy, const float* actions, int32_t n_actions,
                     int32_t device, pi_lookup** out);
int pi_lookup_query(pi_lookup* lookup, const float* points, int64_t n_points, float* out);
void pi_lookup_destroy(pi_lookup* lookup);

/* N5: closed-loop policy rollouts on the device.  Replaces the loop of every runner's evaluate() — get_optimal_action
 * (utils/barycentric.py:76-108) followed by one environment step, once per simulated step on one CPU thread (e.g.
 * runners/pendulum_cuda.py:161-166) — simulated with the plugin's own step_dynamics, compiled by NVRTC with the table
 * builder's options (csrc/rollout_src.cuh).  One CUDA thread runs one whole episode:
 *   x_0 = initial_states[e]; for t = 0..n_steps-1 until terminated:
 *     a_t = the pi_lookup_query action at x_t (query clamped to the grid; x_t itself is never clamped or wrapped);
 *     step_dynamics(x_t, a_t, &x_{t+1}, &r_t, &term_t);
 *     total += (double)r_t;  ret += disc * (double)r_t;  disc *= gamma   (float64, disc starts at 1, no contraction);
 *     length = t + 1; terminated = term_t.
 * Episodes end only when step_dynamics sets *terminated; the terminal mask is not consulted.
 *
 * pi_rollout_create: the policy (reference order, n_states int32, validated like pi_lookup_create) and the action
 * values are uploaded once; grid->axes is not used.  `dynamics_src` is the plugin's _dynamics_cuda_src() text
 * (src/cuda_policy_iteration.py:113-125, :518-530, :941-954); errors as pi_create (PI_ERR_COMPILE with the NVRTC log,
 * PI_ERR_NO_DEVICE: there is no CPU fallback). */
typedef struct pi_rollout pi_rollout;
int pi_rollout_create(const pi_grid* grid, const int32_t* policy, const float* actions, int32_t n_actions,
                      const char* dynamics_src, int32_t device, pi_rollout** out);
/* Host buffers, episode-major: initial_states / final_states n_episodes x D float32 (final = x_length);
 * total_reward, discounted_return (f64), length (i32), terminated (u8) n_episodes each.  traj_*: all three or NULL;
 * traj_states n x (n_steps+1) x D, traj_actions and traj_rewards n x n_steps, NaN after each episode's length.
 * n_episodes == 0 and n_steps == 0 are valid; n_steps < 0 is PI_ERR_INVALID. */
int pi_rollout_run(pi_rollout* r, const float* initial_states, int64_t n_episodes, int32_t n_steps, double gamma,
                   double* total_reward, double* discounted_return, int32_t* length, uint8_t* terminated,
                   float* final_states, float* traj_states, float* traj_actions, float* traj_rewards);
/* One step_dynamics call per (states[i], actions[i]) pair — the environment step of evaluate() alone (n x D states,
 * n actions in; n x D next states, n rewards, n terminated flags out). */
int pi_rollout_step(pi_rollout* r, const float* states, const float* actions, int64_t n,
                    float* next_states, float* rewards, uint8_t* terminated);
void pi_rollout_destroy(pi_rollout* r);
/* Compile-only check of a plugin's dynamics source against the rollout kernels (NVRTC, sm_100a); needs no GPU. */
int pi_rollout_compile_check(const char* dynamics_src, int32_t n_dims, int64_t* cubin_bytes);

/* N8: one-step lookahead on a value table (csrc/lookahead_src.cuh).  For a query point x (not clamped or wrapped) and
 * each action index a = 0..A-1:
 *   step_dynamics(x, actions[a], &x', &r, &term);
 *   ev = term ? 0 : the multilinear interpolation of V at x' with the table builder's cell search and the
 *        improvement's corner order and fmaf chain (csrc/row_value_src.cuh: expected_value);
 *   Q[a] = fmaf(gamma, ev, r)   (float32).
 * The chosen action is the improvement's winner: ascending a, strict '>' from -1e30f, lowest index on ties, NaN never
 * wins, action 0 when nothing beats -1e30f.  The terminal mask is not consulted.  At a non-absorbing grid node, with the
 * values the improvement pass reads, the winner is the action pi_improve writes there.
 *
 * pi_rollout_set_values: the value table V, n_states float32 in reference order (a saved .npz's value_function),
 * uploaded once and replaced by each call; every bit pattern is accepted. */
int pi_rollout_set_values(pi_rollout* r, const float* values);
/* Host buffers: points n x D float32; best_action n int32 and q n x n_actions float32 (row-major), either may be NULL.
 * n == 0 is valid.  PI_ERR_INVALID for a null handle or points, n < 0, or before pi_rollout_set_values. */
int pi_rollout_lookahead(pi_rollout* r, const float* points, int64_t n, float gamma, int32_t* best_action, float* q);
/* pi_rollout_run with the lookahead as the controller: a_t = actions[winner at x_t] with Q under (float)gamma; the
 * step, the returns (discounted with gamma), the buffers and the error rules are those of pi_rollout_run, and it is
 * PI_ERR_INVALID before pi_rollout_set_values. */
int pi_rollout_run_lookahead(pi_rollout* r, const float* initial_states, int64_t n_episodes, int32_t n_steps,
                             double gamma, double* total_reward, double* discounted_return, int32_t* length,
                             uint8_t* terminated, float* final_states, float* traj_states, float* traj_actions,
                             float* traj_rewards);

#ifdef __cplusplus
}
#endif
#endif /* DPB200_H */
