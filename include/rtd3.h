/*
 * rtd3.h - C ABI of librtd3.so: the B200 (sm_100a) hot path of
 * benmcclusky/Residual-TD3-Robot-Navigation.
 *
 * The reference has no FFI of its own (it is pure Python); the functions below are what a
 * ctypes binding placed under the reference's `Environment` / `Robot` / `TD3` / `ReplayBuffer`
 * classes calls.  Each entry point cites the reference interface it replaces (file:line under
 * the reference repo root).  See INTEGRATION.md for the binding stubs.
 *
 * Conventions
 *   - every function returns int32_t: 0 = ok, >0 = cudaError_t, <0 = argument error;
 *     rtd3_last_error() returns a thread-local, NUL-terminated message for the last failure;
 *   - unless a parameter is marked HOST, pointers are DEVICE pointers owned by the caller
 *     (torch tensors); the library never frees user buffers;
 *   - launching entry points take an explicit cudaStream_t (as void*), never synchronise it
 *     and never allocate on it;
 *   - environment-indexed arrays are struct-of-arrays: x[n], y[n] ... ; a "[k][n]" array is k
 *     planes of n elements (plane-major) so that consecutive envs are consecutive in memory;
 *   - sizes are int64_t; handles are per-device and not re-entrant (one host thread per handle).
 */
#ifndef RTD3_H_
#define RTD3_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTD3_VERSION 100
#define RTD3_WORLD_SIZE 100          /* constants.py:6  */
#define RTD3_MAP_CELLS 10000         /* 100 x 100 cells, indexed [x][y] (environment.py:105-111) */
#define RTD3_MT_N 624                /* MT19937 state words */
#define RTD3_DEMO_GRID 100           /* candidate lists of the nearest-demonstration search (rtd3_demo_lists): 100 x 100 cells ... */
#define RTD3_DEMO_CELL 1.0           /* ... of side 1, the world's own cells; queries outside [0,100)^2 sweep the whole set */
#define RTD3_ENV_DEMO_CELLS 625      /* per-env demonstration sets: 25 x 25 grid of 4 x 4 cells (rtd3_robot_process_demonstration) */

#define RTD3_ERR_ARG (-1)
#define RTD3_ERR_STATE (-2)

int32_t rtd3_version(void);
const char* rtd3_last_error(void);
/* Number of kernels this library has launched since load / since the last reset (bench.py's gpu_launches). */
int64_t rtd3_launch_count(void);
void rtd3_launch_count_reset(void);
/* Replaying a captured CUDA graph launches kernels without passing through the library: the owner of the graph adds them here. */
void rtd3_launch_count_add(int64_t n);

/* ------------------------------------------------------------------------------------------------
 * Environment: dynamics / step / rollout        (environment.py:98-127)
 * ---------------------------------------------------------------------------------------------- */
typedef struct rtd3_env rtd3_env;

/* Per-device handle; owns the packed dynamics table (speed*cos(rot), speed*sin(rot)) in HBM. */
int32_t rtd3_env_create(rtd3_env** out, int32_t device);
int32_t rtd3_env_destroy(rtd3_env* h);

/* Replaces assigning Environment.dynamics_speed / dynamics_angle (environment.py:20-21, 84, 95).
 * speed, angle: DEVICE float32 [100*100], row-major [x][y].  Builds the packed table on `stream`:
 * rot = float32(angle*2*pi) (float32 as numpy>=2 evaluates environment.py:107), then
 * (speed*cos(rot), speed*sin(rot)) evaluated in float64 and rounded once to float32.
 * The same as rtd3_env_set_maps with K = 1 followed by clearing the map index: every env steps on this map. */
int32_t rtd3_env_set_map(rtd3_env* h, const float* speed, const float* angle, void* stream);

/* Map bank: a handle holds K maps and, optionally, a map index of length m.  Env v of ANY launch (step, dynamics, rollout,
 * rollout_host, tick, the planner's P*n virtual envs v = p*n + i) steps on map index[v % m]; with no index every env steps on
 * map 0 and every launch runs the single-map kernels.  Kernels clamp an index entry to [0, K), so a bad entry never reads
 * outside the bank (validating it is the caller's job).  A bank costs about 188 KB of HBM per map.
 *
 * rtd3_env_set_maps: speed, angle DEVICE float32 [K][100*100]; builds the K tables on `stream`.  Asynchronous while K does not
 * exceed the number of maps already allocated (the handle starts with one); a larger K reallocates the bank, which synchronises
 * the device and drops the graphs cached by rtd3_env_rollout_host.  The index is kept as it is.
 *
 * rtd3_env_set_map_index: copies `index` (DEVICE int32 [m]) into the handle with a device-to-device cudaMemcpyAsync on `stream`
 * (asynchronous and capturable while m does not exceed the largest m set before; a captured launch reads the handle's copy, so
 * a graph replayed after an index change of the same length sees the new contents).  index == NULL or m == 0 clears the index.
 *
 * Kernels with an index: rtd3_env_step / rtd3_env_dynamics read the tables through the read-only path whatever the variant
 * (RTD3_STEP_SMEM falls back to RTD3_STEP_LDG: a CTA covers envs of many maps, there is no one table to stage); the rollout
 * kernels stage the map of a CTA's first env, and a warp whose envs all use that map runs the single-map loop, while any other
 * warp reads every lane's table from global memory, which is several times slower (DESIGN.md section 3).  Keep the envs of one
 * map in contiguous blocks that cover whole CTAs to stay on the fast path: 32 envs up to 4 736 envs per launch, 64 up to 9 472,
 * 256 above. */
int32_t rtd3_env_set_maps(rtd3_env* h, const float* speed, const float* angle, int32_t K, void* stream);
int32_t rtd3_env_set_map_index(rtd3_env* h, const int32_t* index, int64_t m, void* stream);

/* Environment.set_dynamics (environment.py:59-95) for K seeds: map k of speed / angle (DEVICE float32 [K][100*100], [x][y])
 * is perlin_maps(seeds[k]) (environment.py of this package) under the exactness rules below.  seeds: DEVICE int64 [K],
 * each in [0, 2^63).  Asynchronous on `stream`, no allocation, no synchronisation, capturable.  K in [1, 65536].
 * Exactness:
 *   - the float32 fields before normalisation (n(5) + 0.5 n(10) + 0.25 n(20) for speed, n(5) for angle, each float64 sum
 *     rounded once to float32) are bit-identical to perlin_maps's;
 *   - angle, their float32 min-max normalisation (c - min) / (max - min), is bit-identical to perlin_maps's;
 *   - speed = 1 / (1 + exp(-10 * (norm - 0.5))) in numpy's float32 operation order, except that exp is evaluated in float64
 *     and rounded once to float32.  numpy's float32 exp is a SIMD routine picked by the host CPU and not correctly rounded, so
 *     speed can differ from perlin_maps's by a few ulp (up to 4 measured); it is the same on every host.
 * A flat field (max == min) gives NaN cells, as in numpy; rtd3_env_set_maps makes them dead cells.  Hand the maps to
 * rtd3_env_set_maps on the same stream to install them without a host round trip. */
int32_t rtd3_perlin_maps(const int64_t* seeds, int32_t K, float* speed, float* angle, void* stream);
/* Test hook: 1 makes rtd3_perlin_maps write the float32 fields before normalisation instead of the maps, 0 (the default)
 * restores the maps. */
void rtd3_perlin_set_raw_fields(int32_t on);
/* The map configuration launches capture as kernel arguments: bank address, index address (NULL without an index), K, m.
 * A caller that captures launches into a CUDA graph compares these to decide whether to recapture.  Any output may be NULL. */
int32_t rtd3_env_map_config(const rtd3_env* h, const void** tables, const void** index, int32_t* num_maps, int64_t* index_len);

/* Variant selector for rtd3_env_step (evidence for each lives in profiles/). */
#define RTD3_STEP_AUTO 0
#define RTD3_STEP_SMEM 1   /* table staged in shared memory by one bulk-async copy per CTA */
#define RTD3_STEP_LDG 2    /* table read through the read-only L1 path */

/* Environment.step over n envs (environment.py:122-127 -> dynamics :98-119).
 * x,y: state in/out; ax,ay: actions (clipped to +-5 inside).  A NaN result keeps the old state. */
int32_t rtd3_env_step(rtd3_env* h, float* x, float* y, const float* ax, const float* ay, int64_t n,
                      int32_t variant, void* stream);

/* Environment.dynamics (pure, environment.py:98-119): out_x,out_y = f(x,y,ax,ay); NaN propagates. */
int32_t rtd3_env_dynamics(rtd3_env* h, const float* x, const float* y, const float* ax, const float* ay,
                          float* out_x, float* out_y, int64_t n, void* stream);

/* T consecutive Environment.step calls in one launch (the loop at robot-learning.py:97-100 with
 * actions supplied): actions [T][2][n] float32, traj (nullable) [T][2][n] receives the state after
 * every step; x,y are updated to the final state.  State lives in registers across the T steps. */
int32_t rtd3_env_rollout(rtd3_env* h, float* x, float* y, const float* actions, float* traj, int64_t n,
                         int64_t T, void* stream);
/* Test hook: 1 forces the cp.async variant of the rollout kernel, 2 the single-warp TMA variant (instead of the
 * warp-pair TMA kernel used for latency-bound batches), 0 restores the automatic choice. */
void rtd3_env_force_plain_rollout(int32_t on);
/* Test hook: 0 launches every rollout kernel with a full dependency on the stream's previous work; 1 (the default) lets a
 * rollout launch start while the previous kernel of the stream drains (programmatic dependent launch: the kernel stages its
 * table before it waits for that kernel, and reads state and actions after).  Launches while the stream is capturing, and the
 * first rollout launch after rtd3_env_set_map(s), always take the full dependency.  Results are the same either way. */
void rtd3_env_set_launch_overlap(int32_t on);

/* rtd3_env_rollout for HOST buffers: actions_host / traj_host are page-locked host memory [T][2][n] (same loop, robot-learning.py:97-100).
 * mode is a bit set - 1: the copy engine stages the actions in HBM, 2: the trajectory goes back through the copy engine; an
 * unstaged direction is read / written by the kernel's TMA tiles across PCIe (0 = both: one plain launch).  With a staged direction
 * the T steps run as `chunks` time slices: copy of slice c+1, kernel of slice c and copy-back of slice c-1 overlap, and the whole
 * pipeline is ONE CUDA graph per (buffers, shape), cached in the handle (staging buffers and up to 16 graphs, freed by
 * rtd3_env_destroy).  Asynchronous on `stream` like every other call; x, y end at the final state. */
int32_t rtd3_env_rollout_host(rtd3_env* h, float* x, float* y, const float* actions_host, float* traj_host, int64_t n,
                              int64_t T, int32_t chunks, int32_t mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * numpy-legacy MT19937 streams, one per env      (robot-learning.py:19; numpy RandomState)
 * ---------------------------------------------------------------------------------------------- */
typedef struct rtd3_mt_bank {
  uint32_t* mt;        /* [624][n] state words, word-major                      */
  int32_t* pos;        /* [n] next word index, 624 = regenerate on next draw    */
  int32_t* has_gauss;  /* [n] legacy_gauss spare flag                           */
  double* gauss;       /* [n] legacy_gauss spare value                          */
  int64_t n;
} rtd3_mt_bank;

/* np.random.seed(seeds[i]) for stream i (mt19937_seed / init_genrand). seeds: DEVICE uint32 [n]. */
int32_t rtd3_mt_seed(const rtd3_mt_bank* bank, const uint32_t* seeds, void* stream);
/* Raw draws for tests: out[k][n] = k-th next uint32 of every stream. */
int32_t rtd3_mt_draw_u32(const rtd3_mt_bank* bank, uint32_t* out, int64_t k, void* stream);
/* np.random.normal(0,1) draws (legacy polar method with spare): out[k][n] float64. */
int32_t rtd3_mt_draw_gauss(const rtd3_mt_bank* bank, double* out, int64_t k, void* stream);
/* The same for the streams i with where[i] == equals only (where: DEVICE int8 [n], e.g. the tick types: the reference draws its
 * exploration noise on 'step' ticks only); the other streams are not advanced and receive zeros.  where == NULL: all streams. */
int32_t rtd3_mt_draw_gauss_where(const rtd3_mt_bank* bank, double* out, int64_t k, const int8_t* where, int32_t equals, void* stream);

/* Environment.set_init_and_goal (environment.py:28-56) for n envs, each on its own stream.
 * goal [2][n] float64, region [4][n] float64 = left,right,bottom,top.  Bit-exact vs numpy. */
int32_t rtd3_env_init_goal_region(const rtd3_mt_bank* bank, double* goal, double* region, void* stream);

/* Environment.reset / get_random_robot_init_state (environment.py:130-137) for the envs whose
 * mask byte is non-zero (mask NULL = all), or - with mask_equals >= 0 - equal to mask_equals (so that the int8 action
 * types of rtd3_robot_next_action_type can be passed as they are: mask_equals = 2 resets the 'reset' envs).  Writes float32 state x,y; if state64 ([2][n] float64)
 * is non-NULL also the reference's float64 draw, which is bit-exact vs numpy. */
int32_t rtd3_env_reset(const rtd3_mt_bank* bank, const double* region, const uint8_t* mask, int32_t mask_equals, float* x,
                       float* y, double* state64, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Replay ring + minibatch sampling           (robot.py:58-124)
 * Device layout (36 B per row): s [cap][2], a [cap][2], r [cap], s2 [cap][2], notdone [cap]  float32.
 * ---------------------------------------------------------------------------------------------- */

/* ReplayBuffer.push (robot.py:79-96) for n transitions given as env planes; rows go to
 * (position + i) % capacity; the caller advances position/size.  done: uint8 [n]. */
int32_t rtd3_replay_push(float* s, float* a, float* r, float* s2, float* notdone, int64_t capacity, int64_t position,
                         const float* sx, const float* sy, const float* ax, const float* ay, const float* reward,
                         const float* nx, const float* ny, const uint8_t* done, int64_t n, void* stream);

/* The gather half of ReplayBuffer.sample (robot.py:113-115): rows idx[b] -> dense minibatch arrays. */
int32_t rtd3_replay_gather(const float* s, const float* a, const float* r, const float* s2, const float* notdone,
                           const int32_t* idx, int32_t batch, float* out_s, float* out_a, float* out_r, float* out_s2,
                           float* out_notdone, void* stream);

/* The index half of ReplayBuffer.sample (robot.py:111): `count` consecutive draws of
 * np.random.choice(n, batch, replace=False) from stream `stream_id` of the bank, bit-exact with numpy's
 * legacy shuffle.  out: int32 [count][batch].  scratch: int32 [count][n] (the swap lists; transient).
 * n <= 56000. */
int32_t rtd3_sample_indices_mt19937(const rtd3_mt_bank* bank, int64_t stream_id, int32_t n, int32_t batch, int32_t count,
                                    int32_t* out, int32_t* scratch, void* stream);

/* Throughput-mode index draw (NOT the reference's stream): count x batch indices uniform in [0, n) WITH
 * replacement from Philox4x32-10(seed, offset).  For replay shards too large for the exact sampler. */
int32_t rtd3_sample_indices_philox(uint64_t seed, uint64_t offset, int64_t n, int32_t batch, int32_t count, int32_t* out,
                                   void* stream);

/* ------------------------------------------------------------------------------------------------
 * Residual-TD3 learner                        (robot.py:128-206 networks, :209-398 TD3)
 * Networks: actor 2->H->..->H->2, critic 4->H->..->H->1 with `layers` hidden layers (reference: H=200, 3).
 * Parameters live in ONE float32 arena owned by the caller:
 *   [actor | critic1 | critic2 | target actor | target critic1 | target critic2]
 * every slot in torch's parameters() order (W1 [H][in], b1, W2 [H][H], b2, ..., Wout [out][H], bout) and
 * padded to a multiple of 4 floats.  grads / adam_m / adam_v cover the first three slots.
 * steps: int32 [2] on the device = Adam step counters {actor optimiser, critic optimisers};
 * beta_pows: float64 [4] on the device = {0.9^t, 0.999^t} per optimiser (initialise to 1.0), advanced together
 * with `steps` by the step calls and read by rtd3_td3_adam_polyak for the bias corrections.
 * scratch: rtd3_td3_scratch_floats(batch) floats of device memory, contents are transient.
 * ---------------------------------------------------------------------------------------------- */
typedef struct rtd3_td3 rtd3_td3;

int32_t rtd3_td3_create(rtd3_td3** out, int32_t device, int32_t hidden, int32_t layers);
int32_t rtd3_td3_destroy(rtd3_td3* h);
/* net: 0 actor, 1 critic1, 2 critic2, 3 target actor, 4 target critic1, 5 target critic2 */
int64_t rtd3_td3_param_count(const rtd3_td3* h, int32_t net);
int64_t rtd3_td3_param_offset(const rtd3_td3* h, int32_t net);
int64_t rtd3_td3_arena_floats(const rtd3_td3* h);
/* floats of row scratch a critic/actor step needs for `batch` rows (layer inputs and pre-activation
 * gradients of the trained networks, from which the weight gradients are reduced). */
int64_t rtd3_td3_scratch_floats(const rtd3_td3* h, int32_t batch);

/* TD3.train_critic minus the optimiser steps (robot.py:326-357/361): gathers rows idx[batch] from the
 * replay ring, target-policy smoothing with the supplied unit-normal noise [batch][2] (robot.py:338-339),
 * clipped double-Q target (robot.py:342-345), both critic forward passes, both MSE losses (added into
 * loss2[0..1], which the caller zeroes) and both backward passes; the parameter gradients of both critics
 * are written to grads (for batch > 512 they are accumulated, so grads must be zero on entry -
 * rtd3_td3_adam_polyak re-zeroes what it consumes).
 * q_out (nullable) [2][batch] receives Q1,Q2(s,a) before the update, y_out (nullable) [batch] the targets.
 * Increments steps[1]. */
/* params_t: a second arena of the same size holding the hidden-layer weights transposed ([in][out], what the forward
 * kernels read).  rtd3_td3_adam_polyak keeps it in step; call this after writing weights into `params` directly. */
int32_t rtd3_td3_sync_transposed(rtd3_td3* h, const float* params, float* params_t, void* stream);

int32_t rtd3_td3_critic_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const float* rp_s,
                             const float* rp_a, const float* rp_r, const float* rp_s2, const float* rp_notdone,
                             const int32_t* idx, const float* noise, int32_t batch, float gamma, float policy_noise,
                             float noise_clip, float max_action, float* loss2, float* q_out, float* y_out, int32_t* steps,
                             double* beta_pows, void* stream);

/* TD3.train_actor minus the optimiser step (robot.py:382-394): loss = -mean(Q1(s, pi(s))) added into
 * loss1[0]; gradient w.r.t. the actor parameters only, written to grads (same zero-on-entry rule).
 * Increments steps[0]. */
int32_t rtd3_td3_actor_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const float* rp_s,
                            const int32_t* idx, int32_t batch, float* loss1, int32_t* steps, double* beta_pows, void* stream);

/* torch.optim.Adam step (lr, betas 0.9/0.999, eps 1e-8; robot.py:237-239, 356-363, 393-395) on the nets
 * selected by `nets` (bit 0 actor, bit 1 critic1, bit 2 critic2) using grads*grad_scale (grad_scale = 1/world
 * after a gradient all-reduce), zeroing the consumed gradients; then TD3.soft_update (robot.py:293-310)
 * on the target nets selected by `polyak` (same bit layout) with the freshly updated online parameters.
 * params_uv (nullable): the tensor-core operand copies of the arena (see rtd3_tc_sync_weights), kept in step too. */
int32_t rtd3_td3_adam_polyak(rtd3_td3* h, float* params, float* params_t, float* params_uv, float* grads, float* adam_m, float* adam_v,
                             const double* beta_pows, int32_t nets, double lr_actor, double lr_critic, float grad_scale, int32_t polyak,
                             float tau, void* stream);

/* Forward of one network of the arena (robot.py:153-159 / 193-200): x [batch][in] -> y [batch][out]. */
int32_t rtd3_mlp_forward(rtd3_td3* h, int32_t net, const float* params, const float* params_t, const float* x, float* y,
                         int64_t batch, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Robot per-step hooks                         (robot.py:443-675, 727-762)
 * Per-env robot state lives in caller-owned device arrays: goal [2][n] float64; stuck history ring
 * hist [5][2][n] float32 with hist_count/hist_head int32 [n]; goal_reached / stuck_flag / demo_flag uint8 [n];
 * plan_index / path_length / num_episodes int32 [n]; noise_scale float64 [n].
 * ---------------------------------------------------------------------------------------------- */

/* baseline_action = state - goal as float32 [n][2] (robot.py:556/586, :612) - the actor's input. */
int32_t rtd3_robot_baseline(const float* x, const float* y, const double* goal, float* base, int64_t n, void* stream);

/* get_next_action_training / _testing after the actor forward (robot.py:560-567 / 590-593):
 * action = clip(baseline + residual [n][2] + unit_noise * noise_scale * 5, +-5) evaluated in float64;
 * unit_noise [2][n] float64 standard normals (NULL = testing, no noise; robot.py:640 otherwise).
 * type (nullable int8 [n], the output of rtd3_robot_next_action_type): envs whose type is not 0 ('step') get a
 * null action.  ax, ay receive float32 actions, action64 (nullable) [2][n] the float64 values. */
int32_t rtd3_robot_compose_action(const float* x, const float* y, const double* goal, const float* residual,
                                  const double* unit_noise, const double* noise_scale, const int8_t* type, float* ax,
                                  float* ay, double* action64, int64_t n, void* stream);

/* Robot.process_transition (robot.py:645-675) for n envs: compute_reward (robot.py:727-762: goal radius,
 * distance to goal, 10 x distance to the nearest of the num_demo demonstration states demo [num_demo][2]
 * float64 shared by all envs, applied where demo_flag is set), check_if_stuck on the pre-step state
 * (robot.py:509-538, -50 penalty), done = plan_index == path_length - 1, and the replay push of the n rows at
 * (position + i) % capacity (rp_s == NULL skips the push).  reward float32 [n] (reward64 nullable float64).
 * demo_list_start (nullable int32 [RTD3_DEMO_GRID^2 + 1]) / demo_list (float64 [total][2]): the candidate lists built by
 * rtd3_demo_lists.  When given, a query in cell c = floor(x) * RTD3_DEMO_GRID + floor(y) evaluates only the states
 * demo_list[demo_list_start[c] .. demo_list_start[c+1]) - same float64 operations per candidate as the full sweep and the
 * true nearest state is among them, so the result is bit-identical; `demo` must still hold the whole set (queries outside
 * the grid sweep it).
 * type (nullable int8 [n]): only envs of type 0 ('step') are processed; their rows are then compacted behind the
 * ring's device row counter rp_total (uint64 [1], rows ever pushed; required with type, optional otherwise -
 * when given it is advanced by n). */
/* env_demo_pts / env_demo_cells / env_demo_count / env_demo_cap (nullable): PER-ENV demonstration sets as built by
 * rtd3_robot_process_demonstration; when given, env i's proximity term looks at its own set (exact nearest state by a ring search over
 * the env's 25 x 25 grid - bit-identical to the sweep) and `demo` / the lists are ignored. */
int32_t rtd3_robot_transition(const double* goal, float* hist, int32_t* hist_count, int32_t* hist_head, uint8_t* goal_reached,
                              uint8_t* stuck_flag, const uint8_t* demo_flag, const int32_t* plan_index,
                              const int32_t* path_length, const float* sx, const float* sy, const float* ax, const float* ay,
                              const float* nx, const float* ny, const double* demo, const int32_t* demo_list_start,
                              const double* demo_list, int64_t num_demo, float* reward,
                              double* reward64, uint8_t* done, float* rp_s, float* rp_a, float* rp_r, float* rp_s2,
                              float* rp_notdone, int64_t capacity, int64_t position, uint64_t* rp_total, const int8_t* type,
                              const double* env_demo_pts, const int32_t* env_demo_cells, const int32_t* env_demo_count, int64_t env_demo_cap,
                              int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Demonstrations for a batch of envs          (environment.py:140-179, robot.py:679-718, 771-823)
 * ---------------------------------------------------------------------------------------------- */
/* Workspace of the planner for n envs, P paths, T steps, E elites (HOST struct of DEVICE pointers, all owned by the caller). */
typedef struct rtd3_cem_workspace {
  float* actions;        /* [T][2][P*n]  planning_actions of the current iteration; virtual env v = p*n + i */
  float* x;              /* [P*n] rollout state (final states of the paths after an iteration) */
  float* y;
  float* start_x;        /* [n] robot_current_state of the planner (float32) */
  float* start_y;
  double* start64;       /* nullable [2][n]: its float64 draw */
  double* rewards;       /* [n][P] planning_path_rewards of the current iteration */
  int32_t* elite;        /* [n][E] indices_best_paths (ascending reward) */
  int32_t* best;         /* [n] index_best_path of the current iteration */
  float* mean;           /* [T][2][n] best_paths_action_mean */
  float* std;            /* [T][2][n] best_paths_action_std_dev */
  float* best_actions;   /* [T][2][n] */
  float* traj;           /* [T][2][n] path of the best action sequence */
} rtd3_cem_workspace;

/* Environment.get_demonstration (environment.py:140-179) for the n envs of `bank` (each env's own numpy-legacy stream, own init
 * region [4][n] and goal [2][n]): iterations it_begin..it_end-1 of the cross-entropy-method planner (it_begin == 0 also draws the
 * start state; a full call is 0..iterations) and, with finish != 0, the demonstration itself: demo_states / demo_actions [n][T][2]
 * float32 = the best path of the last iteration run (its start state and first T-1 states) and its actions.  Random draws and their
 * order are the reference's (start: 2 doubles; iteration 0: one 32-bit word per action component; later: legacy_gauss per component;
 * path-major, then step, then component); the P*n rollouts of an iteration are one launch of the rollout kernel. */
int32_t rtd3_env_get_demonstration(rtd3_env* h, const rtd3_mt_bank* bank, const double* region, const double* goal, const rtd3_cem_workspace* w,
                                   int32_t iterations, int32_t paths, int32_t steps, int32_t elites, int32_t it_begin, int32_t it_end,
                                   int32_t finish, float* demo_states, float* demo_actions, void* stream);

/* Robot.process_demonstration (robot.py:679-718) for n envs, each with its own demonstration [n][T][2] (float32 states / actions):
 * appends the T states and `augments` augmentations (robot.py:771-823; noise from env i's stream of `bank`, drawn in the reference's
 * order - the augmented actions' noise included) to env i's set `sets` [n][cap][2] float64 (set_count [n] advanced), rebuilds the env's
 * search grid (sorted [n][cap][2], cells [n][RTD3_ENV_DEMO_CELLS + 1]) and pushes the T-1 transitions of every env into the replay ring
 * behind rp_total (env-major; reward = compute_reward([next_state]), robot.py:727-762, with the env's demo_flag; done on the last one).
 * rp_s == NULL skips the push.  The caller guarantees set_count[i] + T + augments * ((T-1) * (interpolation+1) + 1) <= cap. */
int32_t rtd3_robot_process_demonstration(const rtd3_mt_bank* bank, const double* goal, const uint8_t* demo_flag, const float* demo_states,
                                         const float* demo_actions, int32_t steps, double* sets, int32_t* set_count, double* sorted,
                                         int32_t* cells, int64_t cap, int32_t augments, int32_t interpolation, double noise_level, float* rp_s,
                                         float* rp_a, float* rp_r, float* rp_s2, float* rp_notdone, int64_t capacity, uint64_t* rp_total,
                                         void* stream);

/* Candidate lists for the nearest-demonstration term of compute_reward (robot.py:753: cdist(...).min() over ALL demonstration
 * states).  For every 1 x 1 cell of the world: the states that can be the nearest one for some point of the cell - a state is
 * dropped when another state is closer at all four corners of the cell (then it is closer everywhere in it); tested against the
 * states nearest to the corners and the centre.  Two passes over demo [num_demo][2] float64, one CTA per cell:
 *   list == NULL: counts int32 [RTD3_DEMO_GRID^2] receives the list sizes (the caller turns them into start offsets);
 *   list != NULL: start int32 [RTD3_DEMO_GRID^2 + 1] given, the lists are written to list [start[cells]][2] float64. */
int32_t rtd3_demo_lists(const double* demo, int64_t num_demo, int32_t* counts, const int32_t* start, double* list, void* stream);

/* Robot.get_next_action_type + Robot.reset (robot.py:443-506) for n envs.  type_out int8 [n]: 0 'step',
 * 1 'demo', 2 'reset'; update_out uint8 [n] marks envs whose episode ended (where the reference calls
 * td3_update, robot.py:480-483); any_update int32 [1] (zeroed by the caller) receives how many envs did. */
int32_t rtd3_robot_next_action_type(int32_t* num_episodes, uint8_t* demo_flag, int32_t* plan_index, int32_t* path_length,
                                    uint8_t* goal_reached, uint8_t* stuck_flag, double* noise_scale, int8_t* type_out,
                                    uint8_t* update_out, int32_t* any_update, int64_t n, void* stream);

/* Money counters of the driver loop (robot-learning.py:78, 86, 99: one reset / one step bought) for n envs in one launch:
 * steps[i] += (type[i] == 0), resets[i] += (type[i] == 2). */
int32_t rtd3_trainer_tally(const int8_t* type, int64_t* steps, int64_t* resets, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Data-parallel learner: gradient all-reduce over NVLink peer memory        (SURVEY.md 8e; no counterpart in the reference)
 * ---------------------------------------------------------------------------------------------- */
#define RTD3_P2P_MAX_WORLD 8
/* SUM all-reduce of the ranks' flat gradient buffers in ONE launch per optimiser step over peer memory (CUDA IPC mappings across
 * NVLink / NVSwitch), push model: every rank stores its gradients into slot [step parity][rank] of every rank's receive area,
 * raises the peers' flags, waits for all flags of the step and adds the `world` slots of its own area in rank order (bit-identical
 * sums on all ranks).  peer_recv / peer_flags: HOST arrays of `world` DEVICE pointers - rank r's receive area (2 * world * count
 * floats, 16 B aligned) and flag array (RTD3_P2P_MAX_WORLD uint64, zero-initialised once) as mapped in THIS process.
 * seq_counter: uint64 [1] in device memory, zero-initialised once; the kernel advances it (the step number is what the flags
 * carry; every rank must issue the same sequence of calls).  out (count floats, private) receives the sum; local_grads (count
 * floats, private) is read and cleared.  block_counter: uint32 [1], zero-initialised once.  A rank whose peers do not arrive within
 * 20 s traps (the launch fails) instead of hanging.  A plain launch: it may be captured in a CUDA graph. */
/* slot_floats: distance between two slots of a receive area (>= count, a multiple of 4; the area holds 2 * world * slot_floats
 * floats).  Calls of different `count` may alternate on one area (critic gradients, then actor gradients) as long as they use the
 * same slot_floats. */
int32_t rtd3_p2p_allreduce(float* const* peer_recv, uint64_t* const* peer_flags, int32_t rank, int32_t world, uint64_t* seq_counter,
                           float* out, float* local_grads, int64_t count, int64_t slot_floats, uint32_t* block_counter, void* stream);

/* The same arguments as a HOST struct (what rtd3_td3_update takes). `sum`: private buffer the optimiser reads (same indexing as grads).
 * rtd3_td3_update fuses the optimiser into its all-reduce launches and hands the data over per thread block: for that form every
 * flag array must hold 16 + RTD3_P2P_MAX_WORLD * 256 uint64 (zero-initialised once): [0, 16) as above, then one flag per
 * (rank, block). */
typedef struct rtd3_p2p_state {
  float* const* peer_recv;
  uint64_t* const* peer_flags;
  int32_t rank;
  int32_t world;
  uint64_t* seq_counter;
  float* sum;
  int64_t slot_floats;
  uint32_t* block_counter;
} rtd3_p2p_state;

/* NCCL communicator of the data-parallel learner (north star: "NCCL over NVLink used only for the actor/critic gradient allreduce").
 * librtd3 resolves libnccl.so.2 at run time (the copy already loaded into the process - torch's - else the system one); there is no
 * link-time dependency.  The host creates a unique id on one rank (rtd3_comm_unique_id, HOST buffer of RTD3_COMM_ID_BYTES), hands it
 * to the other ranks over any channel it has, and every rank calls rtd3_comm_create (collective).  Errors: 1000 + ncclResult_t. */
#define RTD3_COMM_ID_BYTES 128
typedef struct rtd3_comm rtd3_comm;
int32_t rtd3_comm_nccl_version(void);                      /* e.g. 22809, -1 if NCCL cannot be loaded */
int32_t rtd3_comm_unique_id(uint8_t* id_out);              /* HOST [RTD3_COMM_ID_BYTES] */
int32_t rtd3_comm_create(rtd3_comm** out, const uint8_t* id /*HOST*/, int32_t rank, int32_t world, int32_t device);
int32_t rtd3_comm_destroy(rtd3_comm* comm);
int32_t rtd3_comm_world(const rtd3_comm* comm);
int32_t rtd3_comm_rank(const rtd3_comm* comm);
/* SUM all-reduce, in place, of the flat fp32 gradient buffer over the ranks of `comm` on `stream` (SURVEY.md 8b/8e).  The optimiser
 * then applies grad_scale = 1/world.  A plain stream operation on our own communicator: capturable in a CUDA graph. */
int32_t rtd3_allreduce_grads(rtd3_comm* comm, float* flat_grads, int64_t count, void* stream);

/* ------------------------------------------------------------------------------------------------
 * TD3.td3_update (robot.py:258-285) in one call
 * ---------------------------------------------------------------------------------------------- */
typedef struct rtd3_td3_update_args {
  /* learner state (arena notes above) */
  float* params;
  float* params_t;
  float* params_uv;              /* nullable unless tf32: tensor-core operand copies, kept in step */
  float* grads;
  float* adam_m;
  float* adam_v;
  float* scratch;                /* rtd3_td3_scratch_floats(batch) floats (fp32 steps) */
  int32_t* steps;                /* [2] */
  double* beta_pows;             /* [4] */
  /* replay ring */
  const float* rp_s;
  const float* rp_a;
  const float* rp_r;
  const float* rp_s2;
  const float* rp_notdone;
  /* minibatches: index sets in the order the reference draws them (critic of epoch 0, actor of epoch 0, critic of epoch 1, ...) */
  const int32_t* idx;            /* [epochs + ceil(epochs / policy_update_delay)][batch] */
  int32_t batch;
  int32_t epochs;
  int32_t policy_update_delay;   /* robot.py:278 */
  /* target-policy smoothing noise (robot.py:338): a unit-normal tensor [epochs][batch][2], or NULL = generated in the critic kernel
   * from Philox4x32-10 keyed (noise_seed, noise_counter[0] + epoch, row); the call then advances noise_counter by `epochs` */
  const float* noise;
  uint64_t noise_seed;
  uint64_t* noise_counter;       /* DEVICE uint64 [1] */
  float gamma, policy_noise, noise_clip, max_action;
  double lr_actor, lr_critic;     /* double, like torch's lr: the step size lr / (1 - 0.9^t) is rounded to float32 once */
  float tau;
  /* outputs: the values the reference collects at robot.py:274-280 */
  float* critic_losses;          /* [epochs][2] */
  float* actor_losses;           /* [ceil(epochs / policy_update_delay)] */
  /* data-parallel learner: world > 1 needs exactly one of comm (NCCL) / p2p (peer memory) */
  int32_t world;
  int32_t tf32;                  /* 1: rtd3_td3_*_step_tf32 (tcgen05) instead of the fp32 steps */
  rtd3_comm* comm;
  const rtd3_p2p_state* p2p;
} rtd3_td3_update_args;

/* The unit normals rtd3_td3_update's critic kernels generate for step `counter` (= noise_counter[0] + epoch): out [rows][2] float32 =
 * Box-Muller of two 53-bit uniforms from Philox4x32-10, counter (row lo, row hi, step lo, step hi), key (seed lo, seed hi). */
int32_t rtd3_td3_target_noise(uint64_t seed, uint64_t counter, float* out, int64_t rows, void* stream);

/* The epoch loop of TD3.td3_update: per epoch rtd3_td3_critic_step -> [all-reduce of the critic gradients] -> Adam on both critics;
 * every policy_update_delay-th epoch rtd3_td3_actor_step -> [all-reduce of the actor gradients] -> Adam on the actor + the three
 * Polyak updates.  Everything is issued on `stream` without synchronising (capturable in one CUDA graph). */
int32_t rtd3_td3_update(rtd3_td3* h, const rtd3_td3_update_args* args, void* stream);

/* The same update as ONE persistent cooperative kernel (csrc/rtd3_coop.cu) - the small-batch learner: one CTA per SM stays
 * resident for all `epochs`, every hidden-layer product is tiled over all SMs, the layers of the chain are separated by grid-wide
 * barriers instead of kernel launches, Adam / Polyak and (world > 1, peer memory only: args->p2p) the gradient all-reduce are stages
 * of the same kernel.  fp32 (FFMA), layers >= 2, batch <= 4096; same arithmetic as the step kernels up to summation order
 * (losses / Q-values within the 1e-3 parity bar).  args->scratch, params_uv, comm and tf32 are not used.
 * coop_scratch: rtd3_td3_coop_scratch_floats(batch) floats, 16 B aligned, ZERO-initialised once by the caller (its first words are
 * the grid barrier) and then left to the kernel. */
int32_t rtd3_td3_coop_supported(const rtd3_td3* h, int32_t batch);
int64_t rtd3_td3_coop_scratch_floats(const rtd3_td3* h, int32_t batch);
int32_t rtd3_td3_update_coop(rtd3_td3* h, const rtd3_td3_update_args* args, float* coop_scratch, void* stream);
/* Development aid: DEVICE buffer of 256 int64 that the following cooperative updates stamp with %globaltimer at every stage boundary
 * of their last epoch (block 0: arrival at the grid barrier, release from it); NULL switches it off. */
int32_t rtd3_debug_coop_prof(long long* device_buf);

/* Small-batch step kernels on thread-block clusters (csrc/rtd3_cluster.cu; the default of rtd3_td3_critic_step / rtd3_td3_actor_step /
 * rtd3_td3_update for fp32 batches that are ONE wave of clusters: 8 rows per cluster, 33 clusters on a B200 = up to 264 rows): 1 if the step of `batch` rows runs on that path, and how many of its 4-CTA clusters the
 * device can hold at once (cudaOccupancyMaxActiveClusters of the critic kernel; negative: CUDA error). */
int32_t rtd3_td3_cluster_supported(const rtd3_td3* h, int32_t batch);
int32_t rtd3_td3_cluster_occupancy(const rtd3_td3* h, int32_t batch);
/* Development / test aid: 0 = the step entry points use the row-tile kernels, 2 = the cluster kernels wherever their plan fits (the
 * default); returns the previous mode (1 = a shape forced through RTD3_CLUSTER=R,CS).  Not thread-safe against running launches. */
int32_t rtd3_debug_cluster_mode(int32_t mode);
/* Development: stage stamps (%globaltimer, ns) of the last weight-gradient launch that exchanged its tiles with the peers
 * (rtd3_td3_update at world > 1 over peer memory, RTD3_P2P_PROF=1): out_host [256 blocks][2 threads][8 stages] uint64.  Returns 1 if
 * the stamps were copied, 0 if profiling is off. */
int32_t rtd3_debug_p2p_prof(uint64_t* out_host);
/* Development aid: DEVICE buffers of 256 int64 each that the following cluster critic / actor kernels fill with clock64 stamps of
 * CTA 0 at every stage boundary ([0] = number of stamps); NULL switches it off. */
int32_t rtd3_debug_cluster_prof(long long* critic_buf, long long* actor_buf);

/* ------------------------------------------------------------------------------------------------
 * Fused tick of the batched driver loop        (robot-learning.py:66-101, training branch)
 * ---------------------------------------------------------------------------------------------- */
/* Everything one tick touches, for n envs.  HOST struct of DEVICE pointers (same arrays as the per-hook entry points above take). */
typedef struct rtd3_tick_state {
  int64_t n;
  /* Environment */
  float* x;                     /* [n] robot_state planes, stepped / reset in place */
  float* y;
  const double* goal;           /* [2][n] */
  const double* region;         /* [4][n] left,right,bottom,top */
  double* state64;              /* nullable [2][n]: float64 value of the last reset draw */
  rtd3_mt_bank env_bank;        /* the envs' reset streams */
  /* Robot episode state (robot.py:421-438) */
  int32_t* num_episodes;        /* [n] */
  uint8_t* demo_flag;
  int32_t* plan_index;
  int32_t* path_length;
  uint8_t* goal_reached;
  uint8_t* stuck_flag;
  double* noise_scale;
  float* hist;                  /* [5][2][n] */
  int32_t* hist_count;
  int32_t* hist_head;
  int8_t* type;                 /* [n] out: 0 'step', 1 'demo', 2 'reset' */
  uint8_t* update;              /* [n] out: episode ended in this tick */
  int32_t* any_update;          /* [1] accumulates the number of ended episodes */
  /* per-tick outputs */
  float* base;                  /* [n][2] actor input (state - goal) written by rtd3_tick_pre */
  float* ax;                    /* [n] action planes */
  float* ay;
  float* prev_x;                /* nullable [n]: pre-step state */
  float* prev_y;
  float* reward;                /* [n] (stepping envs only) */
  double* reward64;             /* nullable */
  uint8_t* done;                /* [n] */
  /* demonstration states shared by all envs (as rtd3_robot_transition) */
  const double* demo;
  const int32_t* demo_list_start;
  const double* demo_list;
  int64_t num_demo;
  /* replay ring (masked push through the device row counter) */
  float* rp_s;
  float* rp_a;
  float* rp_r;
  float* rp_s2;
  float* rp_notdone;
  int64_t capacity;
  uint64_t* rp_total;
  /* money counters (robot-learning.py:78, 86, 99) */
  int64_t* steps_bought;        /* [n] */
  int64_t* resets_bought;       /* [n] */
  /* exploration noise of mode RTD3_TICK_NOISE_PHILOX: normals = f(philox_seed, ticks run incl. this one, env) */
  uint64_t philox_seed;
  uint64_t* tick_counter;       /* nullable [2]: word 0 = ticks completed (advanced by rtd3_tick_post), word 1 = scratch of the tick in flight */
  /* Scheduler of the driver loop (robot-learning.py:45-50 money, :66-103 purchase gates and the switch to testing, :104-117 test
   * branch).  mode == NULL: training branch only, every purchase goes through (the arrays below are then ignored). */
  uint8_t* mode;                /* [n] 0 training, 1 testing, 2 finished */
  int64_t* demos_bought;        /* [n] */
  int32_t* test_ticks;          /* [n] ticks spent in testing */
  double* test_best;            /* [n] best distance to the goal seen in testing (initialise to +inf) */
  uint8_t* test_success;        /* [n] reached the goal: distance <= 5 (constants.py:50) */
  uint8_t* penalty;             /* [n] overspent by more than 1 at the switch (robot-learning.py:73-75) */
  double tick_seconds;          /* deterministic stand-in for the wall-clock money term: cpu_time = ticks elapsed * tick_seconds */
  int64_t test_timeout_ticks;   /* TEST_TIMEOUT (constants.py:53, compared with wall time at robot-learning.py:115) in ticks */
  /* per-env demonstration sets (rtd3_robot_process_demonstration); env_demo_pts == NULL: the shared set above is used */
  const double* env_demo_pts;   /* [n][env_demo_cap][2], sorted by grid cell */
  const int32_t* env_demo_cells; /* [n][RTD3_ENV_DEMO_CELLS + 1] */
  const int32_t* env_demo_count; /* [n] */
  int64_t env_demo_cap;
} rtd3_tick_state;

/* values of rtd3_tick_state.type beyond 0 'step' / 1 'demo' / 2 'reset' (scheduler only) */
#define RTD3_TICK_TYPE_SWITCH 3    /* money < 0: environment.reset() and on to testing (robot-learning.py:70-80) */
#define RTD3_TICK_TYPE_SKIP 4      /* the purchase was not affordable: nothing happens in this tick */
#define RTD3_TICK_TYPE_TEST 5      /* a test step: get_next_action_testing, step, distance check (robot-learning.py:104-117) */
#define RTD3_TICK_TYPE_IDLE 6      /* the env's run is over */

#define RTD3_TICK_NOISE_NONE 0     /* get_next_action_testing: no exploration noise (robot.py:575-595) */
#define RTD3_TICK_NOISE_GIVEN 1    /* unit normals supplied ([2][n] float64, e.g. rtd3_mt_draw_gauss: numpy-exact) */
#define RTD3_TICK_NOISE_PHILOX 2   /* unit normals generated in the kernel (Philox4x32-10 + Box-Muller, throughput mode) */

/* First half of a tick: rtd3_robot_next_action_type (robot.py:443-506; robot-learning.py:68), the scheduler's purchase gates when
 * t->mode is set, and rtd3_robot_baseline (robot.py:556) in one launch.  The caller then runs the actor forward on t->base. */
int32_t rtd3_tick_pre(const rtd3_tick_state* t, void* stream);

/* Second half, one launch: rtd3_robot_compose_action (robot.py:560-567), rtd3_env_step (environment.py:122-127),
 * rtd3_robot_transition with the masked replay push (robot.py:645-675), rtd3_trainer_tally and rtd3_env_reset for the envs whose
 * type is 'reset' (robot-learning.py:82-101).  residual: [n][2] actor output.  Leaves every array bit-identical to the sequence
 * of those calls. */
int32_t rtd3_tick_post(rtd3_env* h, const rtd3_tick_state* t, const float* residual, const double* unit_noise, int32_t noise_mode,
                       void* stream);

/* `ticks` consecutive ticks in ONE launch, the actor (2 -> hidden -> hidden -> 2, network 0 of the arena) evaluated in the kernel
 * by the f16 resident-weight forward (rtd3_mlp_forward_f16; params_h from rtd3_tc_sync_weights_f16): every CTA runs all the ticks
 * of its 128-env tiles - envs are independent - so the hidden weight is loaded once per launch and a tick costs no launch.
 * Leaves every array as `ticks` rounds of rtd3_tick_pre / rtd3_mlp_forward_f16 / rtd3_tick_post would (the replay rows in another
 * order); the Philox noise of tick k is keyed tick_base + k + 1 (tick_base = ticks run so far), and tick_counter is left at
 * tick_base + ticks.  noise_mode NONE or PHILOX; needs demo_list_start (or num_demo == 0); layers == 2, hidden % 32 == 0, 64..256. */
int32_t rtd3_tick_run_f16(rtd3_env* h, const rtd3_tick_state* t, int32_t hidden, int32_t layers, const float* params,
                          const uint16_t* params_h, int32_t noise_mode, int64_t ticks, uint64_t tick_base, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Batched policy evaluation: the test phase of robot-learning.py:104-117 for n envs
 * For t = 1..T: base = state - goal, residual = actor(base), action = clip(base + residual, +-5) (get_next_action_testing,
 * robot.py:572-595), state = Environment.step(action) on env i's map of `h` (map index[i % m]), d = |state - goal| (float64, as
 * np.linalg.norm).  best = min(best, d); d <= 5 (constants.py:50): success, the env stops with steps = t; t == T: it stops with
 * steps = T.  A stopped env keeps its state.  goal [2][n] float64; x, y [n] float32: the start state in, the final state out;
 * success uint8 [n], steps int32 [n], best float64 [n].  traj: [T][2][n] float32, row t-1 = the state after step t, the rows
 * after an env's stop repeat its final state; given exactly when `record` is set.  Both entry points check every argument
 * before any launch, are asynchronous on `stream`, allocate nothing and can be captured.  n < 2^31, 1 <= T < 2^30.
 * ---------------------------------------------------------------------------------------------- */

/* One step for every env that has not stopped (!success[i] && steps[i] < T), given residual [n][2] = actor(base) from any forward;
 * writes the next step's actor input to base [n][2].  Before the first step the caller sets success = 0, steps = 0, best = +inf
 * and base = state - goal (rtd3_robot_baseline), then calls a forward and this function T times. */
int32_t rtd3_eval_step(rtd3_env* h, const double* goal, float* x, float* y, const float* residual, float* base, uint8_t* success,
                       int32_t* steps, double* best, float* traj, int32_t record, int64_t n, int64_t T, void* stream);

/* The whole evaluation in ONE launch, the actor (network 0 of the arena, 2 -> hidden -> hidden -> 2) evaluated in the kernel by
 * the f16 resident-weight forward (params_h from rtd3_tc_sync_weights_f16); writes success, steps and best itself.  CTAs take
 * 128-env tiles from the device word `work` (DEVICE uint32 [1], reset on `stream` by this call) and a tile ends when all of its
 * envs have stopped.  Bit-identical to T rounds of rtd3_mlp_forward_f16 + rtd3_eval_step.  layers == 2, hidden % 32 == 0, 64..256. */
int32_t rtd3_eval_run_f16(rtd3_env* h, int32_t hidden, int32_t layers, const float* params, const uint16_t* params_h, const double* goal,
                          float* x, float* y, uint8_t* success, int32_t* steps, double* best, float* traj, int32_t record, int64_t n,
                          int64_t T, uint32_t* work, void* stream);

/* E test episodes of every env, each from one of the env's own reset draws: bit-identical to E rounds of (rtd3_env_reset, the
 * evaluation above).  Episode e of env i starts from the (e+1)-th draw of stream i, steps on env i's map and is tested against
 * env i's goal.  1 <= E <= 1024, E * n < 2^31; every argument is checked before any launch.
 *
 * rtd3_eval_starts: the E draws of every env of `bank` (n = bank->n) in one launch.  starts [E][2][n] float32 gets the start
 * states in draw order; the stream words and pos end where E rtd3_env_reset calls leave them (streams that wrap included), and
 * state64 [2][n] holds the last draw.  base: nullable [E*n][2] float32, the first actor input state - goal of row e*n + i (for
 * rtd3_eval_step_episodes); goal [2][n] is read only when base is given. */
int32_t rtd3_eval_starts(const rtd3_mt_bank* bank, const double* region, const double* goal, int64_t E, float* starts, float* base,
                         double* state64, void* stream);

/* rtd3_eval_step for a batch of E*n rows, row e*n + i being episode e of env i: xs [E][2][n] the states (the starts in, the final
 * states out), residual / base [E*n][2], success / steps / best [E][n], traj [E][T][2][n]. */
int32_t rtd3_eval_step_episodes(rtd3_env* h, const double* goal, int64_t E, float* xs, const float* residual, float* base, uint8_t* success,
                                int32_t* steps, double* best, float* traj, int32_t record, int64_t n, int64_t T, void* stream);

/* rtd3_eval_run_f16 for E episodes in ONE launch: CTAs take (episode, tile) work items, E * ceil(n / 128) of them.  Episode e
 * starts from starts [E][2][n]; success / steps / best [E][n], traj [E][T][2][n]; x, y [n] get the final states of episode E-1. */
int32_t rtd3_eval_run_f16_episodes(rtd3_env* h, int32_t hidden, int32_t layers, const float* params, const uint16_t* params_h,
                                   const double* goal, const float* starts, int64_t E, float* x, float* y, uint8_t* success, int32_t* steps,
                                   double* best, float* traj, int32_t record, int64_t n, int64_t T, uint32_t* work, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Tensor-core (tcgen05 / TMEM, TF32) large-batch forward - opt-in throughput mode, not the parity path
 * ---------------------------------------------------------------------------------------------- */

/* Rebuild params_uv = [u | v] (2 x arena floats), the chunk-major (UMMA shared-memory operand order) copies of all
 * hidden-to-hidden weights, rounded to TF32 (round to nearest):
 *   u (forward):         Wu[(k/4)*H + n][k%4] = W[n][k]        v (input gradient):  Wv[(n/4)*H + k][n%4] = W[n][k]
 * other entries are copied in place. */
int32_t rtd3_tc_sync_weights(int32_t hidden, int32_t layers, const float* params, float* params_uv, void* stream);

/* Forward of one network (robot.py:153-159 / 193-200) for 128-row batch tiles on the 5th-gen tensor cores:
 * hidden H x H layers as tcgen05.mma.kind::tf32 with fp32 accumulators in TMEM, first / output layer in fp32.
 * param_off = rtd3_td3_param_offset(net). hidden % 32 == 0, 64..256; layers >= 2.  Agrees with rtd3_mlp_forward
 * to TF32 round-off (~1e-3 relative). */
int32_t rtd3_mlp_forward_tf32(int32_t hidden, int32_t layers, int32_t is_actor, int64_t param_off, const float* params,
                              const float* params_u, const float* x, float* y, int64_t batch, void* stream);

/* fp16 copies of the hidden-to-hidden weights for rtd3_mlp_forward_f16: params_h holds 6 * (layers-1) * hidden^2 halves,
 * matrix l of network net at ((net*(layers-1) + l-1) * hidden^2), in UMMA operand order Wh[(k/8)*H + n][k%8] = half(W[n][k]). */
int32_t rtd3_tc_sync_weights_f16(int32_t hidden, int32_t layers, const float* params, uint16_t* params_h, void* stream);

/* Forward of network `net` (0..5, arena order) with fp16 operands - the same 11-bit significand as TF32 in half the bytes, so the
 * hidden weight (128 KB at H = 256) stays RESIDENT in shared memory instead of being streamed from L2 per 128-row tile, the
 * tcgen05.mma.kind::f16 products accumulate in fp32 in two TMEM buffers, and the epilogue (bias, ReLU, fused output layer) of
 * one tile overlaps the products of the next.  layers == 2, hidden % 32 == 0, 64..256.  First / output layer in fp32.
 * Agrees with rtd3_mlp_forward to fp16-operand round-off (~1e-3 relative); opt-in throughput mode, not the parity path. */
int32_t rtd3_mlp_forward_f16(int32_t hidden, int32_t layers, int32_t net, const float* params, const uint16_t* params_h, const float* x,
                             float* y, int64_t batch, void* stream);

/* 1 if the tensor-core learner steps below support this handle's shape (layers == 2, hidden 128 or 256). */
int32_t rtd3_td3_tf32_supported(const rtd3_td3* h);

/* rtd3_td3_critic_step / rtd3_td3_actor_step (robot.py:312-366, 369-398) for large batches on the tensor cores:
 * 64-row batch tiles, hidden products (forward, input gradient, weight gradient) as tcgen05.mma.kind::tf32 with
 * accumulators in TMEM, weight gradients reduced over the batch tiles by TMA reduce-adds into `grads` (which must be
 * zero on entry - rtd3_td3_adam_polyak re-zeroes what it consumes).  Same arguments as the fp32 calls, with
 * params_uv (rtd3_tc_sync_weights / rtd3_td3_adam_polyak keep it) instead of params_t and no row scratch.
 * Agrees with the fp32 calls to TF32 round-off; opt-in throughput mode, not the parity path. */
int32_t rtd3_td3_critic_step_tf32(rtd3_td3* h, const float* params, const float* params_uv, float* grads, const float* rp_s,
                                  const float* rp_a, const float* rp_r, const float* rp_s2, const float* rp_notdone, const int32_t* idx,
                                  const float* noise, int32_t batch, float gamma, float policy_noise, float noise_clip, float max_action,
                                  float* loss2, float* q_out, float* y_out, int32_t* steps, double* beta_pows, void* stream);
int32_t rtd3_td3_actor_step_tf32(rtd3_td3* h, const float* params, const float* params_uv, float* grads, const float* rp_s,
                                 const int32_t* idx, int32_t batch, float* loss1, int32_t* steps, double* beta_pows, void* stream);

/* Development aid: switch the phase timestamps of the tf32 critic kernel (clock64 of CTA 0 / thread 0 at every phase
 * boundary) on or off; `out` (nullable, host memory, 128 entries) receives the stamps of the last launch. */
int32_t rtd3_debug_lt_prof(int32_t on, long long* out);

#ifdef __cplusplus
}
#endif
#endif /* RTD3_H_ */
