// Batched policy evaluation: the reference's test phase (robot-learning.py:104-117) for every env of an environment.
//   for t = 1..T:  base = state - goal;  residual = actor(base);  action = clip(base + residual, +-5) (get_next_action_testing,
//                  robot.py:572-595);  state = step(state, action);  d = |state - goal|;  best = min(best, d);
//                  d <= 5: success, the env stops at t;  t == T: the env stops (time-out)
// A stopped env keeps its state.  Two paths, bit-identical for the same forward:
//   eval_step_kernel : one step for every env that has not stopped, given the residual of any actor forward (fp32, TF32, f16);
//                      it also writes the next step's actor input, so a step is two launches: the forward and this kernel.
//   eval_f16_kernel  : the whole evaluation in ONE launch, the actor evaluated in the kernel by the f16 resident-weight forward
//                      (rtd3_tc_f16.cuh) - per tile exactly the hf_* code rtd3_mlp_forward_f16 runs, so its residuals, and
//                      therefore every output, are bit-identical to eval_step_kernel behind rtd3_mlp_forward_f16.
// E episodes of every env (each from one of the env's own reset draws, eval_starts_kernel) run as E*n rows of the per-step path
// (eval_step_episodes_kernel) or as (episode, tile) work items of one persistent launch (eval_f16_episodes_kernel).
// Both use the per-env functions of the tick kernels (baseline_env, compose_env, step_one on the env's map, norm2_np) in the
// order of the test branch of tick_post_env (rtd3_tick.cu), so they also match the scheduler's test steps bit for bit.
#include "rtd3_common.cuh"
#include "rtd3_env_step.cuh"
#include "rtd3_mt.cuh"
#include "rtd3_robot.cuh"
#include "rtd3_tc_f16.cuh"

namespace rtd3 {

constexpr double kEvalDistance = 5.0;    // constants.py:50
constexpr int64_t kEvalMaxSteps = 1ll << 30;

// One test step of an env that has not stopped; t is the step's number (1-based).  Returns true when the env stops at t.
template <typename TableT>
__device__ __forceinline__ bool eval_env_step(const TableT& table, float& x, float& y, const double gx, const double gy, const float2 res,
                                              const int t, const int T, double& best, bool& succ) {
  double cx, cy;
  compose_env(x, y, gx, gy, res, false, 0.0, 0.0, 0.0, cx, cy);
  float nx, ny;
  step_one<true>(table, x, y, (float)cx, (float)cy, nx, ny);
  x = nx;
  y = ny;
  const double d = norm2_np(__dsub_rn((double)nx, gx), __dsub_rn((double)ny, gy));
  if (d < best) best = d;
  succ = d <= kEvalDistance;
  return succ || t >= T;
}

// One step for every env (thread i).  An env runs while !success[i] && steps[i] < T; its step number is steps[i] + 1.  With a
// trajectory, the running env writes row t - 1 and, when it stops at t, rows t .. T-1 with its final state.
template <bool kBank>
__global__ void __launch_bounds__(256) eval_step_kernel(MapBank bank, const double* __restrict__ goal, float* __restrict__ x_io,
                                                        float* __restrict__ y_io, const float* __restrict__ residual /*[n][2]*/,
                                                        float* __restrict__ base /*[n][2]*/, uint8_t* __restrict__ success,
                                                        int32_t* __restrict__ steps, double* __restrict__ best_io,
                                                        float* __restrict__ traj /*nullable [T][2][n]*/, int64_t n, int T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int done = steps[i];
  if (success[i] || done >= T) return;
  float x = x_io[i], y = y_io[i];
  const double gx = goal[i], gy = goal[n + i];
  double best = best_io[i];
  bool succ = false;
  const int t = done + 1;
  const bool stop = eval_env_step(LdgTable{bank.table<kBank>(i)}, x, y, gx, gy, reinterpret_cast<const float2*>(residual)[i], t, T, best, succ);
  x_io[i] = x;
  y_io[i] = y;
  best_io[i] = best;
  steps[i] = t;
  if (succ) success[i] = 1;
  reinterpret_cast<float2*>(base)[i] = baseline_env(x, y, gx, gy);
  if (traj)
    for (int r = t - 1; r < (stop ? T : t); ++r) {
      traj[(int64_t)(2 * r) * n + i] = x;
      traj[(int64_t)(2 * r + 1) * n + i] = y;
    }
}

// ---- E episodes of every env at once ---------------------------------------------------------------------------------------
// eval_starts_kernel: E resets of every env (Environment.reset E times), one warp per 32 envs drawing them in order; the start
// state of episode e goes to the planes starts [E][2][n], and - for the per-step path - its first actor input to base [E*n][2].
// The stream words and pos end where E launches of env_reset_kernel leave them, state64 at the last draw.
__global__ void eval_starts_kernel(rtd3_mt_bank b, const double* __restrict__ region, const double* __restrict__ goal, int E,
                                   float* __restrict__ starts, float* __restrict__ base, double* __restrict__ state64) {
  const int64_t n = b.n, i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < n;
  for (int e = 0; e < E; ++e) {
    float* const xs = starts + (int64_t)(2 * e) * n;
    reset_env_warp(b, region, active, i, xs, xs + n, e == E - 1 ? state64 : nullptr);
    if (base && active) reinterpret_cast<float2*>(base)[(int64_t)e * n + i] = baseline_env(xs[i], xs[n + i], goal[i], goal[n + i]);
  }
}

// eval_step_kernel for a virtual batch of E*n rows: row r = e*n + i (blockIdx.y = e) is episode e of env i, with env i's goal and
// map; its state is the planes xs [E][2][n], its results success, steps, best [E][n], its trajectory traj [E][T][2][n].
template <bool kBank>
__global__ void __launch_bounds__(256) eval_step_episodes_kernel(MapBank bank, const double* __restrict__ goal, float* __restrict__ xs,
                                                                 const float* __restrict__ residual /*[E*n][2]*/, float* __restrict__ base /*[E*n][2]*/,
                                                                 uint8_t* __restrict__ success, int32_t* __restrict__ steps, double* __restrict__ best_io,
                                                                 float* __restrict__ traj, int64_t n, int T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t e = blockIdx.y, r = e * n + i;
  const int done = steps[r];
  if (success[r] || done >= T) return;
  float* const xp = xs + 2 * e * n + i;                               // x at xp[0], y at xp[n]
  float x = xp[0], y = xp[n];
  const double gx = goal[i], gy = goal[n + i];
  double best = best_io[r];
  bool succ = false;
  const int t = done + 1;
  const bool stop = eval_env_step(LdgTable{bank.table<kBank>(i)}, x, y, gx, gy, reinterpret_cast<const float2*>(residual)[r], t, T, best, succ);
  xp[0] = x;
  xp[n] = y;
  best_io[r] = best;
  steps[r] = t;
  if (succ) success[r] = 1;
  reinterpret_cast<float2*>(base)[r] = baseline_env(x, y, gx, gy);
  if (traj) {
    float* const tp = traj + e * T * 2 * n + i;
    for (int k = t - 1; k < (stop ? T : t); ++k) {
      tp[(int64_t)(2 * k) * n] = x;
      tp[(int64_t)(2 * k + 1) * n] = y;
    }
  }
}

// ---- the whole evaluation in ONE launch (actor 2 -> H -> H -> 2 on the f16 resident-weight forward) ---------------------------
// A CTA takes 128-env tiles from a device work counter and runs up to T steps of a tile before it takes the next: a tile lasts
// from 1 to T steps (it ends when all of its envs have stopped), so tiles handed out statically would leave SMs idle at the end.
// Per step:
//   owner threads (warps 0-3, one env each; x, y, goal, best, steps and the stop flag live in their registers for the whole tile):
//     actor input, and a vote "some env of the tile still runs" (double-buffered by step parity)     -> barrier 1
//   16 row warps: no env runs -> meet the MMA warp at barrier 2 and leave the tile; else first layer into X -> barrier 2 ->
//     products -> epilogue -> barrier 1
//   MMA warp: barrier 2, reads the vote and issues the products only when some env runs (so the acc_ready parity stays in step)
//   owner threads: residual from the partial sums, then the test step of their env and the trajectory row
// The only global access per step is the env's table cell, through the read-only path (as in the tick kernels).
// kEp: the work items are (episode e, tile) pairs, e-major, E x tiles of them.  Item e reads its start from the planes
// starts [E][2][n], writes its results at [e][n] and its trajectory at traj + e*T*2*n; only e = E-1 writes the env state back.
// Without kEp there is one episode from x_io / y_io (starts and E unused).
template <bool kBank, bool kEp>
__device__ __forceinline__ void eval_f16_body(NetShape s, const float* __restrict__ P, const uint16_t* __restrict__ Wh, MapBank bank,
                                              const double* __restrict__ goal, const float* __restrict__ starts, int E, float* __restrict__ x_io,
                                              float* __restrict__ y_io, uint8_t* __restrict__ success, int32_t* __restrict__ steps_out,
                                              double* __restrict__ best_out, float* __restrict__ traj, int64_t n, int T,
                                              uint32_t* __restrict__ work, uint32_t tmem_cols) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int H = s.hid;
  const HfSmem m = hf_carve(smem_raw, H);
  float2* sbase = reinterpret_cast<float2*>(m.extra);                 // [128] actor input of the tile's envs
  int* svote = reinterpret_cast<int*>(sbase + kHfRows);               // [2 step parities][4 owner warps]
  uint32_t* stile = reinterpret_cast<uint32_t*>(svote + 8);           // the tile this CTA works on
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rt = (warp & 3) * 32 + lane, cpart = warp >> 2;
  int c_lo, c_hi;
  hf_columns(H, cpart, c_lo, c_hi);
  const uint32_t tiles = (uint32_t)((n + kHfRows - 1) / kHfRows);
  const uint32_t items = kEp ? tiles * (uint32_t)E : tiles;
  const uint32_t tmem = hf_setup(m, s, P, Wh, tmem_cols);
  const uint32_t idesc = hf_idesc(H);
  bool first = true;                                                  // MMA warp: the resident weight has not been waited for
  uint32_t phase = 0;                                                 // row warps: parity of acc_ready
  for (;;) {
    __syncthreads();                                                  // every thread has read the previous tile number
    if (tid == 0) *stile = atomicAdd(work, 1u);
    __syncthreads();
    const uint32_t item = *stile;
    if (item >= items) break;
    const uint32_t e = kEp ? item / tiles : 0u, tile = kEp ? item - e * tiles : item;
    if (warp == kHfRowWarps) {
      for (int k = 0; k < T; ++k) {
        bar_sync(2, kHfRowMma);                       // X of this step is in shared memory (or no env runs), the accumulator is drained
        const int* v = svote + (k & 1) * 4;
        if (!(v[0] | v[1] | v[2] | v[3])) break;
        if (lane == 0) {
          if (first) mbar_wait(m.w_full, 0);
          hf_issue_tile(m, H, tmem, idesc, m.acc_ready);
        }
        first = false;
        __syncwarp();
      }
    } else {
      const bool owner = cpart == 0;
      const int64_t i = (int64_t)tile * kHfRows + rt;
      const bool in = i < n;
      const int64_t ii = in ? i : 0;
      const float* const xs = kEp ? starts + (int64_t)(2 * e) * n : x_io;
      const float* const ys = kEp ? xs + n : y_io;
      const int64_t ro = kEp ? (int64_t)e * n : 0;                   // this episode's result row
      float* const trj = kEp && traj ? traj + (int64_t)e * T * 2 * n : traj;
      float x = 0.f, y = 0.f;
      double gx = 0.0, gy = 0.0, best = INFINITY;
      int done_at = 0;
      bool stopped = !in, succ = false;
      if (owner && in) { x = xs[i]; y = ys[i]; gx = goal[i]; gy = goal[n + i]; }
      const float2* table = owner ? bank.table<kBank>(ii) : nullptr;
      int k = 0;
      for (; k < T; ++k) {
        if (owner) {
          sbase[rt] = stopped ? make_float2(0.f, 0.f) : baseline_env(x, y, gx, gy);
          const uint32_t alive = __ballot_sync(0xffffffffu, !stopped);
          if (lane == 0) svote[(k & 1) * 4 + warp] = alive != 0u;
        }
        bar_sync(1, kHfRowThreads);
        const int* v = svote + (k & 1) * 4;
        if (!(v[0] | v[1] | v[2] | v[3])) {           // every env of the tile has stopped: release the MMA warp, leave the tile
          bar_sync(2, kHfRowMma);
          break;
        }
        const float2 b = sbase[rt];
        const float x0[4] = {b.x, b.y, 0.f, 0.f};
        hf_first_layer(m, x0, true, rt, c_lo, c_hi);
        bar_sync(2, kHfRowMma);
        mbar_wait(m.acc_ready, phase);
        phase ^= 1;
        tc_fence_after();
        hf_epilogue(m, tmem + ((uint32_t)((warp & 3) * 32) << 16), rt, cpart, c_lo, c_hi, 0);
        bar_sync(1, kHfRowThreads);
        // the other twelve warps go on to wait for the next step's actor input; sbase / part are rewritten only after barriers the
        // owners reach after they are done reading them
        if (owner) {
          if (!stopped) {
            stopped = eval_env_step(LdgTable{table}, x, y, gx, gy, hf_output(m, rt, 0), k + 1, T, best, succ);
            done_at = k + 1;
          }
          if (trj && in) {                             // coalesced plane rows: 32 consecutive envs per warp
            trj[(int64_t)(2 * k) * n + i] = x;
            trj[(int64_t)(2 * k + 1) * n + i] = y;
          }
        }
      }
      if (owner && in) {
        if (trj)
          for (int r = k; r < T; ++r) {                // the tile ended early: its envs keep their final state
            trj[(int64_t)(2 * r) * n + i] = x;
            trj[(int64_t)(2 * r + 1) * n + i] = y;
          }
        if (!kEp || e == (uint32_t)(E - 1)) {
          x_io[i] = x;
          y_io[i] = y;
        }
        success[ro + i] = succ ? 1 : 0;
        steps_out[ro + i] = done_at;
        best_out[ro + i] = best;
      }
    }
  }
  // a CTA that found no tile left never waited for its weight copies: they must land before the CTA's shared memory goes away
  if (warp == kHfRowWarps && lane == 0 && first) mbar_wait(m.w_full, 0);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
}

template <bool kBank>
__global__ void __launch_bounds__(kHfThreads, 1)
eval_f16_kernel(NetShape s, const float* __restrict__ P, const uint16_t* __restrict__ Wh, MapBank bank, const double* __restrict__ goal,
                float* __restrict__ x_io, float* __restrict__ y_io, uint8_t* __restrict__ success, int32_t* __restrict__ steps_out,
                double* __restrict__ best_out, float* __restrict__ traj, int64_t n, int T, uint32_t* __restrict__ work, uint32_t tmem_cols) {
  eval_f16_body<kBank, false>(s, P, Wh, bank, goal, nullptr, 1, x_io, y_io, success, steps_out, best_out, traj, n, T, work, tmem_cols);
}

// E episodes of every env in one launch: success, steps, best [E][n]; traj [E][T][2][n]; x_io / y_io get episode E-1's final state
template <bool kBank>
__global__ void __launch_bounds__(kHfThreads, 1)
eval_f16_episodes_kernel(NetShape s, const float* __restrict__ P, const uint16_t* __restrict__ Wh, MapBank bank, const double* __restrict__ goal,
                         const float* __restrict__ starts, int E, float* __restrict__ x_io, float* __restrict__ y_io, uint8_t* __restrict__ success,
                         int32_t* __restrict__ steps_out, double* __restrict__ best_out, float* __restrict__ traj, int64_t n, int T,
                         uint32_t* __restrict__ work, uint32_t tmem_cols) {
  eval_f16_body<kBank, true>(s, P, Wh, bank, goal, starts, E, x_io, y_io, success, steps_out, best_out, traj, n, T, work, tmem_cols);
}

static int32_t check_eval(const double* goal, const float* x, const float* y, const uint8_t* success, const int32_t* steps,
                          const double* best, const float* traj, int32_t record, int64_t n, int64_t T) {
  RTD3_CHECK_ARG(goal && x && y && success && steps && best, "null env or result array");
  RTD3_CHECK_ARG(n >= 0 && n < (1ll << 31), "n must lie in [0, 2^31)");
  RTD3_CHECK_ARG(T >= 1 && T < kEvalMaxSteps, "T must lie in [1, 2^30)");
  RTD3_CHECK_ARG((traj != nullptr) == (record != 0), "traj must be given exactly when record is set");
  return 0;
}

constexpr int64_t kEvalMaxEpisodes = 1024;

static int32_t check_episodes(int64_t E, int64_t n) {
  RTD3_CHECK_ARG(E >= 1 && E <= kEvalMaxEpisodes, "E must lie in [1, 1024]");
  RTD3_CHECK_ARG(n >= 0 && n < (1ll << 31) && E * n < (1ll << 31), "E * n must lie below 2^31");
  return 0;
}

static int32_t check_run_f16(const rtd3_env* h, int32_t hidden, int32_t layers, const float* params, const uint16_t* params_h, const uint32_t* work) {
  RTD3_CHECK_ARG(params && params_h && work, "null parameters or work counter");
  RTD3_CHECK_ARG(hidden % 32 == 0 && hidden >= 64 && hidden <= 256 && layers == 2, "needs layers == 2 and hidden in {64..256} divisible by 32");
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  return 0;
}

// The launch of either f16 kernel: dynamic shared memory, TMEM columns, and one CTA per work item up to one per SM.  Resets the
// work counter on the stream (a stream operation: captured with the launch).
struct F16Launch {
  NetShape s;
  size_t smem;
  uint32_t cols;
  int grid;
};
static int32_t f16_launch(const rtd3_env* h, const void* kern, int32_t hidden, int32_t layers, int64_t items, uint32_t* work,
                          cudaStream_t st, F16Launch& l) {
  l.s = NetShape{2, hidden, layers, 2};
  l.smem = hf_smem_bytes(hidden) + kHfRows * sizeof(float2) + 16 * sizeof(int);
  RTD3_CUDA(ensure_dyn_smem(kern, l.smem));
  l.cols = 32;
  while (l.cols < (uint32_t)hidden) l.cols <<= 1;
  l.grid = (int)(items < h->num_sms ? items : h->num_sms);
  RTD3_CUDA(cudaMemsetAsync(work, 0, sizeof(uint32_t), st));
  return 0;
}

}  // namespace rtd3

using namespace rtd3;

extern "C" {

int32_t rtd3_eval_step(rtd3_env* h, const double* goal, float* x, float* y, const float* residual, float* base, uint8_t* success,
                       int32_t* steps, double* best, float* traj, int32_t record, int64_t n, int64_t T, void* stream) {
  if (int32_t e = check_eval(goal, x, y, success, steps, best, traj, record, n, T)) return e;
  RTD3_CHECK_ARG(residual && base, "null residual or actor input");
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  if (n == 0) return 0;
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? eval_step_kernel<true> : eval_step_kernel<false>;
  kern<<<(int)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>(bank, goal, x, y, residual, base, success, steps, best, traj, n, (int)T);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_eval_run_f16(rtd3_env* h, int32_t hidden, int32_t layers, const float* params, const uint16_t* params_h, const double* goal,
                          float* x, float* y, uint8_t* success, int32_t* steps, double* best, float* traj, int32_t record, int64_t n,
                          int64_t T, uint32_t* work, void* stream) {
  if (int32_t e = check_eval(goal, x, y, success, steps, best, traj, record, n, T)) return e;
  if (int32_t e = check_run_f16(h, hidden, layers, params, params_h, work)) return e;
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? eval_f16_kernel<true> : eval_f16_kernel<false>;
  F16Launch l;
  if (int32_t e = f16_launch(h, (const void*)kern, hidden, layers, ceil_div(n, kHfRows), work, st, l)) return e;
  kern<<<l.grid, kHfThreads, l.smem, st>>>(l.s, params, params_h, bank, goal, x, y, success, steps, best, traj, n, (int)T, work, l.cols);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_eval_starts(const rtd3_mt_bank* bank, const double* region, const double* goal, int64_t E, float* starts, float* base,
                         double* state64, void* stream) {
  RTD3_CHECK_ARG(bank && bank->mt && bank->pos && region && starts && state64, "null MT bank, region, starts or state64");
  RTD3_CHECK_ARG(!base || goal, "base needs the goal");
  if (int32_t e = check_episodes(E, bank->n)) return e;
  if (bank->n == 0) return 0;
  eval_starts_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, region, goal, (int)E, starts, base, state64);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_eval_step_episodes(rtd3_env* h, const double* goal, int64_t E, float* xs, const float* residual, float* base, uint8_t* success,
                                int32_t* steps, double* best, float* traj, int32_t record, int64_t n, int64_t T, void* stream) {
  if (int32_t e = check_eval(goal, xs, xs, success, steps, best, traj, record, n, T)) return e;
  if (int32_t e = check_episodes(E, n)) return e;
  RTD3_CHECK_ARG(residual && base, "null residual or actor input");
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  if (n == 0) return 0;
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? eval_step_episodes_kernel<true> : eval_step_episodes_kernel<false>;
  kern<<<dim3((unsigned)ceil_div(n, 256), (unsigned)E), 256, 0, (cudaStream_t)stream>>>(bank, goal, xs, residual, base, success, steps, best, traj,
                                                                                         n, (int)T);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_eval_run_f16_episodes(rtd3_env* h, int32_t hidden, int32_t layers, const float* params, const uint16_t* params_h,
                                   const double* goal, const float* starts, int64_t E, float* x, float* y, uint8_t* success, int32_t* steps,
                                   double* best, float* traj, int32_t record, int64_t n, int64_t T, uint32_t* work, void* stream) {
  if (int32_t e = check_eval(goal, x, y, success, steps, best, traj, record, n, T)) return e;
  if (int32_t e = check_episodes(E, n)) return e;
  RTD3_CHECK_ARG(starts, "null start planes");
  if (int32_t e = check_run_f16(h, hidden, layers, params, params_h, work)) return e;
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? eval_f16_episodes_kernel<true> : eval_f16_episodes_kernel<false>;
  F16Launch l;
  if (int32_t e = f16_launch(h, (const void*)kern, hidden, layers, E * ceil_div(n, kHfRows), work, st, l)) return e;
  kern<<<l.grid, kHfThreads, l.smem, st>>>(l.s, params, params_h, bank, goal, starts, (int)E, x, y, success, steps, best, traj, n, (int)T,
                                           work, l.cols);
  RTD3_LAUNCHED();
  return 0;
}

}  // extern "C"
