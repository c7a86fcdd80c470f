// Demonstrations for a whole batch of envs (SURVEY.md 8 f-1 / f-2):
//   Environment.get_demonstration  - the cross-entropy-method planner, environment.py:140-179
//   Robot.process_demonstration    - robot.py:679-718 with augment_demonstration_data, robot.py:771-823
// Every env plans for itself, from its own start / goal, on its own numpy-legacy MT19937 stream, drawing exactly what the reference
// draws in the reference's order: the start state (2 doubles), iteration 0 `choice([-5, 5], 2)` per step (one 32-bit word per
// component), later iterations `normal(mean[step], std[step])` (legacy_gauss per component), 100 paths x 200 steps per iteration.
// The 100 x n rollouts of an iteration are ONE launch of the rollout kernel over 100 n "virtual envs" (path-major, so that the
// lanes of a warp - consecutive envs - touch consecutive addresses); elite selection, the float32 mean / std refit (numpy's
// operation order) and the choice of the best path stay on the device.  Paths are float32 (the reference carries float64): the
// random draws and the planner's logic are the reference's, the states agree step by step to the 1e-5 tolerance, not bit for bit.
#include "rtd3_common.cuh"
#include "rtd3_env_step.cuh"
#include "rtd3_mt.cuh"
#include "rtd3_robot.cuh"

namespace rtd3 {

// ---- planner ------------------------------------------------------------------------------------------------------------------------
// actions[(t*2 + c) * NV + p*n + i], NV = P*n.  One lane per env, warp-synchronous draws (a wrapping stream is twisted by its warp).
__global__ void __launch_bounds__(128) cem_draw_kernel(rtd3_mt_bank b, int iteration0, const float* __restrict__ mean /*[T][2][n]*/,
                                                       const float* __restrict__ sd, float* __restrict__ actions, int P, int T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = b.n;
  const bool active = i < n;
  if (!__any_sync(0xffffffffu, active)) return;
  const int64_t ii = active ? i : 0;
  const int64_t NV = (int64_t)P * n;
  MtStream s{b.mt + ii, n, active ? b.pos[ii] : 0};
  int hg = active ? b.has_gauss[ii] : 0;
  double sp = active ? b.gauss[ii] : 0.0;
  for (int p = 0; p < P; ++p) {
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        float v;
        if (iteration0) {
          // np.random.choice([-5, 5], 2): randint(0, 2) per component = one 32-bit word masked with 1 (always accepted)
          const uint32_t w = mt_next_u32_warp(s, active);
          v = (w & 1u) ? kMaxAction : -kMaxAction;
        } else {
          // np.random.normal(mean[step], std[step]): loc + scale * legacy_gauss() in float64, stored as float32 (environment.py:159-160)
          const double z = mt_gauss_warp(s, active, hg, sp);
          const int64_t q = (int64_t)(t * 2 + c) * n + ii;
          v = (float)__dadd_rn((double)mean[q], __dmul_rn((double)sd[q], z));
        }
        if (active) actions[(int64_t)(t * 2 + c) * NV + (int64_t)p * n + i] = v;
      }
    }
  }
  if (!active) return;
  b.pos[i] = s.pos;
  b.has_gauss[i] = hg;
  b.gauss[i] = sp;
}

__global__ void cem_spread_kernel(const float* __restrict__ sx, const float* __restrict__ sy, float* __restrict__ x, float* __restrict__ y,
                                  int64_t n, int64_t NV) {
  const int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= NV) return;
  x[v] = sx[v % n];
  y[v] = sy[v % n];
}

// compute_reward of every path (environment.py:182-183: -||path[-1] - goal||, float32 state against the float64 goal), the `E` best in
// ascending order (np.argsort(...)[-E:]) and the best one (np.argmax).  One thread per env.
__global__ void cem_select_kernel(const float* __restrict__ x, const float* __restrict__ y, const double* __restrict__ goal, int64_t n, int P,
                                  int E, double* __restrict__ rewards /*[n][P]*/, int32_t* __restrict__ elite /*[n][E]*/,
                                  int32_t* __restrict__ best /*[n]*/) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double* r = rewards + i * P;
  const double gx = goal[i], gy = goal[n + i];
  double top = -INFINITY;
  int arg = 0;
  for (int p = 0; p < P; ++p) {
    const int64_t v = (int64_t)p * n + i;
    const double rw = -norm2_np(__dsub_rn((double)x[v], gx), __dsub_rn((double)y[v], gy));
    r[p] = rw;
    if (rw > top) { top = rw; arg = p; }                 // first maximum, like np.argmax
  }
  best[i] = arg;
  // E largest, written in ascending order of reward; among equal rewards the later index ranks higher (a stable ascending sort)
  double bound = INFINITY;
  int bound_idx = P;
  for (int e = E - 1; e >= 0; --e) {
    double m = -INFINITY;
    int mi = -1;
    for (int p = 0; p < P; ++p) {
      const double rw = r[p];
      const bool below = rw < bound || (rw == bound && p < bound_idx);
      if (below && (rw > m || (rw == m && p > mi))) { m = rw; mi = p; }
    }
    elite[i * E + e] = mi;
    bound = m;
    bound_idx = mi;
  }
}

// mean / std over the elite paths per (step, component) in float32 with numpy's operation order (environment.py:172-173:
// np.mean / np.std over axis 0 of a float32 array = sequential adds in gather order, one division; std = sqrt(mean(|x - mean|^2))).
__global__ void cem_refit_kernel(const float* __restrict__ actions, const int32_t* __restrict__ elite, int64_t n, int P, int T, int E,
                                 float* __restrict__ mean, float* __restrict__ sd) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // (t*2 + c) * n + i
  if (g >= (int64_t)T * 2 * n) return;
  const int64_t tc = g / n, i = g - tc * n;
  const int64_t NV = (int64_t)P * n;
  float a[16];
  float sum = 0.f;
  for (int e = 0; e < E; ++e) {
    a[e] = actions[tc * NV + (int64_t)elite[i * E + e] * n + i];
    sum = e == 0 ? a[0] : __fadd_rn(sum, a[e]);
  }
  const float mu = __fdiv_rn(sum, (float)E);
  float ss = 0.f;
  for (int e = 0; e < E; ++e) {
    const float d = __fsub_rn(a[e], mu);
    const float d2 = __fmul_rn(d, d);
    ss = e == 0 ? d2 : __fadd_rn(ss, d2);
  }
  mean[g] = mu;
  sd[g] = __fsqrt_rn(__fdiv_rn(ss, (float)E));
}

__global__ void cem_gather_kernel(const float* __restrict__ actions, const int32_t* __restrict__ best, int64_t n, int P, int T,
                                  float* __restrict__ best_actions /*[T][2][n]*/) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= (int64_t)T * 2 * n) return;
  const int64_t tc = g / n, i = g - tc * n;
  best_actions[g] = actions[tc * (int64_t)P * n + (int64_t)best[i] * n + i];
}

// demonstration_states = planning_paths[-1, best, 0:T] (the start state and the first T-1 states of the path),
// demonstration_actions = planning_actions[-1, best]                      environment.py:176-179
__global__ void cem_pack_kernel(const float* __restrict__ sx, const float* __restrict__ sy, const float* __restrict__ traj /*[T][2][n]*/,
                                const float* __restrict__ best_actions, int64_t n, int T, float* __restrict__ demo_states /*[n][T][2]*/,
                                float* __restrict__ demo_actions) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // t * n + i
  if (g >= (int64_t)T * n) return;
  const int64_t t = g / n, i = g - t * n;
  const float px = t == 0 ? sx[i] : traj[((t - 1) * 2 + 0) * n + i], py = t == 0 ? sy[i] : traj[((t - 1) * 2 + 1) * n + i];
  reinterpret_cast<float2*>(demo_states)[i * T + t] = make_float2(px, py);
  reinterpret_cast<float2*>(demo_actions)[i * T + t] = make_float2(best_actions[(t * 2 + 0) * n + i], best_actions[(t * 2 + 1) * n + i]);
}

// ---- process_demonstration ----------------------------------------------------------------------------------------------------------
// Appends the demonstration's T states and its augmentations (robot.py:771-823: per transition five interpolated states and the
// current state, each plus N(0, 2.5) noise, finally the noisy last state; the action noise is drawn as well - the stream must move
// as the reference's does - but augmented actions are never read again) to env i's demonstration set.  One lane per env.
__global__ void __launch_bounds__(128) demo_augment_kernel(rtd3_mt_bank b, const float* __restrict__ demo_states /*[n][T][2]*/, int T,
                                                           double* __restrict__ sets /*[n][cap][2]*/, int32_t* __restrict__ count, int64_t cap,
                                                           int augments, int interp, double noise_level) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = b.n;
  const bool active = i < n;
  if (!__any_sync(0xffffffffu, active)) return;
  const int64_t ii = active ? i : 0;
  MtStream s{b.mt + ii, n, active ? b.pos[ii] : 0};
  int hg = active ? b.has_gauss[ii] : 0;
  double sp = active ? b.gauss[ii] : 0.0;
  const float2* S = reinterpret_cast<const float2*>(demo_states) + ii * T;
  double2* out = reinterpret_cast<double2*>(sets) + ii * cap;
  int m = active ? count[ii] : 0;
  if (active)
    for (int t = 0; t < T; ++t) out[m + t] = make_double2((double)S[t].x, (double)S[t].y);     // self.demonstration_states.extend(...)
  m += T;
  // np.random.normal(0, noise_level, shape (2,)): 0 + noise_level * gauss per component
  auto noise2 = [&](double& zx, double& zy) {
    zx = __dadd_rn(0.0, __dmul_rn(noise_level, mt_gauss_warp(s, active, hg, sp)));
    zy = __dadd_rn(0.0, __dmul_rn(noise_level, mt_gauss_warp(s, active, hg, sp)));
  };
  for (int a = 0; a < augments; ++a) {
    for (int t = 0; t + 1 < T; ++t) {
      const float2 cur = S[t], nxt = S[t + 1];
      double zx, zy, ux, uy;
      for (int st = 1; st <= interp; ++st) {
        // fraction is a Python float: weak against the float32 states, the interpolation stays float32 (NEP 50)
        const float fr = (float)((double)st / (double)(interp + 1));
        const float sxv = __fadd_rn(cur.x, __fmul_rn(fr, __fsub_rn(nxt.x, cur.x))), syv = __fadd_rn(cur.y, __fmul_rn(fr, __fsub_rn(nxt.y, cur.y)));
        noise2(zx, zy);
        noise2(ux, uy);                                  // the action's noise
        if (active) out[m] = make_double2(__dadd_rn((double)sxv, zx), __dadd_rn((double)syv, zy));
        ++m;
      }
      noise2(zx, zy);
      noise2(ux, uy);
      if (active) out[m] = make_double2(__dadd_rn((double)cur.x, zx), __dadd_rn((double)cur.y, zy));
      ++m;
    }
    double zx, zy, ux, uy;
    noise2(zx, zy);
    noise2(ux, uy);
    if (active) out[m] = make_double2(__dadd_rn((double)S[T - 1].x, zx), __dadd_rn((double)S[T - 1].y, zy));
    ++m;
  }
  if (!active) return;
  count[i] = m;
  b.pos[i] = s.pos;
  b.has_gauss[i] = hg;
  b.gauss[i] = sp;
}

// Counting sort of env blockIdx.x's states into the cells of its 25 x 25 grid (see nearest_demo_env_sq, rtd3_robot.cuh).
__global__ void __launch_bounds__(256) demo_grid_build_kernel(const double* __restrict__ sets, const int32_t* __restrict__ count, int64_t cap,
                                                              double* __restrict__ sorted, int32_t* __restrict__ cells /*[n][kEnvCells+1]*/) {
  __shared__ int cnt[kEnvCells + 1];
  const int64_t i = blockIdx.x;
  const int m = count[i];
  const double2* in = reinterpret_cast<const double2*>(sets) + i * cap;
  double2* out = reinterpret_cast<double2*>(sorted) + i * cap;
  int32_t* cs = cells + i * (kEnvCells + 1);
  for (int c = threadIdx.x; c <= kEnvCells; c += blockDim.x) cnt[c] = 0;
  __syncthreads();
  for (int k = threadIdx.x; k < m; k += blockDim.x) {
    const double2 p = in[k];
    atomicAdd(&cnt[env_cell_coord(p.x) * kEnvGrid + env_cell_coord(p.y)], 1);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int run = 0;
    for (int c = 0; c < kEnvCells; ++c) {
      const int k = cnt[c];
      cnt[c] = run;
      cs[c] = run;
      run += k;
    }
    cs[kEnvCells] = run;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < m; k += blockDim.x) {
    const double2 p = in[k];
    out[atomicAdd(&cnt[env_cell_coord(p.x) * kEnvGrid + env_cell_coord(p.y)], 1)] = p;
  }
}

// The T-1 transitions of every env's demonstration into the replay ring (robot.py:700-716): reward = compute_reward([next_state])
// - GOAL_REWARD inside the goal radius, else -distance, plus 10 x (-distance to the nearest demonstration state) once demo_flag is
// set -, done on the last one.  Rows are laid out env-major behind the ring's row counter; when more rows arrive than the ring holds,
// the rows a sequential push would have kept (the last `capacity`) are written.
__global__ void demo_rows_kernel(const float* __restrict__ demo_states, const float* __restrict__ demo_actions, int T, int64_t n,
                                 const double* __restrict__ goal, const uint8_t* __restrict__ demo_flag, const double* __restrict__ env_pts,
                                 const int32_t* __restrict__ env_cells, const int32_t* __restrict__ env_count, int64_t cap, ReplayRing ring) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // i * (T-1) + t
  const int64_t rows = n * (T - 1);
  if (g >= rows) return;
  const int64_t i = g / (T - 1), t = g - i * (T - 1);
  const float2 s = reinterpret_cast<const float2*>(demo_states)[i * T + t], s2 = reinterpret_cast<const float2*>(demo_states)[i * T + t + 1];
  const float2 a = reinterpret_cast<const float2*>(demo_actions)[i * T + t];
  const double gd = norm2_np(__dsub_rn((double)s2.x, goal[i]), __dsub_rn((double)s2.y, goal[n + i]));
  double reward;
  if (-gd >= -kGoalRadius) {
    reward = kGoalReward;
  } else {
    double prox = 0.0;
    if (demo_flag[i] && env_count[i] > 0)
      prox = -sqrt(nearest_demo_env_sq((double)s2.x, (double)s2.y, reinterpret_cast<const double2*>(env_pts) + i * cap,
                                       env_cells + i * (kEnvCells + 1)));
    reward = __dadd_rn(-gd, __dmul_rn(10.0, prox));
  }
  if (rows > ring.capacity && g < rows - ring.capacity) return;            // overwritten by later rows of the same push
  const unsigned long long base = *ring.total;
  const int64_t p = (int64_t)((base + (unsigned long long)g) % (unsigned long long)ring.capacity);
  ring.s[p] = s;
  ring.a[p] = a;
  ring.r[p] = (float)reward;
  ring.s2[p] = s2;
  ring.notdone[p] = (t == T - 2) ? 0.f : 1.f;
}

__global__ void add_u64_kernel(unsigned long long* p, unsigned long long by) { p[0] += by; }

}  // namespace rtd3

using namespace rtd3;

extern "C" {

int32_t rtd3_env_get_demonstration(rtd3_env* h, const rtd3_mt_bank* bank, const double* region, const double* goal, const rtd3_cem_workspace* w,
                                   int32_t iterations, int32_t paths, int32_t steps, int32_t elites, int32_t it_begin, int32_t it_end,
                                   int32_t finish, float* demo_states, float* demo_actions, void* stream) {
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(bank && bank->mt && bank->pos && bank->has_gauss && bank->gauss && bank->n >= 0, "bad MT19937 bank");
  RTD3_CHECK_ARG(region && goal && w, "null argument");
  RTD3_CHECK_ARG(w->actions && w->x && w->y && w->start_x && w->start_y && w->rewards && w->elite && w->best && w->mean && w->std &&
                     w->best_actions && w->traj,
                 "incomplete workspace");
  RTD3_CHECK_ARG(iterations >= 1 && paths >= 1 && steps >= 2 && elites >= 1 && elites <= 16 && elites <= paths, "bad planner sizes (elites <= 16)");
  RTD3_CHECK_ARG(it_begin >= 0 && it_begin <= it_end && it_end <= iterations, "bad iteration range");
  RTD3_CHECK_ARG(!finish || (demo_states && demo_actions), "finish needs the output arrays");
  const int64_t n = bank->n;
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t NV = (int64_t)paths * n;
  RTD3_CHECK_ARG(NV < (1ll << 31), "paths * n must stay below 2^31");
  if (it_begin == 0) {
    // robot_current_state = self.get_random_robot_init_state()   environment.py:151 (a draw that does not move the robot)
    const int32_t rc = rtd3_env_reset(bank, region, nullptr, -1, w->start_x, w->start_y, w->start64, stream);
    if (rc) return rc;
  }
  for (int it = it_begin; it < it_end; ++it) {
    cem_draw_kernel<<<(int)ceil_div(n, 128), 128, 0, st>>>(*bank, it == 0 ? 1 : 0, w->mean, w->std, w->actions, paths, steps);
    RTD3_LAUNCHED();
    cem_spread_kernel<<<(int)ceil_div(NV, 256), 256, 0, st>>>(w->start_x, w->start_y, w->x, w->y, n, NV);
    RTD3_LAUNCHED();
    const int32_t rc = rtd3_env_rollout(h, w->x, w->y, w->actions, nullptr, NV, steps, stream);
    if (rc) return rc;
    cem_select_kernel<<<(int)ceil_div(n, 128), 128, 0, st>>>(w->x, w->y, goal, n, paths, elites, w->rewards, w->elite, w->best);
    RTD3_LAUNCHED();
    cem_refit_kernel<<<(int)ceil_div((int64_t)steps * 2 * n, 256), 256, 0, st>>>(w->actions, w->elite, n, paths, steps, elites, w->mean, w->std);
    RTD3_LAUNCHED();
  }
  if (finish) {
    cem_gather_kernel<<<(int)ceil_div((int64_t)steps * 2 * n, 256), 256, 0, st>>>(w->actions, w->best, n, paths, steps, w->best_actions);
    RTD3_LAUNCHED();
    cem_spread_kernel<<<(int)ceil_div(n, 256), 256, 0, st>>>(w->start_x, w->start_y, w->x, w->y, n, n);
    RTD3_LAUNCHED();
    const int32_t rc = rtd3_env_rollout(h, w->x, w->y, w->best_actions, w->traj, n, steps, stream);
    if (rc) return rc;
    cem_pack_kernel<<<(int)ceil_div((int64_t)steps * n, 256), 256, 0, st>>>(w->start_x, w->start_y, w->traj, w->best_actions, n, steps, demo_states,
                                                                            demo_actions);
    RTD3_LAUNCHED();
  }
  return 0;
}

int32_t rtd3_robot_process_demonstration(const rtd3_mt_bank* bank, const double* goal, const uint8_t* demo_flag, const float* demo_states,
                                         const float* demo_actions, int32_t steps, double* sets, int32_t* set_count, double* sorted,
                                         int32_t* cells, int64_t cap, int32_t augments, int32_t interpolation, double noise_level, float* rp_s,
                                         float* rp_a, float* rp_r, float* rp_s2, float* rp_notdone, int64_t capacity, uint64_t* rp_total,
                                         void* stream) {
  RTD3_CHECK_ARG(bank && bank->mt && bank->pos && bank->has_gauss && bank->gauss && bank->n >= 0, "bad MT19937 bank");
  RTD3_CHECK_ARG(goal && demo_flag && demo_states && demo_actions && sets && set_count && sorted && cells, "null argument");
  RTD3_CHECK_ARG(steps >= 2 && augments >= 0 && interpolation >= 0, "bad sizes");
  RTD3_CHECK_ARG(cap >= (int64_t)steps + (int64_t)augments * ((int64_t)(steps - 1) * (interpolation + 1) + 1),
                 "cap is smaller than one demonstration with its augmentations");
  RTD3_CHECK_ARG((rp_s == nullptr) || (rp_a && rp_r && rp_s2 && rp_notdone && rp_total && capacity > 0), "bad replay ring");
  const int64_t n = bank->n;
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // (the caller guarantees count[i] + states of this demonstration <= cap for every env: counts are device-side)
  demo_augment_kernel<<<(int)ceil_div(n, 128), 128, 0, st>>>(*bank, demo_states, steps, sets, set_count, cap, augments, interpolation, noise_level);
  RTD3_LAUNCHED();
  demo_grid_build_kernel<<<(int)n, 256, 0, st>>>(sets, set_count, cap, sorted, cells);
  RTD3_LAUNCHED();
  if (rp_s) {
    const ReplayRing ring{(float2*)rp_s, (float2*)rp_a, rp_r, (float2*)rp_s2, rp_notdone, capacity, 0, (unsigned long long*)rp_total};
    const int64_t rows = n * (steps - 1);
    demo_rows_kernel<<<(int)ceil_div(rows, 256), 256, 0, st>>>(demo_states, demo_actions, steps, n, goal, demo_flag, sorted, cells, set_count, cap, ring);
    RTD3_LAUNCHED();
    add_u64_kernel<<<1, 1, 0, st>>>((unsigned long long*)rp_total, (unsigned long long)rows);
    RTD3_LAUNCHED();
  }
  return 0;
}

int32_t rtd3_robot_demo_grids(const double* sets, const int32_t* set_count, int64_t cap, int64_t n, double* sorted, int32_t* cells,
                              void* stream) {
  RTD3_CHECK_ARG(sets && set_count && sorted && cells, "null argument");
  RTD3_CHECK_ARG(cap >= 1, "cap must be >= 1");
  RTD3_CHECK_ARG(n >= 0 && n < (1ll << 31), "n must lie in [0, 2^31)");
  if (n == 0) return 0;
  demo_grid_build_kernel<<<(int)n, 256, 0, (cudaStream_t)stream>>>(sets, set_count, cap, sorted, cells);
  RTD3_LAUNCHED();
  return 0;
}

}  // extern "C"
