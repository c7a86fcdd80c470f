// One tick of the batched driver loop (robot-learning.py:66-101, training branch) in TWO launches around the actor forward:
//   rtd3_tick_pre  : get_next_action_type + reset state machine (robot.py:443-506), actor input = state - goal (robot.py:556)
//   [actor forward : rtd3_mlp_forward / rtd3_mlp_forward_tf32]
//   rtd3_tick_post : action = clip(baseline + residual + noise) (robot.py:560-567), Environment.step (environment.py:98-127),
//                    process_transition incl. reward / stuck / done / replay push (robot.py:645-675), the money counters
//                    (robot-learning.py:78, 86, 99) and Environment.reset for the envs whose tick is a 'reset' (environment.py:130-137)
// The same device functions as the one-hook-per-launch entry points (rtd3_robot.cuh, rtd3_env_step.cuh) are used, in the same
// order per env, so a fused tick leaves every array bit-identical to the sequence
//   next_action_type, baseline, forward, compose_action, env_step, robot_transition, env_reset(mask = type 2), trainer_tally
// (tests/test_tick_gpu.py).  At 8 192 envs per GPU that sequence is ten dependent launches of 3-6 us each around a 15 us forward:
// launch latency, not arithmetic, was the tick.
#include "rtd3_common.cuh"
#include "rtd3_env_step.cuh"
#include "rtd3_mt.cuh"
#include "rtd3_robot.cuh"
#include "rtd3_tc_f16.cuh"

namespace rtd3 {

// Tick types: 0 'step', 1 'demo', 2 'reset' (what get_next_action_type returned, and - with the scheduler - the purchase went through),
// 3 training budget exhausted: environment.reset() and on to testing (robot-learning.py:70-80), 4 not affordable: nothing happens this
// tick (robot-learning.py:86-87, 93-94, 96), 5 a test step (robot-learning.py:104-117), 6 the env's run is over.
constexpr int kTypeSwitch = RTD3_TICK_TYPE_SWITCH, kTypeSkip = RTD3_TICK_TYPE_SKIP, kTypeTest = RTD3_TICK_TYPE_TEST,
              kTypeIdle = RTD3_TICK_TYPE_IDLE;
constexpr double kStartingMoney = 100.0, kCostStep = 0.01, kCostCpuSecond = 0.03;   // constants.py:43-45
constexpr long long kCostDemo = 20, kCostReset = 5;                                   // constants.py:46-47
constexpr double kTestDistance = 5.0;                                                 // constants.py:50

// calculate_remaining_money (robot-learning.py:45-50) with the wall clock replaced by ticks * tick_seconds: Python adds the two
// integer products first, then the two float products, left to right
__device__ __forceinline__ double money_remaining(long long demos, long long resets, long long steps, uint64_t ticks, double tick_seconds) {
  const double cpu = __dmul_rn((double)ticks, tick_seconds);
  const double spent = __dadd_rn(__dadd_rn((double)(demos * kCostDemo + resets * kCostReset), __dmul_rn((double)steps, kCostStep)),
                                 __dmul_rn(cpu, kCostCpuSecond));
  return __dsub_rn(kStartingMoney, spent);
}

// The training / testing dispatch of update(dt) (robot-learning.py:66-103) for env i at tick `tick_index` (ticks elapsed before this
// one).  Without the scheduler arrays (t.mode == NULL) it is get_next_action_type alone: every purchase goes through.
__device__ __forceinline__ int schedule_env(const rtd3_tick_state& t, const int64_t i, const uint64_t tick_index, bool& upd) {
  upd = false;
  if (t.mode) {
    const int mode = t.mode[i];
    if (mode == 1) return kTypeTest;
    if (mode == 2) return kTypeIdle;
  }
  int type = action_type_env(t.num_episodes, t.demo_flag, t.plan_index, t.path_length, t.goal_reached, t.stuck_flag, t.noise_scale, i, upd);
  if (!t.mode) return type;
  const double money = money_remaining(t.demos_bought[i], t.resets_bought[i], t.steps_bought[i], tick_index, t.tick_seconds);
  if (money < 0.0) {                                       // robot-learning.py:70-80
    if (money < -1.0) t.penalty[i] = 1;
    t.mode[i] = 1;
    return kTypeSwitch;
  }
  if (type == 2) return money >= (double)kCostReset ? 2 : kTypeSkip;
  if (type == 1) {
    if (!(money >= (double)kCostDemo)) return kTypeSkip;
    t.demos_bought[i] += 1;                                // robot-learning.py:92 (the demonstration itself is the caller's job)
    return 1;
  }
  return money >= kCostStep ? 0 : kTypeSkip;
}

__global__ void __launch_bounds__(256) tick_pre_kernel(rtd3_tick_state t) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = t.n;
  bool upd = false;
  if (i < n) {
    t.type[i] = (int8_t)schedule_env(t, i, t.tick_counter ? t.tick_counter[0] : 0ull, upd);
    t.update[i] = upd ? 1 : 0;
    reinterpret_cast<float2*>(t.base)[i] = baseline_env(t.x[i], t.y[i], t.goal[i], t.goal[n + i]);
  }
  const uint32_t ended = __ballot_sync(0xffffffffu, upd);
  if (ended && (threadIdx.x & 31) == 0) atomicAdd(t.any_update, __popc(ended));
  // tick counter: every thread of this kernel reads word 0 (ticks completed), so the advanced value goes to word 1, which
  // tick_post_kernel reads (all threads) and copies back to word 0 - no kernel writes a word its other blocks read
  if (i == 0 && t.tick_counter) t.tick_counter[1] = t.tick_counter[0] + 1ull;
}

// Second half of a tick for env i (`in`: i < n; whole warps call this): compose the action from the actor's residual, step,
// process_transition, money counters, masked reset.  tick_index keys the Philox noise.
template <bool kAllowSweep>
__device__ __forceinline__ void tick_post_env(const rtd3_tick_state& t, const float2* __restrict__ table, const int64_t i, const bool in,
                                              const int type, const float2 res, const double* __restrict__ unit_noise, const int noise_mode,
                                              const uint64_t tick_index) {
  const int64_t n = t.n;
  const int64_t ii = in ? i : 0;
  const bool live = in && type == 0;
  const bool testing = in && type == kTypeTest;
  const bool resets = in && (type == 2 || type == kTypeSwitch);
  const float x = t.x[ii], y = t.y[ii];
  // the 'reset' envs' draws: loads issued now, consumed after the transition work (they do not depend on it)
  ResetLoads rl = reset_load_warp(t.env_bank, t.region, resets, i);
  const int64_t steps_before = (in && type == 0) ? t.steps_bought[i] : 0, resets_before = (in && type == 2) ? t.resets_bought[i] : 0;
  // get_next_action_training: envs that do not step in this tick get a null action (robot-learning.py:82-95)
  float ax = 0.f, ay = 0.f;
  if (live) {
    double zx = 0.0, zy = 0.0;
    if (noise_mode == RTD3_TICK_NOISE_GIVEN) { zx = unit_noise[i]; zy = unit_noise[n + i]; }
    else if (noise_mode == RTD3_TICK_NOISE_PHILOX) philox_normal2(t.philox_seed, tick_index, (uint64_t)i, zx, zy);
    double cx, cy;
    compose_env(x, y, t.goal[i], t.goal[n + i], res, noise_mode != RTD3_TICK_NOISE_NONE, zx, zy,
                noise_mode != RTD3_TICK_NOISE_NONE ? t.noise_scale[i] : 0.0, cx, cy);
    ax = (float)cx;
    ay = (float)cy;
  } else if (testing) {                                   // get_next_action_testing: no exploration noise (robot.py:572-595)
    double cx, cy;
    compose_env(x, y, t.goal[i], t.goal[n + i], res, false, 0.0, 0.0, 0.0, cx, cy);
    ax = (float)cx;
    ay = (float)cy;
  }
  // Environment.step
  float nx, ny;
  step_one<true>(LdgTable{table}, x, y, ax, ay, nx, ny);
  // process_transition (reward, stuck ring, done, compacted replay push)
  const RobotState st{t.goal, t.hist, t.hist_count, t.hist_head, t.goal_reached, t.stuck_flag, t.demo_flag, t.plan_index, t.path_length,
                      t.env_demo_pts, t.env_demo_cells, t.env_demo_count, t.env_demo_cap};
  const ReplayRing ring{(float2*)t.rp_s, (float2*)t.rp_a, t.rp_r, (float2*)t.rp_s2, t.rp_notdone, t.capacity, 0,
                        (unsigned long long*)t.rp_total};
  transition_env<kAllowSweep>(st, x, y, ax, ay, nx, ny, live, i, n, t.demo, t.demo_list_start, t.demo_list, t.num_demo, t.reward, t.reward64, t.done,
                              ring, true);
  if (in) {
    t.ax[i] = ax;
    t.ay[i] = ay;
    if (t.prev_x) { t.prev_x[i] = x; t.prev_y[i] = y; }
    t.x[i] = nx;
    t.y[i] = ny;
    if (type == 0) t.steps_bought[i] = steps_before + 1;
    else if (type == 2) t.resets_bought[i] = resets_before + 1;
  }
  if (testing) {                                          // robot-learning.py:107-117
    const double dist = norm2_np(__dsub_rn((double)nx, t.goal[i]), __dsub_rn((double)ny, t.goal[n + i]));
    const int ticks = t.test_ticks[i] + 1;
    t.test_ticks[i] = ticks;
    bool over = false;
    if (dist <= kTestDistance) { t.test_success[i] = 1; over = true; }
    if (dist < t.test_best[i]) t.test_best[i] = dist;
    if ((int64_t)ticks >= t.test_timeout_ticks) over = true;
    if (over) t.mode[i] = 2;
  }
  // Environment.reset where the tick is a 'reset' (warp-synchronous: wrapping MT19937 streams are twisted by the whole warp)
  reset_finish_warp(t.env_bank, resets, i, rl, t.x, t.y, t.state64);
}

// kBank: env i steps on its own map of the bank, else on map 0
template <bool kBank = false>
__global__ void __launch_bounds__(256, 2) tick_post_kernel(rtd3_tick_state t, const float* __restrict__ residual /*[n][2]*/,
                                                           const double* __restrict__ unit_noise /*[2][n], mode 1*/, int noise_mode,
                                                           MapBank bank) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool in = i < t.n;
  const int64_t ii = in ? i : 0;
  // the Philox noise of a tick is keyed by the number of ticks run including this one (word 1 of the counter, see tick_pre_kernel)
  const uint64_t tick_index = t.tick_counter ? t.tick_counter[1] : 0ull;
  tick_post_env<true>(t, bank.table<kBank>(ii), i, in, in ? (int)t.type[ii] : 1, reinterpret_cast<const float2*>(residual)[ii], unit_noise,
                      noise_mode, tick_index);
  if (i == 0 && t.tick_counter) t.tick_counter[0] = tick_index;
}

// ---- K ticks in ONE launch (actor 2 -> H -> H -> 2 on the f16 resident-weight forward, rtd3_tc_f16.cuh) -------------------------
// Envs are independent, so a CTA can run all K ticks of its 128-env tile without talking to any other CTA: the actor's hidden
// weight is loaded into shared memory once per launch instead of once per tick, and a tick costs no launch at all.  Per tick:
//   owner threads (warps 0-3, one env each): state machine + actor input  -> barrier
//   16 row warps: first layer into X                                       -> barrier with the MMA warp -> products -> epilogue -> barrier
//   owner threads: residual from the partial sums, then tick_post_env (action, step, transition, replay push, reset)
// Same device functions, same order per env as rtd3_tick_pre / rtd3_mlp_forward_f16 / rtd3_tick_post: bit-identical arrays
// (tests/test_tick_gpu.py).  Needs candidate lists or no demonstration states (no block-wide sweep here) and Philox or no noise.
template <bool kBank = false>
__global__ void __launch_bounds__(kHfThreads, 1)
tick_f16_kernel(rtd3_tick_state t, NetShape s, const float* __restrict__ P, const uint16_t* __restrict__ Wh, int noise_mode, int K,
                uint64_t tick_base, uint32_t tmem_cols, MapBank bank) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int H = s.hid;
  const HfSmem m = hf_carve(smem_raw, H);
  float2* sbase = reinterpret_cast<float2*>(m.extra);                 // [128] actor input of the tile's envs
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rt = (warp & 3) * 32 + lane, cpart = warp >> 2;
  int c_lo, c_hi;
  hf_columns(H, cpart, c_lo, c_hi);
  const int64_t n = t.n;
  const int tiles = (int)((n + kHfRows - 1) / kHfRows);
  const uint32_t tmem = hf_setup(m, s, P, Wh, tmem_cols);
  const uint32_t idesc = hf_idesc(H);

  if (warp == kHfRowWarps) {
    bool first = true;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x)
      for (int k = 0; k < K; ++k) {
        bar_sync(2, kHfRowMma);                       // X of this (tile, tick) is in shared memory, the accumulator has been drained
        if (lane == 0) {
          if (first) mbar_wait(m.w_full, 0);
          hf_issue_tile(m, H, tmem, idesc, m.acc_ready);
        }
        first = false;
        __syncwarp();
      }
  } else {
    const bool owner = cpart == 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      const int64_t i = (int64_t)tile * kHfRows + rt;
      const bool in = i < n;
      for (int k = 0; k < K; ++k) {
        int type = 1;
        if (owner) {
          bool upd = false;
          float2 base = make_float2(0.f, 0.f);
          if (in) {
            type = schedule_env(t, i, tick_base + (uint64_t)k, upd);
            t.type[i] = (int8_t)type;
            t.update[i] = upd ? 1 : 0;
            base = baseline_env(t.x[i], t.y[i], t.goal[i], t.goal[n + i]);
            reinterpret_cast<float2*>(t.base)[i] = base;
          }
          const uint32_t ended = __ballot_sync(0xffffffffu, upd);
          if (ended && lane == 0) atomicAdd(t.any_update, __popc(ended));
          sbase[rt] = base;
        }
        bar_sync(1, kHfRowThreads);
        const float2 b = sbase[rt];
        const float x0[4] = {b.x, b.y, 0.f, 0.f};
        hf_first_layer(m, x0, true, rt, c_lo, c_hi);
        bar_sync(2, kHfRowMma);
        mbar_wait(m.acc_ready, phase);
        phase ^= 1;
        tc_fence_after();
        hf_epilogue(m, tmem + ((uint32_t)((warp & 3) * 32) << 16), rt, cpart, c_lo, c_hi, 0);
        bar_sync(1, kHfRowThreads);
        // the other twelve warps go on to wait for the next tick's actor input; sbase / part are rewritten only after barriers the
        // owners reach after they are done reading them
        if (owner) tick_post_env<false>(t, bank.table<kBank>(in ? i : 0), i, in, type, hf_output(m, rt, 0), nullptr, noise_mode,
                                        tick_base + (uint64_t)k + 1ull);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
  if (blockIdx.x == 0 && tid == 0 && t.tick_counter) t.tick_counter[0] = t.tick_counter[1] = tick_base + (uint64_t)K;   // as K ticks leave it
}

static int32_t check_state(const rtd3_tick_state* t) {
  RTD3_CHECK_ARG(t, "null tick state");
  RTD3_CHECK_ARG(t->n >= 0, "negative n");
  RTD3_CHECK_ARG(t->x && t->y && t->goal && t->region, "null env array");
  RTD3_CHECK_ARG(t->env_bank.mt && t->env_bank.pos && t->env_bank.n == t->n, "env MT19937 bank missing or of another size");
  RTD3_CHECK_ARG(t->num_episodes && t->demo_flag && t->plan_index && t->path_length && t->goal_reached && t->stuck_flag && t->noise_scale,
                 "null robot episode state");
  RTD3_CHECK_ARG(t->hist && t->hist_count && t->hist_head && t->type && t->update && t->any_update, "null robot state");
  RTD3_CHECK_ARG(t->base && t->ax && t->ay && t->reward && t->done, "null tick output");
  RTD3_CHECK_ARG((t->prev_x == nullptr) == (t->prev_y == nullptr), "prev_x / prev_y go together");
  RTD3_CHECK_ARG(t->num_demo >= 0 && (t->num_demo == 0 || t->demo), "demo set missing");
  RTD3_CHECK_ARG((t->demo_list_start == nullptr) == (t->demo_list == nullptr), "demo_list_start and demo_list go together");
  RTD3_CHECK_ARG(t->rp_s && t->rp_a && t->rp_r && t->rp_s2 && t->rp_notdone && t->rp_total && t->capacity > 0 && t->n <= t->capacity,
                 "bad replay ring");
  RTD3_CHECK_ARG(t->steps_bought && t->resets_bought, "null money counters");
  RTD3_CHECK_ARG(!t->env_demo_pts || (t->env_demo_cells && t->env_demo_count && t->env_demo_cap > 0), "incomplete per-env demonstration sets");
  if (t->mode) {
    RTD3_CHECK_ARG(t->demos_bought && t->test_ticks && t->test_best && t->test_success && t->penalty, "scheduler arrays missing (mode is set)");
    RTD3_CHECK_ARG(t->tick_counter, "the scheduler charges time per tick: tick_counter is required");
    RTD3_CHECK_ARG(t->tick_seconds >= 0.0 && t->test_timeout_ticks > 0, "bad tick_seconds / test_timeout_ticks");
  }
  return 0;
}

}  // namespace rtd3

using namespace rtd3;

extern "C" {

int32_t rtd3_tick_pre(const rtd3_tick_state* t, void* stream) {
  if (int32_t e = check_state(t)) return e;
  if (t->n == 0) return 0;
  tick_pre_kernel<<<(int)ceil_div(t->n, 256), 256, 0, (cudaStream_t)stream>>>(*t);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_tick_post(rtd3_env* h, const rtd3_tick_state* t, const float* residual, const double* unit_noise, int32_t noise_mode,
                       void* stream) {
  if (int32_t e = check_state(t)) return e;
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(residual, "null residual");
  RTD3_CHECK_ARG(noise_mode >= RTD3_TICK_NOISE_NONE && noise_mode <= RTD3_TICK_NOISE_PHILOX, "unknown noise mode");
  RTD3_CHECK_ARG(noise_mode != RTD3_TICK_NOISE_GIVEN || unit_noise, "noise mode 'given' needs unit_noise");
  RTD3_CHECK_ARG(noise_mode != RTD3_TICK_NOISE_PHILOX || t->tick_counter, "noise mode 'philox' needs the tick counter");
  if (t->n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // elementwise work plus a few candidate demo states per env: small CTAs spread a small batch over more SMs
  const int block = t->n <= (int64_t)h->num_sms * 256 ? 128 : 256;
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? tick_post_kernel<true> : tick_post_kernel<false>;
  kern<<<(int)ceil_div(t->n, block), block, 0, st>>>(*t, residual, unit_noise, noise_mode, bank);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_tick_run_f16(rtd3_env* h, const rtd3_tick_state* t, int32_t hidden, int32_t layers, const float* params,
                          const uint16_t* params_h, int32_t noise_mode, int64_t ticks, uint64_t tick_base, void* stream) {
  if (int32_t e = check_state(t)) return e;
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(params && params_h, "null parameters");
  RTD3_CHECK_ARG(hidden % 32 == 0 && hidden >= 64 && hidden <= 256 && layers == 2, "needs layers == 2 and hidden in {64..256} divisible by 32");
  RTD3_CHECK_ARG(noise_mode == RTD3_TICK_NOISE_NONE || noise_mode == RTD3_TICK_NOISE_PHILOX, "noise must be none or philox");
  RTD3_CHECK_ARG(t->num_demo == 0 || t->demo_list_start || t->env_demo_pts, "needs candidate lists (rtd3_demo_lists), per-env sets or no demonstration states");
  RTD3_CHECK_ARG(ticks >= 0 && ticks < (1ll << 30), "bad tick count");
  // CTAs run their ticks without a grid-wide barrier, so two CTAs can be up to `ticks` ticks apart: the rows they reserve through
  // the ring counter must not alias, i.e. everything one launch can push has to fit in the ring.
  RTD3_CHECK_ARG(ticks * t->n <= t->capacity, "replay ring smaller than ticks * n rows: CTAs of a multi-tick launch could overwrite each other's rows");
  if (t->n == 0 || ticks == 0) return 0;
  const NetShape s{2, hidden, layers, 2};
  const size_t smem = hf_smem_bytes(hidden) + kHfRows * sizeof(float2);
  const MapBank bank = map_bank(h);
  const auto kern = bank.index ? tick_f16_kernel<true> : tick_f16_kernel<false>;
  RTD3_CUDA(ensure_dyn_smem((const void*)kern, smem));
  uint32_t cols = 32;
  while (cols < (uint32_t)hidden) cols <<= 1;
  const int64_t tiles = ceil_div(t->n, kHfRows);
  const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
  kern<<<grid, kHfThreads, smem, (cudaStream_t)stream>>>(*t, s, params, params_h, noise_mode, (int)ticks, tick_base, cols, bank);
  RTD3_LAUNCHED();
  return 0;
}

}  // extern "C"
