// Single env-step arithmetic shared by the step / rollout kernels (rtd3_env.cu) and the fused tick (rtd3_tick.cu).
// Reference behaviour: /root/reference/environment.py:98-127.
#pragma once
#include "rtd3_common.cuh"
#include "rtd3_mt.cuh"

struct rtd3_env {
  int device = 0;
  int num_sms = 0;
  void* host_pipe = nullptr;   // rtd3::HostPipe of rtd3_env_rollout_host (rtd3_env_host.cu), created on first use
  // Map bank (rtd3_env_set_maps / rtd3_env_set_map_index): map_cap maps allocated, num_maps of them set (none before the first
  // rtd3_env_set_map(s)).  Env v of a launch steps on map index[v % index_len]; with index_len == 0 there is no index and every
  // launch runs the single-map kernels on map 0.
  float2* tables = nullptr;   // [map_cap][100*100] (speed*cos(rot), speed*sin(rot)), indexed x*100+y
  float2* halos = nullptr;    // [map_cap][116*116] the same tables with an 8-cell border, read by the warp-pair rollout (rtd3_env.cu: build_halo_kernel)
  int* fits = nullptr;        // [map_cap] 1 when every cell moves a state by less than the border per step (kMaxAction*(|c|+|s|) <= kHaloReach)
  int num_maps = 0, map_cap = 0;
  int32_t* index = nullptr;
  int64_t index_len = 0, index_cap = 0;
  // The tables were rebuilt (rtd3_env_set_maps) since the last rollout launch, or may be by a replayed graph: the next rollout
  // launch waits for the whole previous grid, since its table staging could otherwise read the tables before they are written.
  bool maps_rebuilt = true;
};

namespace rtd3 {

void host_pipe_destroy(rtd3_env* h);   // rtd3_env_host.cu: streams, staging buffers and cached graphs of the host-buffer rollout
void host_pipe_drop_graphs(rtd3_env* h);   // rtd3_env_host.cu: the cached graphs only (they hold the bank / index addresses)
// rtd3_env_rollout (rtd3_env.cu) with traj_host: the trajectory is host memory, whose writes the kernel waits for before it exits
int32_t env_rollout(rtd3_env* h, float* x, float* y, const float* actions, float* traj, int64_t n, int64_t T, bool traj_host,
                    cudaStream_t st);

// What a kernel needs to step env v on its own map.  Passed by value; index == nullptr (single map) in the launches without a bank.
struct MapBank {
  const float2* tables;   // [K][kCells]
  const float2* halos;    // [K][116*116]
  const int* fits;        // [K]
  const int32_t* index;   // [m]
  int64_t m;
  int K;
  // the map of env v, clamped to [0, K) so that a bad index can never read outside the bank
  __device__ __forceinline__ int map_of(int64_t v) const {
    const int k = __ldg(index + (v < m ? v : v % m));
    return min(max(k, 0), K - 1);
  }
  // the map env v steps on in a kernel instantiated with or without the bank: its own, or map 0 (the launches without an index)
  template <bool kBank>
  __device__ __forceinline__ int map(int64_t v) const { return kBank ? map_of(v) : 0; }
  template <bool kBank>
  __device__ __forceinline__ const float2* table(int64_t v) const { return tables + (size_t)map<kBank>(v) * kCells; }
  // the same launch arguments: a launch captured with one is a launch with the other
  bool operator==(const MapBank& o) const {
    return tables == o.tables && halos == o.halos && fits == o.fits && index == o.index && m == o.m && K == o.K;
  }
};

// The only place a MapBank is built: what every step, rollout and tick launch of `h` passes.
inline MapBank map_bank(const rtd3_env* h) {
  return MapBank{h->tables, h->halos, h->fits, h->index_len ? h->index : nullptr, h->index_len, h->num_maps};
}

// One env-step, the rotation form of environment.py:100-117 (no atan2):
//   s' = clip(s + speed*(ax*cos(rot) - ay*sin(rot), ax*sin(rot) + ay*cos(rot)), 0, 98.9999)
// split into the part that does not depend on the state (StepIn, off the dependent chain of a rollout) and the
// state recurrence itself, which is FADD.RZ -> IMAD -> IMAD -> LDS.64 -> FFMA -> FFMA -> FMNMX -> FMNMX.
struct StepIn {
  float ax, ay;   // clipped action (np.clip keeps NaN), zeroed when NaN
  float lo, hi;   // clip bounds: [0, 98.9999], or [-inf, +inf] when the action is NaN so that the state is kept
  bool bad;       // NaN action: environment.py:125 rejects the (NaN) next state and keeps robot_state
};

__device__ __forceinline__ StepIn prep_action(float ax, float ay) {
  StepIn in;
  ax = clip_keep_nan(ax, -kMaxAction, kMaxAction);
  ay = clip_keep_nan(ay, -kMaxAction, kMaxAction);
  in.bad = (ax != ax) || (ay != ay);
  in.ax = in.bad ? 0.0f : ax;
  in.ay = in.bad ? 0.0f : ay;
  in.lo = in.bad ? -INFINITY : 0.0f;
  in.hi = in.bad ? INFINITY : kClipHi;
  return in;
}

// s' from (s, table entry). Two dependent FFMAs per axis; the only roundings are at the magnitude of the state.
__device__ __forceinline__ void advance(float2 cs, const StepIn& in, float& x, float& y) {
  const float nx = fmaf(in.ax, cs.x, fmaf(-in.ay, cs.y, x));
  const float ny = fmaf(in.ax, cs.y, fmaf(in.ay, cs.x, y));
  x = fminf(fmaxf(nx, in.lo), in.hi);
  y = fminf(fmaxf(ny, in.lo), in.hi);
}

// int(state) -> cell, clamped so that any input stays inside the table (used by the single-step kernels)
__device__ __forceinline__ int cell_index(float x, float y) {
  const int cx = min(max(__float2int_rz(x), 0), kWorld - 1);
  const int cy = min(max(__float2int_rz(y), 0), kWorld - 1);
  return cx * kWorld + cy;
}

template <bool kKeepOnNan, typename TableT>
__device__ __forceinline__ void step_one(const TableT& table, float x, float y, float ax, float ay, float& ox, float& oy) {
  const StepIn in = prep_action(ax, ay);
  const float2 cs = table[cell_index(x, y)];
  advance(cs, in, x, y);
  if (!kKeepOnNan && in.bad) { x = NAN; y = NAN; }   // pure dynamics(): the NaN propagates
  ox = x;
  oy = y;
}

struct LdgTable {
  const float2* __restrict__ p;
  __device__ __forceinline__ float2 operator[](int i) const { return __ldg(p + i); }
};
struct SmemTable {
  const float2* p;
  __device__ __forceinline__ float2 operator[](int i) const { return p[i]; }
};

// Environment.reset for the lanes of one warp (environment.py:130-137): `active` lanes draw a new start state from their env's
// MT19937 stream.  All 32 lanes must call both halves (streams that wrap are twisted by the whole warp, rtd3_mt.cuh).
// Split in two so that a caller can put other work between the loads and their use: reset_load_warp issues the loads (stream
// position, init region and - unless a lane's stream wraps within the next four words, ~0.6 % of the draws - the four state
// words themselves, independent of each other), reset_finish_warp turns them into the state.
struct ResetLoads {
  int pos;
  double left, right, bottom, top;
  uint32_t w[4];
  bool have_words;   // warp-uniform
};

__device__ __forceinline__ ResetLoads reset_load_warp(const rtd3_mt_bank& b, const double* __restrict__ region, bool active, int64_t i) {
  ResetLoads r;
  r.pos = 0; r.left = r.right = r.bottom = r.top = 0.0; r.have_words = false;
#pragma unroll
  for (int q = 0; q < 4; ++q) r.w[q] = 0u;
  if (!__any_sync(0xffffffffu, active)) return r;
  const int64_t n = b.n;
  if (active) {
    r.pos = b.pos[i];
    r.left = region[i]; r.right = region[n + i]; r.bottom = region[2 * n + i]; r.top = region[3 * n + i];
  }
  r.have_words = !__any_sync(0xffffffffu, active && r.pos + 4 > RTD3_MT_N);
  if (r.have_words && active) {
#pragma unroll
    for (int q = 0; q < 4; ++q) r.w[q] = mt_temper(b.mt[(int64_t)(r.pos + q) * n + i]);
  }
  return r;
}

__device__ __forceinline__ void reset_finish_warp(const rtd3_mt_bank& b, bool active, int64_t i, ResetLoads& r, float* __restrict__ x,
                                                  float* __restrict__ y, double* __restrict__ state64) {
  if (!__any_sync(0xffffffffu, active)) return;
  const int64_t n = b.n;
  int pos_after = r.pos + 4;
  if (!r.have_words) {                               // a stream of this warp wraps: draw word by word through the warp twist
    int pos = r.pos;
    mt_next_words4_warp_slow(b.mt + (active ? i : 0), n, &pos, active, r.w);
    pos_after = pos;
  }
  if (!active) return;
  // lo + (hi - lo) * u with numpy's two roundings
  const double ux = mt_double_from_words(r.w[0], r.w[1]), uy = mt_double_from_words(r.w[2], r.w[3]);
  const double sx = __dadd_rn(r.left, __dmul_rn(__dsub_rn(r.right, r.left), ux));        // x in [left, right)
  const double sy = __dadd_rn(r.bottom, __dmul_rn(__dsub_rn(r.top, r.bottom), uy));      // y in [bottom, top)
  // float32 rounding must not reach 100.0 (the cell index would leave the map): cap at the largest float below it
  x[i] = fminf((float)sx, 99.99999f); y[i] = fminf((float)sy, 99.99999f);
  if (state64) { state64[i] = sx; state64[n + i] = sy; }
  b.pos[i] = pos_after;
}

__device__ __forceinline__ void reset_env_warp(const rtd3_mt_bank& b, const double* __restrict__ region, bool active, int64_t i,
                                               float* __restrict__ x, float* __restrict__ y, double* __restrict__ state64) {
  ResetLoads r = reset_load_warp(b, region, active, i);
  reset_finish_warp(b, active, i, r, x, y, state64);
}

}  // namespace rtd3
