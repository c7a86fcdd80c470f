// Environment hot path: dynamics / step / T-step rollout / seeded init + reset.
// Reference behaviour: /root/reference/environment.py:28-56, 98-137 (see include/rtd3.h per entry point).
#include <cuda.h>

#include <memory>
#include <type_traits>
#include <utility>

#include "rtd3_common.cuh"
#include "rtd3_env_step.cuh"
#include "rtd3_mt.cuh"


namespace rtd3 {

constexpr uint32_t kTableBytes = kCells * sizeof(float2);   // 80 000 B, a multiple of 16
constexpr int kTableChunks = 4;                             // bulk copies of 20 000 B each
static_assert(kTableBytes % (16 * kTableChunks) == 0, "bulk copy sizes must be multiples of 16 B");

// rot = float32(angle*2*pi): numpy >= 2 keeps float32*int*pyfloat in float32 (environment.py:107).
// cos/sin are taken in float64 like the reference does for (action_angle + rotation).
// Runs over the cells of all `cells / kCells` maps of a bank: map k's table is table[k * kCells ...].
__global__ void build_table_kernel(const float* __restrict__ speed, const float* __restrict__ angle,
                                   float2* __restrict__ table, int64_t cells) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cells) return;
  float rot = __fmul_rn(__fmul_rn(angle[i], 2.0f), 3.14159274101257324f);
  double s, c;
  sincos((double)rot, &s, &c);
  double sp = (double)speed[i];
  float tc = (float)(sp * c), ts = (float)(sp * s);
  // A non-finite map cell would make the reference raise (int(nan)); here it becomes a dead cell so that the
  // state recurrence below can never leave [0, 100) and index out of the table.
  if (!isfinite(tc) || !isfinite(ts)) { tc = 0.0f; ts = 0.0f; }
  table[i] = make_float2(tc, ts);
}


// ---- halo table of the warp-pair rollout -----------------------------------------------------------------------------
// The pair kernel's chain warp takes the table address of step t+1 from the UNCLIPPED next state of step t, which keeps the
// clip to [0, 98.9999] off its dependent chain.  On a map that fits (every cell moves a state by at most kHaloReach < 8 per
// step under actions clipped to +-kMaxAction) an unclipped coordinate v of a state that was in [0, 98.9999] lies in
// [-8, 107), and the halo table is laid out so that halo[floor(v) + 8] == table[floor(clip(v))] there: indices 0..7 repeat
// cell 0, 8..106 are cells 0..98 and 107..114 repeat cell 98.  Cell 99 is reachable only from a state in [99, 100) (a start
// state, or one kept through NaN actions); it sits at index 115, and an address taken from a state maps 107 to it.
constexpr int kHalo = 8;
constexpr int kHaloDim = kWorld + 2 * kHalo;                                   // 116
constexpr uint32_t kHaloBytes = kHaloDim * kHaloDim * sizeof(float2);          // 107 648 B
constexpr uint32_t kHaloRowBytes = kHaloDim * sizeof(float2);
constexpr float kHaloReach = 7.99f;   // < 8 with room for the two roundings of the step
static_assert(kHaloBytes % (16 * kTableChunks) == 0, "bulk copy sizes must be multiples of 16 B");

__device__ __forceinline__ int halo_cell(int i) {
  return i < kHalo ? 0 : i < kWorld - 1 + kHalo ? i - kHalo : i < kHaloDim - 1 ? kWorld - 2 : kWorld - 1;
}

// One CTA per map of the bank: copies the finished table into the halo layout and writes whether the map fits, in device memory so
// that rtd3_env_set_map(s) stays asynchronous (and capturable).  Non-finite cells were zeroed by build_table_kernel and fit.
__global__ void __launch_bounds__(1024) build_halo_kernel(const float2* __restrict__ table, float2* __restrict__ halo, int* __restrict__ fits) {
  table += (size_t)blockIdx.x * kCells;
  halo += (size_t)blockIdx.x * (kHaloDim * kHaloDim);
  fits += blockIdx.x;
  bool ok = true;
  for (int i = threadIdx.x; i < kCells; i += blockDim.x) {
    const float2 cs = table[i];
    ok = ok && kMaxAction * (fabsf(cs.x) + fabsf(cs.y)) <= kHaloReach;
  }
  for (int i = threadIdx.x; i < kHaloDim * kHaloDim; i += blockDim.x)
    halo[i] = table[halo_cell(i / kHaloDim) * kWorld + halo_cell(i % kHaloDim)];
  ok = __syncthreads_and(ok);
  if (threadIdx.x == 0) *fits = ok ? 1 : 0;
}

// Stage a table (kBytes: the 80 KB plain one or the 105 KB halo one) into shared memory with bulk-async copies signalled
// on one mbarrier.  All threads of the CTA call this; returns once the copies are issued, mbar_wait(bar, 0) waits for them.
template <uint32_t kBytes = kTableBytes>
__device__ __forceinline__ void stage_table(float2* s_table, uint64_t* bar, const float2* __restrict__ g_table) {
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    mbar_arrive_expect_tx(bar, kBytes);
    constexpr uint32_t chunk = kBytes / kTableChunks;
#pragma unroll
    for (int c = 0; c < kTableChunks; ++c)
      bulk_g2s(reinterpret_cast<char*>(s_table) + c * chunk, reinterpret_cast<const char*>(g_table) + c * chunk, chunk,
               bar);
  }
}

// ---- single step over n envs ------------------------------------------------------------------
// Each thread owns 4 consecutive envs per iteration: four 16 B loads (x,y,ax,ay) and two 16 B stores,
// all coalesced (a warp covers 512 B contiguous per plane).  kKeepOnNan=false gives pure dynamics().
// kBank: env j steps on its own map, bank.table<true>(j), read through the read-only path (a CTA covers envs of many maps, so
// there is no one table to stage: kBank goes with kSmem == false).  Without it every env steps on map 0.
// Parameter order: the scalar first puts the six pointers at 8 mod 16 in the constant bank, where ptxas pairs their loads
// into the schedule this kernel was measured with (62 registers for dynamics()).
template <bool kSmem, bool kKeepOnNan, bool kBank = false>
__global__ void __launch_bounds__(kSmem ? 512 : 256, kSmem ? 2 : 4)
env_step_kernel(int vec_ok, const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ ax, const float* __restrict__ ay,
                float* __restrict__ ox, float* __restrict__ oy, int64_t n, MapBank bank) {
  static_assert(!(kBank && kSmem), "a bank step reads its tables from global memory");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float2* s_table = reinterpret_cast<float2*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + kTableBytes);

  const int64_t n4 = vec_ok ? (n >> 2) : 0;   // planes not 16 B aligned (odd n): everything goes the scalar way
  const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nthreads = (int64_t)gridDim.x * blockDim.x;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  const float4* y4 = reinterpret_cast<const float4*>(y);
  const float4* ax4 = reinterpret_cast<const float4*>(ax);
  const float4* ay4 = reinterpret_cast<const float4*>(ay);

  if constexpr (kSmem) stage_table(s_table, bar, bank.tables);

  // issue the first iteration's streaming loads before waiting for the table
  int64_t i = tid;
  float4 vx, vy, vax, vay;
  bool have = i < n4;
  if (have) { vx = __ldcs(x4 + i); vy = __ldcs(y4 + i); vax = __ldcs(ax4 + i); vay = __ldcs(ay4 + i); }
  if constexpr (kSmem) mbar_wait(bar, 0);

  // env j's table: env j's own map with the bank, else the one table of every env, built once (a table object built per call
  // reorders ptxas's schedule of the loop)
  const auto one_table = [&]() {
    if constexpr (kSmem) return SmemTable{s_table};
    else return LdgTable{bank.tables};
  }();
  auto table = [&](int64_t j) -> decltype(auto) {
    if constexpr (kBank) return LdgTable{bank.table<kBank>(j)};
    else return std::as_const(one_table);
  };

  while (have) {
    const int64_t inext = i + nthreads;
    const bool have_next = inext < n4;
    float4 px, py, pax, pay;
    if (have_next) { px = __ldcs(x4 + inext); py = __ldcs(y4 + inext); pax = __ldcs(ax4 + inext); pay = __ldcs(ay4 + inext); }
    float4 rx, ry;
    step_one<kKeepOnNan>(table(4 * i), vx.x, vy.x, vax.x, vay.x, rx.x, ry.x);
    step_one<kKeepOnNan>(table(4 * i + 1), vx.y, vy.y, vax.y, vay.y, rx.y, ry.y);
    step_one<kKeepOnNan>(table(4 * i + 2), vx.z, vy.z, vax.z, vay.z, rx.z, ry.z);
    step_one<kKeepOnNan>(table(4 * i + 3), vx.w, vy.w, vax.w, vay.w, rx.w, ry.w);
    __stcs(reinterpret_cast<float4*>(ox) + i, rx);
    __stcs(reinterpret_cast<float4*>(oy) + i, ry);
    i = inext; have = have_next;
    if (have) { vx = px; vy = py; vax = pax; vay = pay; }
  }

  // ragged tail (n % 4 envs), handled by the first threads of the grid
  for (int64_t j = (n4 << 2) + tid; j < n; j += nthreads) {
    float rx, ry;
    step_one<kKeepOnNan>(table(j), x[j], y[j], ax[j], ay[j], rx, ry);
    ox[j] = rx; oy[j] = ry;
  }
}

// ---- T-step rollout: state stays in registers, table in smem, actions prefetched kU steps ahead ----
constexpr int kU = 16;
constexpr int kDeep = 8;      // chunks in flight per thread, latency-bound launches (128 steps of lead)
constexpr int kShallow = 2;   // chunks in flight per thread, occupancy-bound launches

__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}

// The dependent chain of one rollout step.  trunc(x) comes from a round-toward-zero add of 2^23 (the low mantissa
// bits of x + 2^23 are floor(x) for 0 <= x < 2^23), so the shared-memory byte address is two IMADs away from the state:
//   addr = bits(x+2^23)*800 + bits(y+2^23)*8 + (table_base - 0x4B000000*808)
__device__ __forceinline__ void rollout_step(uint32_t addr_bias, const StepIn& in, float& x, float& y) {
  const uint32_t bx = __float_as_uint(__fadd_rz(x, 8388608.0f));
  const uint32_t by = __float_as_uint(__fadd_rz(y, 8388608.0f));
  const uint32_t addr = bx * 800u + (by * 8u + addr_bias);
  advance(lds_f2(addr), in, x, y);
}

// Halo-table addresses (addr_bias = table base - 0x4B000000 * (kHaloRowBytes + 8)).  With 2^23 + 8 every v in [-8, 107)
// stays in the binade whose grid is 1, so the low bits of v + 2^23 + 8, rounded toward zero, are exactly floor(v) + 8
// (with 2^23 a v in (-1, 0) would fall to the 0.5 grid below 2^23 and floor wrongly).
__device__ __forceinline__ uint32_t halo_addr(uint32_t addr_bias, float x, float y) {
  const uint32_t bx = __float_as_uint(__fadd_rz(x, 8388616.0f));
  const uint32_t by = __float_as_uint(__fadd_rz(y, 8388616.0f));
  return bx * kHaloRowBytes + (by * 8u + addr_bias);
}
// the address of table[floor(x)][floor(y)] for a state in [0, 100): index 107 (floor 99) is cell 99, stored at 115
__device__ __forceinline__ uint32_t halo_addr_state(uint32_t addr_bias, float x, float y) {
  constexpr uint32_t k99 = 0x4B000000u + kHalo + kWorld - 1;
  uint32_t bx = __float_as_uint(__fadd_rz(x, 8388616.0f));
  uint32_t by = __float_as_uint(__fadd_rz(y, 8388616.0f));
  bx = bx == k99 ? bx + kHalo : bx;
  by = by == k99 ? by + kHalo : by;
  return bx * kHaloRowBytes + (by * 8u + addr_bias);
}

// Rollout kernels with a map bank (kBank): the CTA stages the map of its first env (map 0 without the bank).  A warp whose live envs
// all step on that map runs the shared-memory loop unchanged; a warp that mixes maps (mixed) steps every lane from its own map's
// plain table in global memory, addressed from the state like the careful path - the same cell, the same values, so the same bits.
struct BankLanes {
  bool mixed;      // warp-uniform
  const float2* table;   // this lane's plain table
};
__device__ __forceinline__ BankLanes bank_lanes(const MapBank& b, int staged, int64_t i, bool live) {
  BankLanes r;
  const int mine = live ? b.map_of(i) : staged;
  r.mixed = !__all_sync(0xffffffffu, mine == staged);
  r.table = b.tables + (size_t)mine * kCells;
  return r;
}
// one state-addressed step from the lane's own table (the mixed-warp path)
__device__ __forceinline__ void ldg_step(const float2* __restrict__ table, const StepIn& in, float& x, float& y) {
  advance(__ldg(table + cell_index(x, y)), in, x, y);
}

// Actions reach the SM through a per-thread cp.async ring in shared memory: kStages chunks of kU steps are in
// flight, so the HBM latency (~1 us) is hidden even when a CTA is a single warp (4096 envs on 148 SMs); every
// thread reads back only the words it copied itself, so cp.async.wait_group is the only synchronisation.
__device__ __forceinline__ void cp_async4(uint32_t smem_addr, const float* g) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int kN>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(kN) : "memory"); }

// Parameter order: n first for the same reason as env_step_kernel's vec_ok.
template <bool kTraj, int kStages, bool kBank = false>
__global__ void __launch_bounds__(256)
env_rollout_kernel(int64_t n, float* __restrict__ x, float* __restrict__ y, const float* __restrict__ actions, float* __restrict__ traj,
                   int64_t T, MapBank bank) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float2* s_table = reinterpret_cast<float2*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + kTableBytes);
  float* ring = reinterpret_cast<float*>(smem_raw + kTableBytes + 16);   // [kStages][kU][2][blockDim]
  launch_dependents();                  // launch overlap as in env_rollout_pair_kernel
  int staged = 0;
  BankLanes bl{};
  // contains the only __syncthreads of the kernel
  const auto stage = [&] { stage_table(s_table, bar, bank.tables + (size_t)staged * kCells); };
  if constexpr (!kBank) stage();
  grid_dep_wait();
  if constexpr (kBank) {
    staged = bank.map<kBank>((int64_t)blockIdx.x * blockDim.x);
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bl = bank_lanes(bank, staged, env, env < n);
    stage();
  }

  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;                   // thread 0 of every launched CTA is live, so the bulk copy always has an owner
  // Sanitise once: inside [0, 100) the recurrence can never leave the table (finite table, clamped or kept state).
  // States outside the world are invalid input for the reference as well (IndexError at environment.py:107).
  float sx = fminf(fmaxf(x[i], 0.0f), 99.99999f);
  float sy = fminf(fmaxf(y[i], 0.0f), 99.99999f);
  const int64_t n2 = 2 * n;
  const float* pa = actions + i;        // ax(t) = pa[0], ay(t) = pa[n]; advances by 2n per step
  float* pt = traj + i;
  const uint32_t addr_bias = smem_u32(s_table) - 0x4B000000u * 808u;
  const uint32_t bd = blockDim.x;
  const uint32_t my_ring = smem_u32(ring) + threadIdx.x * 4u;
  const uint32_t stage_bytes = kU * 2u * bd * 4u;

  const int64_t full = T / kU;          // chunks of kU steps without per-step bounds checks
  auto issue_chunk = [&](int64_t c) {   // chunk c -> ring slot c % kStages
    if (c < full) {
      const float* src = pa + c * (kU * n2);
      const uint32_t dst = my_ring + (uint32_t)(c % kStages) * stage_bytes;
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        cp_async4(dst + (2 * u) * bd * 4u, src + u * n2);
        cp_async4(dst + (2 * u + 1) * bd * 4u, src + u * n2 + n);
      }
    }
    cp_async_commit();                  // always commit, so that group counting stays uniform
  };
#pragma unroll
  for (int sgi = 0; sgi < kStages; ++sgi) issue_chunk(sgi);
  mbar_wait(bar, 0);

  for (int64_t c = 0; c < full; ++c) {
    cp_async_wait<kStages - 1>();       // chunk c has landed
    StepIn in[kU];
    const uint32_t src = my_ring + (uint32_t)(c % kStages) * stage_bytes;
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      float ax, ay;
      asm volatile("ld.shared.f32 %0, [%1];" : "=f"(ax) : "r"(src + (2 * u) * bd * 4u));
      asm volatile("ld.shared.f32 %0, [%1];" : "=f"(ay) : "r"(src + (2 * u + 1) * bd * 4u));
      in[u] = prep_action(ax, ay);
    }
    issue_chunk(c + kStages);           // refill the slot just drained (its values are in registers now)
    if (kBank && bl.mixed) {
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        ldg_step(bl.table, in[u], sx, sy);
        if (kTraj) { __stcs(pt, sx); __stcs(pt + n, sy); pt += n2; }
      }
    } else {
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        rollout_step(addr_bias, in[u], sx, sy);
        if (kTraj) { __stcs(pt, sx); __stcs(pt + n, sy); pt += n2; }
      }
    }
  }
  pa += full * (kU * n2);
  for (int64_t t = full * kU; t < T; ++t) {   // ragged tail, T % kU steps
    const StepIn in = prep_action(__ldcs(pa), __ldcs(pa + n));
    pa += n2;
    if (kBank && bl.mixed) ldg_step(bl.table, in, sx, sy);
    else rollout_step(addr_bias, in, sx, sy);
    if (kTraj) { __stcs(pt, sx); __stcs(pt + n, sy); pt += n2; }
  }
  cp_async_wait<0>();
  x[i] = sx;
  y[i] = sy;
}

// ---- T-step rollout, TMA variant (n % 4 == 0): one warp = 32 envs = one independent pipeline -------------------------
// Actions [T][2][n] and trajectories are 2-D tensors (inner dim n, outer dim 2T) described by CUtensorMaps; a warp moves
// its [kU steps x 2][32 envs] tile (32 rows of 128 B) with ONE cp.async.bulk.tensor.2d (SASS UTMALDG / UTMASTG) per
// chunk and direction: loads complete on a per-stage mbarrier, stores are tracked by the bulk async-group.  This removes
// the per-step LDGSTS/STG and their 64-bit address arithmetic from the single warp that has to issue everything
// (ncu r1: 47 instr/step at IPC 0.38 bounded the cp.async version; 32 row-wise 128 B bulk copies per chunk were tried
// first and were 2.6x SLOWER - the TMA unit is op-bound, not byte-bound, at that size).  Out-of-range rows / envs of
// edge tiles are zero-filled on load and clipped on store by the TMA unit itself.
constexpr int kTileFloats = kU * 2 * 32;          // 1024 floats = 4 KB per warp per stage

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, int c0, int c1, const void* smem_src) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(reinterpret_cast<uint64_t>(tm)),
               "r"(c0), "r"(c1), "r"(smem_u32(smem_src))
               : "memory");
}

__device__ __forceinline__ void prefetch_tensormap(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// Pulls a tile into L2 only: safe before grid_dep_wait, since L2 is where writes of the previous grid become coherent.
__device__ __forceinline__ void tma_prefetch_l2_2d(const CUtensorMap* tm, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1)
               : "memory");
}

// Parameter order: n first for the same reason as env_step_kernel's vec_ok.  Launch overlap and traj_host as in
// env_rollout_pair_kernel.
template <bool kTraj, int kStages, bool kBank = false>
__global__ void __launch_bounds__(256)
env_rollout_tma_kernel(int64_t n, float* __restrict__ x, float* __restrict__ y, const __grid_constant__ CUtensorMap tm_act,
                       const __grid_constant__ CUtensorMap tm_traj, int64_t T, MapBank bank, int traj_host) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  launch_dependents();
  float2* s_table = reinterpret_cast<float2*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + kTableBytes);            // table barrier
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kTableBytes + 16) + warp * kStages;     // [nwarps][kStages]
  // tiles start on a 128 B boundary behind the barriers
  float* tiles = reinterpret_cast<float*>(smem_raw + ((kTableBytes + 16 + nwarps * kStages * 8 + 127) & ~127u));
  float* my_in = tiles + (size_t)warp * kStages * kTileFloats;                                     // action ring of this warp
  float* my_out = tiles + (size_t)nwarps * kStages * kTileFloats + (size_t)warp * 2 * kTileFloats; // 2 trajectory staging tiles
  if (lane == 0) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(full + s, 1);
    fence_mbar_init();
  }
  if (threadIdx.x == 0) {
    prefetch_tensormap(&tm_act);
    if (kTraj) prefetch_tensormap(&tm_traj);
  }
  int staged = 0;
  BankLanes bl{};
  // init + fence + __syncthreads, then the table's bulk copies
  const auto stage = [&] { stage_table(s_table, bar, bank.tables + (size_t)staged * kCells); };
  if constexpr (!kBank) stage();
  grid_dep_wait();
  if constexpr (kBank) {
    staged = bank.map<kBank>((int64_t)blockIdx.x * nwarps * 32);
    const int64_t env = ((int64_t)blockIdx.x * nwarps + warp) * 32 + lane;
    bl = bank_lanes(bank, staged, env, env < n);
    stage();
  }

  const int64_t i0 = ((int64_t)blockIdx.x * nwarps + warp) * 32;                  // first env of this warp
  if (i0 >= n) return;
  const int64_t i = i0 + lane;
  const bool live = i < n;
  float sx = live ? fminf(fmaxf(x[i], 0.0f), 99.99999f) : 0.0f;
  float sy = live ? fminf(fmaxf(y[i], 0.0f), 99.99999f) : 0.0f;
  const uint32_t addr_bias = smem_u32(s_table) - 0x4B000000u * 808u;
  const int64_t chunks = (T + kU - 1) / kU;

  auto issue_chunk = [&](int64_t c) {
    if (c < chunks && lane == 0) {
      const int s = (int)(c % kStages);
      mbar_arrive_expect_tx(full + s, kTileFloats * 4);
      tma_load_2d(my_in + s * kTileFloats, &tm_act, (int)i0, (int)(c * (2 * kU)), full + s);
    }
  };
#pragma unroll
  for (int s = 0; s < kStages; ++s) issue_chunk(s);
  mbar_wait(bar, 0);

  for (int64_t c = 0; c < chunks; ++c) {
    const int s = (int)(c % kStages);
    mbar_wait(full + s, (uint32_t)((c / kStages) & 1));
    float cax[kU], cay[kU];
    float nanacc = 0.0f;
    const float* tin = my_in + s * kTileFloats + lane;
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      cax[u] = tin[(2 * u) * 32];
      cay[u] = tin[(2 * u + 1) * 32];
      nanacc = fmaf(cax[u], 0.0f, nanacc);      // stays 0 unless an action is NaN or inf
      nanacc = fmaf(cay[u], 0.0f, nanacc);
    }
    __syncwarp();                               // every lane holds its values: the slot can be refilled
    issue_chunk(c + kStages);
    float* tout = my_out + (c & 1) * kTileFloats + lane;
    if (kTraj && lane == 0) bulk_wait_read<1>();   // the staging tile used two chunks ago has been read by its store
    __syncwarp();
    const int steps = (int)min((int64_t)kU, T - c * kU);
    const bool careful = __any_sync(0xffffffffu, nanacc != 0.0f) || steps < kU;
    if (!careful && !(kBank && bl.mixed)) {
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        StepIn in;
        in.ax = fminf(fmaxf(cax[u], -kMaxAction), kMaxAction);
        in.ay = fminf(fmaxf(cay[u], -kMaxAction), kMaxAction);
        in.lo = 0.0f; in.hi = kClipHi; in.bad = false;
        rollout_step(addr_bias, in, sx, sy);
        if (kTraj) { tout[(2 * u) * 32] = sx; tout[(2 * u + 1) * 32] = sy; }
      }
    } else if (kBank && bl.mixed) {
      // A loop of its own: folded into the loop below (the table read chosen per step), it made the mixed-warp launches
      // ~2 % slower.
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (u < steps) ldg_step(bl.table, prep_action(cax[u], cay[u]), sx, sy);
        if (kTraj) { tout[(2 * u) * 32] = sx; tout[(2 * u + 1) * 32] = sy; }
      }
    } else {
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (u < steps) {
          const StepIn in = prep_action(cax[u], cay[u]);
          rollout_step(addr_bias, in, sx, sy);
        }
        if (kTraj) { tout[(2 * u) * 32] = sx; tout[(2 * u + 1) * 32] = sy; }
      }
    }
    if (kTraj) {
      fence_proxy_async();                      // generic-proxy writes of the tile -> visible to the TMA (async proxy) read
      __syncwarp();
      if (lane == 0) {
        tma_store_2d(&tm_traj, (int)i0, (int)(c * (2 * kU)), my_out + (c & 1) * kTileFloats);
        bulk_commit();
      }
    }
  }
  if (live) { x[i] = sx; y[i] = sy; }
  if (kTraj && lane == 0) {                     // the stores must have left shared memory before the CTA exits
    if (traj_host) bulk_wait<0>();
    else bulk_wait_read<0>();
  }
}

// ---- T-step rollout, warp-pair variant: chain warps + helper warp per 32 envs ------------------------------------------
// At 4096 envs every SM gets one warp, and that warp's issue slots - not memory - bound the TMA kernel above (31
// instr/step, of which only 13 are the state recurrence; ncu r1: 42 % fixed-latency waits).  Here the recurrence runs
// alone on the CHAIN warps (per step: one LDS.64 of the pre-clipped action, the chain, two STS of the new state); a
// HELPER warp on another scheduler of the same SM waits for the TMA action tiles, clips them (or flags the chunk for the
// careful NaN path), re-arms the loads and issues the trajectory tile stores.  They meet on mbarriers over
// double-buffered shared-memory tiles of 32 envs.  The table is the halo table (see kHalo), so that on a map that fits, the
// chain of a step is FFMA, FFMA -> FADD.RZ -> IMAD, IMAD -> LDS.64: the clip, the action load and the trajectory stores are
// issued while the table load is in flight.
// A chain warp steps kChainLanes envs of the tile, one per lane, and its other lanes idle: the table gather of a step reads
// one 8-byte cell per active lane from unrelated places, and the bank conflicts of that gather sit on the dependent chain of
// every step (tools/lds_chain/lds_chain.cu on a B200: 34.4 cycles per dependent gather at 32 lanes, 28.3 at 16, 24.1 without
// conflicts).  A chain warp issues the same instructions per step whatever its width, and the SM's other schedulers are idle
// at these batch sizes.  16 lanes rather than 8: at 8 the helper shares a scheduler with a chain warp, and with two tiles per
// CTA (8 192 envs) the step got slower than with 32 lanes (DESIGN.md).
constexpr int kPairU = 32;        // steps per tile of the pair kernel
constexpr int kPairStages = 4;    // action tiles in flight (128 steps of lead, as kDeep x kU), one tile per CTA
constexpr int kPairStages2 = 3;   // two tiles per CTA: 4 stages do not fit next to the halo table
constexpr int kChainLanes = 16;     // envs per chain warp
constexpr int pair_warps(int lanes) { return 32 / lanes + 1; }   // warps per 32-env tile: the chain warps, then the helper
struct PairSmem {
  static constexpr int kBars = 16;   // full[8] | prepped[2] | consumed[2] | outfull[2] | outfree[2]
};

// ---- launch phase stamps (builds with -DRTD3_ROLLOUT_STAMPS only; tools/rollout_launch_stamps.py) --------------------------------
// Every CTA of the pair kernel takes one record of kStampWords %globaltimer values in the buffer armed by rtd3_rollout_stamps_arm.
// Records are handed out in CTA start order; the launch a record belongs to is recovered from the start stamps (every CTA of
// launch k starts before any CTA of launch k+1, with or without programmatic dependent launch).
enum StampPhase {
  kStampStart,        // CTA start
  kStampWaited,       // grid_dep_wait returned
  kStampTable,        // the chain warp saw the table land
  kStampPrepped0,     // the helper prepped the first tile
  kStampChain0,       // the chain warp starts chunk 0
  kStampChainEnd,     // the chain warp ends the last chunk
  kStampLastStore,    // the helper issued the last trajectory store
  kStampHelperExit,   // the helper's last instruction
  kStampChainExit,    // the chain warp's last instruction
  kStampMeta,         // blockIdx.x | smid << 32
  kStampWords
};
#ifdef RTD3_ROLLOUT_STAMPS
__device__ unsigned long long* g_stamps = nullptr;
__device__ unsigned long long g_stamp_next = 0, g_stamp_cap = 0;
__device__ __forceinline__ unsigned long long globaltimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void stamp(uint32_t slot, int phase) {
  if (g_stamps && slot < g_stamp_cap) g_stamps[(size_t)slot * kStampWords + phase] = globaltimer();
}
#define RTD3_STAMP_SLOT_DECL __shared__ uint32_t s_stamp_slot;
#define RTD3_STAMP_SLOT_TAKE()                                                                                             \
  if (threadIdx.x == 0) {                                                                                                  \
    s_stamp_slot = (uint32_t)atomicAdd(&g_stamp_next, 1ull);                                                               \
    stamp(s_stamp_slot, kStampStart);                                                                                      \
    uint32_t smid;                                                                                                         \
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));                                                                      \
    if (g_stamps && s_stamp_slot < g_stamp_cap) g_stamps[(size_t)s_stamp_slot * kStampWords + kStampMeta] = blockIdx.x | (unsigned long long)smid << 32; \
  }
#define RTD3_STAMP(cond, phase) \
  if (cond) stamp(s_stamp_slot, phase)
#else
#define RTD3_STAMP_SLOT_DECL
#define RTD3_STAMP_SLOT_TAKE()
#define RTD3_STAMP(cond, phase)
#endif

// Launch overlap: every CTA lets the next launch of the stream start at once, and does before grid_dep_wait only what cannot depend
// on the grid before it - barrier inits, tensor-map and L2 prefetches, and (single map) the table staging: the host launches with
// programmatic serialization only when the tables were not rebuilt since the previous rollout launch.  State, actions and (bank)
// the map index are read after the wait.  traj_host: the trajectory is host memory, so the helper waits for its last store to
// complete before exiting; for device memory the completion of the grid covers it, and the helper only waits for the store to
// have read its shared-memory tile.
template <bool kTraj, int kStages, int kUp, int kLanes, bool kBank = false>
__global__ void __launch_bounds__(2 * pair_warps(kLanes) * 32)
env_rollout_pair_kernel(float* __restrict__ x, float* __restrict__ y, const __grid_constant__ CUtensorMap tm_act,
                        const __grid_constant__ CUtensorMap tm_traj, int64_t n, int64_t T, MapBank bank, int traj_host) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  RTD3_STAMP_SLOT_DECL
  RTD3_STAMP_SLOT_TAKE()
  launch_dependents();
  constexpr int kU = kUp;                            // steps per action / trajectory tile of this kernel (shadows the file-wide kU)
  constexpr int kTileFloats = kU * 2 * 32;
  constexpr int kChains = 32 / kLanes;               // chain warps per tile
  static_assert(kLanes * kChains == 32, "the chain warps of a tile cover its 32 envs");
  float2* s_table = reinterpret_cast<float2*>(smem_raw);
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + kHaloBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, ntiles = blockDim.x / (pair_warps(kLanes) * 32);
  const int tile = warp / pair_warps(kLanes);
  const int cw = warp % pair_warps(kLanes);          // chain warp cw of the tile, or the helper (cw == kChains)
  const bool is_chain = cw < kChains;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + kHaloBytes + 16) + tile * PairSmem::kBars;
  uint64_t* full = bars, *prepped = bars + 8, *consumed = bars + 10, *outfull = bars + 12, *outfree = bars + 14;
  // per tile: kStages raw tiles | 2 prepped tiles (float2 per step and env = 2 tiles' worth each... [kU][32] float2 = 4 KB) | 2 out tiles
  float* tiles = reinterpret_cast<float*>(smem_raw + ((kHaloBytes + 16 + ntiles * PairSmem::kBars * 8 + 127) & ~127u));
  float* my = tiles + (size_t)tile * (kStages + 4) * kTileFloats;
  float* raw = my;                                   // [kStages][kU*2][32]
  float2* prep = reinterpret_cast<float2*>(my + kStages * kTileFloats);                 // [2][kU][32]
  float* outt = my + (kStages + 2) * kTileFloats;    // [2][kU*2][32]
  __shared__ int s_flag[2][2];                       // careful flag per tile and prepped buffer
  // consumed / outfull count one arrival per env of the tile: the active lanes of its chain warps
  if (lane == 0 && !is_chain) {
#pragma unroll
    for (int s = 0; s < kStages; ++s) mbar_init(full + s, 1);
    for (int b = 0; b < 2; ++b) { mbar_init(prepped + b, 32); mbar_init(consumed + b, 32); mbar_init(outfull + b, 32); mbar_init(outfree + b, 1); }
    fence_mbar_init();
  }
  const int64_t i0 = ((int64_t)blockIdx.x * ntiles + tile) * 32;
  const int64_t chunks = (T + kU - 1) / kU;
  if (lane == 0 && !is_chain) {
    prefetch_tensormap(&tm_act);
    if (kTraj) prefetch_tensormap(&tm_traj);
    if (i0 < n)
      for (int s = 0; s < kStages && s < chunks; ++s) tma_prefetch_l2_2d(&tm_act, (int)i0, s * (2 * kU));
  }
  const int col = cw * kLanes + lane;                // a chain lane's env within the tile (lane < kLanes)
  int staged = 0;
  BankLanes bl{};
  const auto stage = [&] {   // contains the __syncthreads that publishes the barrier inits
    stage_table<kHaloBytes>(s_table, bar, bank.halos + (size_t)staged * (kHaloDim * kHaloDim));
  };
  if constexpr (!kBank) stage();
  grid_dep_wait();
  RTD3_STAMP(threadIdx.x == 0, kStampWaited);
  if constexpr (kBank) {
    staged = bank.map<kBank>((int64_t)blockIdx.x * ntiles * 32);   // the CTA stages the halo table of its first env's map
    const int64_t env = i0 + col;                    // mixed: over the active lanes of this chain warp
    bl = bank_lanes(bank, staged, env, is_chain && lane < kLanes && env < n);
    stage();
  }

  if (i0 >= n) return;

  if (!is_chain) {
    // ================================= helper warp =================================
    auto issue_load = [&](int64_t c) {
      if (c < chunks && lane == 0) {
        const int s = (int)(c % kStages);
        mbar_arrive_expect_tx(full + s, kTileFloats * 4);
        tma_load_2d(raw + s * kTileFloats, &tm_act, (int)i0, (int)(c * (2 * kU)), full + s);
      }
    };
#pragma unroll
    for (int s = 0; s < kStages; ++s) issue_load(s);
    for (int64_t c = 0; c < chunks; ++c) {
      const int s = (int)(c % kStages), b = (int)(c & 1);
      mbar_wait(full + s, (uint32_t)((c / kStages) & 1));
      mbar_wait(consumed + b, (uint32_t)(((c >> 1) & 1) ^ 1));       // the chain warp is done with prepped tile b (first two pass)
      const float* tin = raw + s * kTileFloats + lane;
      float ax[kU], ay[kU], nanacc = 0.0f;
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        ax[u] = tin[(2 * u) * 32];
        ay[u] = tin[(2 * u + 1) * 32];
        nanacc = fmaf(ax[u], 0.0f, nanacc);
        nanacc = fmaf(ay[u], 0.0f, nanacc);
      }
      const bool careful = __any_sync(0xffffffffu, nanacc != 0.0f) || (T - c * kU) < kU;
      float2* tp = prep + b * (kU * 32) + lane;
#pragma unroll
      for (int u = 0; u < kU; ++u)
        tp[u * 32] = careful ? make_float2(ax[u], ay[u])
                             : make_float2(fminf(fmaxf(ax[u], -kMaxAction), kMaxAction), fminf(fmaxf(ay[u], -kMaxAction), kMaxAction));
      if (lane == 0) s_flag[tile][b] = careful ? 1 : 0;
      __syncwarp();
      issue_load(c + kStages);                                       // raw stage s is in registers / prepped now
      mbar_arrive(prepped + b);
      RTD3_STAMP(lane == 0 && c == 0, kStampPrepped0);
      // Out tile b is freed before the store of chunk c-1 is issued: the chain warp's wait for it at the start of chunk c then
      // depends only on the store of chunk c-2 (issued a chunk earlier), not on its own arrival at the end of chunk c-1.
      if (kTraj && c >= 2 && lane == 0) {
        bulk_wait_read<0>();                                         // the store of chunk c-2 has read its tile ...
        mbar_arrive(outfree + b);                                    // ... which is the tile chunk c will write
      }
      if (kTraj && c >= 1) {                                         // trajectory tile of the previous chunk
        const int pb = (int)((c - 1) & 1);
        mbar_wait(outfull + pb, (uint32_t)(((c - 1) >> 1) & 1));
        fence_proxy_async();
        if (lane == 0) {
          tma_store_2d(&tm_traj, (int)i0, (int)((c - 1) * (2 * kU)), outt + pb * kTileFloats);
          bulk_commit();
        }
        __syncwarp();
      }
    }
    if (kTraj) {
      const int pb = (int)((chunks - 1) & 1);
      mbar_wait(outfull + pb, (uint32_t)(((chunks - 1) >> 1) & 1));
      fence_proxy_async();
      if (lane == 0) {
        tma_store_2d(&tm_traj, (int)i0, (int)((chunks - 1) * (2 * kU)), outt + pb * kTileFloats);
        bulk_commit();
        RTD3_STAMP(true, kStampLastStore);
        if (traj_host) bulk_wait<0>();
        else bulk_wait_read<0>();
      }
      __syncwarp();
    }
    RTD3_STAMP(lane == 0, kStampHelperExit);
    return;
  }

  // ================================= chain warps =================================
  if (lane >= kLanes) return;
  const int64_t i = i0 + col;
  const bool live = i < n;
  const bool fits = __ldg(bank.fits + staged) != 0;  // lands while the table is staging
  float sx = live ? fminf(fmaxf(x[i], 0.0f), 99.99999f) : 0.0f;
  float sy = live ? fminf(fmaxf(y[i], 0.0f), 99.99999f) : 0.0f;
  const uint32_t addr_bias = smem_u32(s_table) - 0x4B000000u * (kHaloRowBytes + 8u);
  mbar_wait(bar, 0);
  RTD3_STAMP(col == 0, kStampTable);
  // Between two fast chunks nothing waits on the chain: the next chunk's barriers and careful flag are probed a few steps before
  // the end of a chunk (ready, next_careful), and its first table address is the one the last step computed (carried).
  constexpr int kProbeStep = kU - 4;
  constexpr uint32_t kPrepBytes = kU * 32 * sizeof(float2), kOutBytes = kTileFloats * sizeof(float);
  const uint32_t tp0 = smem_u32(prep + col), tout0 = smem_u32(outt + col);
  uint32_t addr = 0;
  bool carried = false, ready = false;
  int next_careful = 0;
  for (int64_t c = 0; c < chunks; ++c) {
    int b = (int)(c & 1);
    int careful = next_careful;
    if (!ready) {
      mbar_wait(prepped + b, (uint32_t)((c >> 1) & 1));
      if (kTraj && c >= 2) mbar_wait(outfree + b, (uint32_t)(((c >> 1) - 1) & 1));   // out tile b has been stored (chunk c-2)
      careful = s_flag[tile][b];
    }
    RTD3_STAMP(col == 0 && c == 0, kStampChain0);
    ready = false;
    uint32_t tp = tp0 + b * kPrepBytes, tout = tout0 + b * kOutBytes;
    auto store_state = [&](int u) {                  // the state after step u into the trajectory tile
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(tout + (2 * u) * 128u), "f"(sx) : "memory");
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(tout + (2 * u + 1) * 128u), "f"(sy) : "memory");
    };
    // Chunk c+1's prepped tile (and out tile) without blocking; a step later its careful flag, which is only used when both
    // tests passed.  No branches on the chain: at c+1 == 1 the out-tile test passes (the phase before a barrier's first one
    // counts as complete, as with mbar_wait), and at c+1 == chunks the loop ends whatever they return.
    auto probe_next = [&] {
      const uint32_t cn = (uint32_t)c + 1u;
      ready = mbar_test(prepped + (b ^ 1), (cn >> 1) & 1u);
      if (kTraj) ready &= mbar_test(outfree + (b ^ 1), ((cn >> 1) - 1u) & 1u);
    };
    auto probed_go_on = [&] { return ready && next_careful == 0 && c + 1 < chunks; };
    // Step 0 of a chunk is addressed from the state (which may be in [99, 100) after NaN actions) and step 1 from its clipped
    // successor, unless the chunk before ran this path too: its last step started from a clipped state, so the carried address
    // of its unclipped successor is as good as any inside a chunk.  Every later step is addressed from the unclipped successor
    // of the step before.  The previous step's trajectory stores follow the table load in program order: issued before it,
    // ptxas put them between the address IMAD and the load (a store may not move past a load that could alias it).  The next
    // step's action is loaded one step ahead.
    //
    // A carried run stays in this loop from chunk to chunk while the probes find the next chunk ready and fast: the last step
    // already loads the next chunk's first action, and the previous chunk's consumed / outfull arrivals go after the next
    // chunk's first table load, so the boundary adds two stores, the loop bookkeeping and one branch to the chain.
    auto fast_chunks = [&](auto from_carry) {
      float2 a = lds_f2(tp);
      if (!from_carry) addr = halo_addr_state(addr_bias, sx, sy);
      bool pending = false;                          // chunk c-1 of this run still owes its arrivals
      while (true) {
        const uint32_t tp_next = tp0 + (b ^ 1) * kPrepBytes;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const float2 cs = lds_f2(addr);
          if (u == 0 && pending) {
            mbar_arrive(consumed + (b ^ 1));
            if (kTraj) mbar_arrive(outfull + (b ^ 1));
          }
          if (kTraj && u > 0) store_state(u - 1);
          if (u == kProbeStep) probe_next();
          if (u == kProbeStep + 1) next_careful = s_flag[tile][b ^ 1];
          const float2 an = u + 1 < kU ? lds_f2(tp + (u + 1) * 256u) : from_carry ? lds_f2(tp_next) : a;
          const float nx = fmaf(a.x, cs.x, fmaf(-a.y, cs.y, sx));
          const float ny = fmaf(a.x, cs.y, fmaf(a.y, cs.x, sy));
          sx = fminf(fmaxf(nx, 0.0f), kClipHi);
          sy = fminf(fmaxf(ny, 0.0f), kClipHi);
          addr = !from_carry && u == 0 ? halo_addr(addr_bias, sx, sy) : halo_addr(addr_bias, nx, ny);
          a = an;
        }
        if (kTraj) store_state(kU - 1);
        if (!from_carry || !probed_go_on()) break;
        ++c;
        b ^= 1;
        tp = tp_next;
        tout = tout0 + b * kOutBytes;
        ready = false;
        pending = true;
      }
    };
    const bool fast = !careful && fits && !(kBank && bl.mixed);
    if (fast && carried) {
      fast_chunks(std::true_type{});
    } else if (fast) {
      fast_chunks(std::false_type{});
    } else if (kBank && bl.mixed) {
      // lanes on different maps: each steps from its own map's plain table, addressed from the state as below (a loop of its
      // own for the same reason as in env_rollout_tma_kernel)
      const int steps = (int)min((int64_t)kU, T - c * kU);
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (u < steps) {
          const float2 a = lds_f2(tp + u * 256u);
          ldg_step(bl.table, prep_action(a.x, a.y), sx, sy);
        }
        if (kTraj) store_state(u);
      }
    } else {
      // NaN / inf actions, the ragged last chunk, or a map that does not fit: every step addressed from the state
      const int steps = (int)min((int64_t)kU, T - c * kU);
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (u < steps) {
          const float2 a = lds_f2(tp + u * 256u);
          const StepIn in = prep_action(a.x, a.y);
          advance(lds_f2(halo_addr_state(addr_bias, sx, sy)), in, sx, sy);
        }
        if (kTraj) store_state(u);
      }
    }
    carried = fast;
    mbar_arrive(consumed + b);
    if (kTraj) mbar_arrive(outfull + b);
  }
  RTD3_STAMP(col == 0, kStampChainEnd);
  if (live) { x[i] = sx; y[i] = sy; }
  RTD3_STAMP(col == 0, kStampChainExit);
}

// ---- seeded init / reset on per-env legacy MT19937 streams ------------------------------------
__global__ void mt_seed_kernel(rtd3_mt_bank b, const uint32_t* __restrict__ seeds) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b.n) return;
  MtStream s{b.mt + i, b.n, 0};
  s.seed(seeds[i]);
  b.pos[i] = s.pos;
  b.has_gauss[i] = 0;
  b.gauss[i] = 0.0;
}

__global__ void mt_draw_u32_kernel(rtd3_mt_bank b, uint32_t* __restrict__ out, int64_t k) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= b.n) return;
  MtStream s{b.mt + i, b.n, b.pos[i]};
  for (int64_t j = 0; j < k; ++j) out[j * b.n + i] = s.next_u32();
  b.pos[i] = s.pos;
}

__global__ void mt_draw_gauss_kernel(rtd3_mt_bank b, double* __restrict__ out, int64_t k, const int8_t* __restrict__ where, int equals) {
  // legacy_gauss (rtd3_mt.cuh: mt_gauss) for one stream per lane, warp-synchronous so that wrapping streams are twisted by the whole
  // warp: this is the exploration noise of every tick in the exact-noise mode, and ~1 % of the streams wrap per call
  // `where` (nullable): only the streams with where[i] == equals draw - the others keep their position and get zeros (the
  // reference draws its exploration noise on 'step' ticks only, robot.py:560 via robot-learning.py:97)
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool inside = i < b.n;
  const bool active = inside && (!where || (int)where[i] == equals);
  if (inside && !active)
    for (int64_t j = 0; j < k; ++j) out[j * b.n + i] = 0.0;
  if (!__any_sync(0xffffffffu, active)) return;
  const int64_t ii = active ? i : 0;
  MtStream s{b.mt + ii, b.n, active ? b.pos[ii] : 0};
  int hg = active ? b.has_gauss[ii] : 0;
  double sp = active ? b.gauss[ii] : 0.0;
  for (int64_t j = 0; j < k; ++j) {
    double v = 0.0;
    bool searching = active && !hg;
    if (active && hg) { v = sp; sp = 0.0; hg = 0; }
    while (__any_sync(0xffffffffu, searching)) {
      double u1, u2;
      mt_next_double2_warp(s, searching, u1, u2);
      if (searching) {
        const double x1 = __dsub_rn(__dmul_rn(2.0, u1), 1.0), x2 = __dsub_rn(__dmul_rn(2.0, u2), 1.0);
        const double r2 = __dadd_rn(__dmul_rn(x1, x1), __dmul_rn(x2, x2));
        if (!(r2 >= 1.0 || r2 == 0.0)) {
          const double f = sqrt(__ddiv_rn(__dmul_rn(-2.0, log(r2)), r2));
          sp = __dmul_rn(f, x1);
          hg = 1;
          v = __dmul_rn(f, x2);
          searching = false;
        }
      }
    }
    if (active) out[j * b.n + i] = v;
  }
  if (!active) return;
  b.pos[i] = s.pos;
  b.has_gauss[i] = hg;
  b.gauss[i] = sp;
}

// environment.py:28-56
__global__ void init_goal_region_kernel(rtd3_mt_bank b, double* __restrict__ goal, double* __restrict__ region) {
  // Warp-synchronous: the goal rejection loop (acceptance ~3 %) consumes ~130 words per env on average, so a fifth of the streams
  // wrap at least once in here; with the per-lane serial twist this launch took 19 ms for 65 536 envs (ncu launch list r1).
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n = b.n;
  const bool active = i < n;
  if (!__any_sync(0xffffffffu, active)) return;
  const int64_t ii = active ? i : 0;
  MtStream s{b.mt + ii, n, active ? b.pos[ii] : 0};
  auto uni = [](double lo, double hi, double u) { return __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), u)); };   // numpy's two roundings
  const double W = (double)kWorld, R = 25.0;   // constants.py:6, 25
  const uint32_t side = mt_next_u32_warp(s, active) & 3u;   // np.random.choice([0,1,2,3]): one masked draw, never rejected
  const double free_edge = uni(0.0, W - R, mt_next_double_warp(s, active));
  double l, r, bt, tp;
  if (side == 0)      { l = 0.0;       r = R;            bt = free_edge; tp = __dadd_rn(free_edge, R); }
  else if (side == 1) { l = free_edge; r = __dadd_rn(free_edge, R); bt = W - R; tp = W; }
  else if (side == 2) { l = W - R;     r = W;            bt = free_edge; tp = __dadd_rn(free_edge, R); }
  else                { l = free_edge; r = __dadd_rn(free_edge, R); bt = 0.0;   tp = R; }
  const double mx = __dmul_rn(0.5, __dadd_rn(l, r)), my = __dmul_rn(0.5, __dadd_rn(bt, tp));
  double gx = 0.0, gy = 0.0;
  bool searching = active;
  while (__any_sync(0xffffffffu, searching)) {
    double ux, uy;
    mt_next_double2_warp(s, searching, ux, uy);
    if (searching) {
      gx = uni(5.0, W - 5.0, ux);
      gy = uni(5.0, W - 5.0, uy);
      if (!(norm2_np(__dsub_rn(gx, mx), __dsub_rn(gy, my)) < 90.0)) searching = false;
    }
  }
  if (!active) return;
  goal[i] = gx; goal[n + i] = gy;
  region[i] = l; region[n + i] = r; region[2 * n + i] = bt; region[3 * n + i] = tp;
  b.pos[i] = s.pos;
}

// environment.py:130-137
__global__ void env_reset_kernel(rtd3_mt_bank b, const double* __restrict__ region, const uint8_t* __restrict__ mask, int mask_equals,
                                 float* __restrict__ x, float* __restrict__ y, double* __restrict__ state64) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < b.n && (!mask || (mask_equals >= 0 ? mask[i] == (uint8_t)mask_equals : mask[i] != 0));
  reset_env_warp(b, region, active, i, x, y, state64);
}

static int32_t check_bank(const rtd3_mt_bank* b) {
  RTD3_CHECK_ARG(b && b->mt && b->pos && b->has_gauss && b->gauss, "null MT bank pointer");
  RTD3_CHECK_ARG(b->n >= 0, "negative stream count");
  return 0;
}

}  // namespace rtd3

using namespace rtd3;

static int g_rollout_hook = 0;   // rtd3_env_force_plain_rollout: 1 = the cp.async kernel, 2 = the single-warp TMA kernel for every size
static bool g_launch_overlap = true;   // rtd3_env_set_launch_overlap

// Every kernel instantiation a launch can pick.  The launches index these tables, and rtd3_env_create sets the shared-memory
// limit of every entry.
// env_step_kernel, [table][keep_on_nan]; table 0: read-only path, 1: staged in shared memory, 2: each env's own map of the bank
using StepKernel = decltype(&env_step_kernel<false, false>);
static const StepKernel kStepKernels[3][2] = {{env_step_kernel<false, false>, env_step_kernel<false, true>},
                                              {env_step_kernel<true, false>, env_step_kernel<true, true>},
                                              {env_step_kernel<false, false, true>, env_step_kernel<false, true, true>}};
// rollout kernels, [bank][traj][stages]; stages 1: kDeep (latency-bound batches), 0: kShallow
using RolloutKernel = decltype(&env_rollout_kernel<false, kDeep>);
static const RolloutKernel kRolloutKernels[2][2][2] = {
    {{env_rollout_kernel<false, kShallow>, env_rollout_kernel<false, kDeep>},
     {env_rollout_kernel<true, kShallow>, env_rollout_kernel<true, kDeep>}},
    {{env_rollout_kernel<false, kShallow, true>, env_rollout_kernel<false, kDeep, true>},
     {env_rollout_kernel<true, kShallow, true>, env_rollout_kernel<true, kDeep, true>}}};
using TmaKernel = decltype(&env_rollout_tma_kernel<false, kDeep>);
static const TmaKernel kTmaKernels[2][2][2] = {
    {{env_rollout_tma_kernel<false, kShallow>, env_rollout_tma_kernel<false, kDeep>},
     {env_rollout_tma_kernel<true, kShallow>, env_rollout_tma_kernel<true, kDeep>}},
    {{env_rollout_tma_kernel<false, kShallow, true>, env_rollout_tma_kernel<false, kDeep, true>},
     {env_rollout_tma_kernel<true, kShallow, true>, env_rollout_tma_kernel<true, kDeep, true>}}};
// pair kernel, [bank][traj][two tiles per CTA]
using PairKernel = decltype(&env_rollout_pair_kernel<false, kPairStages, kPairU, kChainLanes>);
static const PairKernel kPairKernels[2][2][2] = {
    {{env_rollout_pair_kernel<false, kPairStages, kPairU, kChainLanes>, env_rollout_pair_kernel<false, kPairStages2, kPairU, kChainLanes>},
     {env_rollout_pair_kernel<true, kPairStages, kPairU, kChainLanes>, env_rollout_pair_kernel<true, kPairStages2, kPairU, kChainLanes>}},
    {{env_rollout_pair_kernel<false, kPairStages, kPairU, kChainLanes, true>, env_rollout_pair_kernel<false, kPairStages2, kPairU, kChainLanes, true>},
     {env_rollout_pair_kernel<true, kPairStages, kPairU, kChainLanes, true>, env_rollout_pair_kernel<true, kPairStages2, kPairU, kChainLanes, true>}}};

// A rollout launch; with `overlap` it may start while the stream's previous kernel drains (programmatic dependent launch, see
// env_rollout_pair_kernel).
template <typename... KArgs, typename... Args>
static cudaError_t launch_rollout(void (*kernel)(KArgs...), int grid, int block, int smem, cudaStream_t st, bool overlap, Args&&... args) {
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = &attr;
  cfg.numAttrs = overlap ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

template <typename... Args>
static cudaError_t set_max_smem(void (*kernel)(Args...), int bytes) {
  return cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
}
template <typename T, size_t N>
static cudaError_t set_max_smem(const T (&kernels)[N], int bytes) {
  for (const T& k : kernels)
    if (cudaError_t e = set_max_smem(k, bytes)) return e;
  return cudaSuccess;
}

// cuTensorMapEncodeTiled comes from the driver (libcuda); it is looked up at run time so that librtd3.so links against
// the runtime only.  If the lookup fails the rollout falls back to the cp.async kernel.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode_tiled = nullptr;

static void load_encode_tiled() {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
    g_encode_tiled = (EncodeTiledFn)fn;
}

// [T][2][n] float32 planes as a 2-D tensor: inner dim n, outer dim 2T, box = 32 envs x 2*steps_per_tile rows
static int32_t make_plane_map(CUtensorMap* tm, const float* base, int64_t n, int64_t T, int steps_per_tile) {
  const cuuint64_t dims[2] = {(cuuint64_t)n, (cuuint64_t)(2 * T)};
  const cuuint64_t strides[1] = {(cuuint64_t)n * 4};
  const cuuint32_t box[2] = {32, (cuuint32_t)(2 * steps_per_tile)};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = g_encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    rtd3::set_error("cuTensorMapEncodeTiled failed (%d)", (int)r);
    return RTD3_ERR_STATE;
  }
  return 0;
}

// (Re)allocates the bank for `cap` maps (synchronous: kernels in flight may read the old bank).  The contents are not kept.
static int32_t alloc_bank(rtd3_env* h, int cap) {
  if (h->tables) {
    rtd3::host_pipe_drop_graphs(h);   // they hold the old bank addresses
    cudaDeviceSynchronize();
    cudaFree(h->tables);
    cudaFree(h->halos);
    cudaFree(h->fits);
  }
  h->tables = h->halos = nullptr;
  h->fits = nullptr;
  h->map_cap = h->num_maps = 0;
  RTD3_CUDA(cudaMalloc(&h->tables, (size_t)cap * kTableBytes));
  RTD3_CUDA(cudaMalloc(&h->halos, (size_t)cap * kHaloBytes));
  RTD3_CUDA(cudaMalloc(&h->fits, (size_t)cap * sizeof(int)));
  h->map_cap = cap;
  return 0;
}

extern "C" {

void rtd3_env_force_plain_rollout(int32_t on) { g_rollout_hook = on == 1 || on == 2 ? on : 0; }
void rtd3_env_set_launch_overlap(int32_t on) { g_launch_overlap = on != 0; }

int32_t rtd3_env_create(rtd3_env** out, int32_t device) {
  RTD3_CHECK_ARG(out, "out is null");
  DeviceGuard guard;
  RTD3_CUDA(guard.enter(device));
  std::unique_ptr<rtd3_env, int32_t (*)(rtd3_env*)> h(new rtd3_env(), rtd3_env_destroy);   // freed on every error return
  h->device = device;
  RTD3_CUDA(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device));
  if (int32_t e = alloc_bank(h.get(), 1)) return e;
  if (!g_encode_tiled) load_encode_tiled();
  RTD3_CUDA(set_max_smem(kStepKernels[1], kTableBytes + 16));
  const int smem_roll = 227 * 1024;
  RTD3_CUDA(set_max_smem(kRolloutKernels, smem_roll));
  RTD3_CUDA(set_max_smem(kTmaKernels, smem_roll));
  RTD3_CUDA(set_max_smem(kPairKernels, smem_roll - 1024));
  *out = h.release();
  return 0;
}

int32_t rtd3_env_destroy(rtd3_env* h) {
  if (!h) return 0;
  rtd3::host_pipe_destroy(h);
  if (h->tables) cudaFree(h->tables);
  if (h->halos) cudaFree(h->halos);
  if (h->fits) cudaFree(h->fits);
  if (h->index) cudaFree(h->index);
  delete h;
  return 0;
}

int32_t rtd3_env_set_maps(rtd3_env* h, const float* speed, const float* angle, int32_t K, void* stream) {
  RTD3_CHECK_ARG(h && speed && angle, "null argument");
  RTD3_CHECK_ARG(K >= 1 && K <= kMaxMaps, "map count K must be in [1, 65536]");
  if (K > h->map_cap) {
    DeviceGuard guard;
    RTD3_CUDA(guard.enter(h->device));
    if (int32_t e = alloc_bank(h, K)) return e;
  }
  const int64_t cells = (int64_t)K * kCells;
  build_table_kernel<<<(int)ceil_div(cells, 256), 256, 0, (cudaStream_t)stream>>>(speed, angle, h->tables, cells);
  RTD3_LAUNCHED();
  build_halo_kernel<<<K, 1024, 0, (cudaStream_t)stream>>>(h->tables, h->halos, h->fits);
  RTD3_LAUNCHED();
  h->num_maps = K;
  h->maps_rebuilt = true;
  return 0;
}

int32_t rtd3_env_set_map(rtd3_env* h, const float* speed, const float* angle, void* stream) {
  if (int32_t e = rtd3_env_set_maps(h, speed, angle, 1, stream)) return e;
  return rtd3_env_set_map_index(h, nullptr, 0, stream);
}

int32_t rtd3_env_set_map_index(rtd3_env* h, const int32_t* index, int64_t m, void* stream) {
  RTD3_CHECK_ARG(h, "null handle");
  RTD3_CHECK_ARG(m >= 0, "negative index length");
  if (!index || m == 0) {
    h->index_len = 0;
    return 0;
  }
  if (m > h->index_cap) {
    DeviceGuard guard;
    RTD3_CUDA(guard.enter(h->device));
    rtd3::host_pipe_drop_graphs(h);   // they hold the old index address
    cudaDeviceSynchronize();          // kernels in flight may still read the old index
    if (h->index) cudaFree(h->index);
    h->index = nullptr;
    h->index_len = h->index_cap = 0;
    const cudaError_t ce = cudaMalloc(&h->index, (size_t)m * sizeof(int32_t));
    if (ce != cudaSuccess) {
      rtd3::set_error("cudaMalloc of a %lld-entry map index -> %s", (long long)m, cudaGetErrorString(ce));
      return (int32_t)ce;
    }
    h->index_cap = m;
  }
  RTD3_CUDA(cudaMemcpyAsync(h->index, index, (size_t)m * sizeof(int32_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  h->index_len = m;
  return 0;
}

int32_t rtd3_env_map_config(const rtd3_env* h, const void** tables, const void** index, int32_t* num_maps, int64_t* index_len) {
  RTD3_CHECK_ARG(h, "null handle");
  const MapBank b = map_bank(h);
  if (tables) *tables = b.tables;
  if (index) *index = b.index;
  if (num_maps) *num_maps = b.K;
  if (index_len) *index_len = b.m;
  return 0;
}

static int32_t launch_step(rtd3_env* h, const float* x, const float* y, const float* ax, const float* ay, float* ox,
                           float* oy, int64_t n, int32_t variant, bool keep_on_nan, cudaStream_t st) {
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(n >= 0, "negative n");
  if (n == 0) return 0;
  RTD3_CHECK_ARG(x && y && ax && ay && ox && oy, "null state/action pointer");
  const int vec_ok =
      (((uintptr_t)x | (uintptr_t)y | (uintptr_t)ax | (uintptr_t)ay | (uintptr_t)ox | (uintptr_t)oy) % 16 == 0) ? 1 : 0;
  RTD3_CHECK_ARG(variant >= RTD3_STEP_AUTO && variant <= RTD3_STEP_LDG, "unknown step variant");
  const int64_t n4 = vec_ok ? (n + 3) / 4 : n;
  if (variant == RTD3_STEP_AUTO) variant = (n >= 262144) ? RTD3_STEP_SMEM : RTD3_STEP_LDG;
  const MapBank bank = map_bank(h);
  // with an index there is one table per env and none to stage: every variant reads through the read-only path
  const bool smem = !bank.index && variant == RTD3_STEP_SMEM;
  const int block = smem ? 512 : 256;
  const int grid = (int)std::min<int64_t>(ceil_div(n4, block), (int64_t)h->num_sms * (smem ? 2 : 4));
  const StepKernel kern = kStepKernels[bank.index ? 2 : smem ? 1 : 0][keep_on_nan];
  kern<<<grid, block, smem ? kTableBytes + 16 : 0, st>>>(vec_ok, x, y, ax, ay, ox, oy, n, bank);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_env_step(rtd3_env* h, float* x, float* y, const float* ax, const float* ay, int64_t n, int32_t variant,
                      void* stream) {
  return launch_step(h, x, y, ax, ay, x, y, n, variant, true, (cudaStream_t)stream);
}

int32_t rtd3_env_dynamics(rtd3_env* h, const float* x, const float* y, const float* ax, const float* ay, float* out_x,
                          float* out_y, int64_t n, void* stream) {
  return launch_step(h, x, y, ax, ay, out_x, out_y, n, RTD3_STEP_AUTO, false, (cudaStream_t)stream);
}

int32_t rtd3_env_rollout(rtd3_env* h, float* x, float* y, const float* actions, float* traj, int64_t n, int64_t T,
                         void* stream) {
  // a trajectory in host (or managed) memory: the kernel waits for its writes to complete before exiting
  bool traj_host = false;
  if (traj) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, traj) != cudaSuccess) cudaGetLastError();
    else traj_host = a.type != cudaMemoryTypeDevice;
  }
  return env_rollout(h, x, y, actions, traj, n, T, traj_host, (cudaStream_t)stream);
}

}  // extern "C"

int32_t rtd3::env_rollout(rtd3_env* h, float* x, float* y, const float* actions, float* traj, int64_t n, int64_t T, bool traj_host,
                          cudaStream_t st) {
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(n >= 0 && T >= 0, "negative n or T");
  if (n == 0 || T == 0) return 0;
  RTD3_CHECK_ARG(x && y && actions, "null state/action pointer");
  // Small batches are latency-bound (one dependent chain per env): spread them over all SMs in CTAs as small as a
  // warp and keep kDeep chunks of actions in flight per thread.  Large batches hide latency with occupancy instead:
  // 128-thread CTAs, kShallow chunks in flight, up to 2 CTAs per SM next to the 80 KB table.
  const int64_t per_sm = ceil_div(n, (int64_t)h->num_sms);
  const bool deep = per_sm <= 64;
  const int stages = deep ? kDeep : kShallow;
  // Launch overlap (see env_rollout_pair_kernel) needs the tables unchanged since the previous rollout launch.  A captured launch
  // runs without it (a graph may replay a table rebuild or be launched after any work), and leaves the flag set for the next one.
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) {
    cudaGetLastError();
    cap = cudaStreamCaptureStatusActive;
  }
  const bool capturing = cap != cudaStreamCaptureStatusNone;
  const bool overlap = g_launch_overlap && !h->maps_rebuilt && !capturing;
  h->maps_rebuilt = capturing;
  const int th = traj_host ? 1 : 0;
  const MapBank bank = map_bank(h);   // bank.index == nullptr: the single-map kernels
  const bool with_bank = bank.index != nullptr, with_traj = traj != nullptr;
  // latency-bound batches run the warp-pair kernel, with tiles of kPairU steps (the per-tile hand-over - two barrier waits, the
  // flag read, two arrives - was ~20 % of the chain warp's samples at 16)
  const bool pair = deep && g_rollout_hook != 2;
  const bool tma_ok = (n % 4 == 0) && (n < (1ll << 31)) && (2 * T < (1ll << 31)) && ((uintptr_t)actions % 16 == 0) &&
                      (!traj || (uintptr_t)traj % 16 == 0) && g_rollout_hook != 1 && g_encode_tiled;
  CUtensorMap tm_act, tm_traj;
  const int tile_steps = pair ? kPairU : kU;
  // an encode failure (unexpected shape limits) is not an error: the cp.async kernel below handles every shape
  if (tma_ok && make_plane_map(&tm_act, actions, n, T, tile_steps) == 0 &&
      make_plane_map(&tm_traj, traj ? traj : actions, n, T, tile_steps) == 0) {
    const int64_t warps_total = ceil_div(n, 32);
    if (pair) {
      // chain warps + one helper warp per 32-env tile, up to 2 tiles per CTA
      const int tpc = (int)std::max<int64_t>(1, std::min<int64_t>(2, ceil_div(warps_total, (int64_t)h->num_sms)));
      const int pstages = tpc == 1 ? kPairStages : kPairStages2;
      const int psmem = ((kHaloBytes + 16 + tpc * PairSmem::kBars * 8 + 127) & ~127) + tpc * (pstages + 4) * (kPairU * 2 * 32) * 4;
      const PairKernel kern = kPairKernels[with_bank][with_traj][tpc == 2];
      RTD3_CUDA(launch_rollout(kern, (int)ceil_div(warps_total, tpc), tpc * pair_warps(kChainLanes) * 32, psmem, st, overlap, x, y, tm_act,
                               tm_traj, n, T, bank, th));
    } else {
      // one warp per 32 envs; few warps per CTA while the batch cannot fill the SMs, 8 once it can
      const int wpc = deep ? (int)std::max<int64_t>(1, std::min<int64_t>(8, ceil_div(warps_total, (int64_t)h->num_sms))) : 8;
      const int bsmem = ((kTableBytes + 16 + wpc * stages * 8 + 127) & ~127) + wpc * (stages + 2) * kTileFloats * 4;
      const TmaKernel kern = kTmaKernels[with_bank][with_traj][deep];
      RTD3_CUDA(launch_rollout(kern, (int)ceil_div(warps_total, wpc), wpc * 32, bsmem, st, overlap, n, x, y, tm_act, tm_traj, T, bank, th));
    }
    RTD3_LAUNCHED();
    return 0;
  }
  const int block = deep ? (int)std::max<int64_t>(32, ceil_div(per_sm, 32) * 32) : 128;
  const int smem = kTableBytes + 16 + stages * kU * 2 * block * 4;
  const RolloutKernel kern = kRolloutKernels[with_bank][with_traj][deep];
  RTD3_CUDA(launch_rollout(kern, (int)ceil_div(n, block), block, smem, st, overlap, n, x, y, actions, traj, T, bank));
  RTD3_LAUNCHED();
  return 0;
}

extern "C" {

int32_t rtd3_mt_seed(const rtd3_mt_bank* bank, const uint32_t* seeds, void* stream) {
  if (int32_t e = check_bank(bank)) return e;
  RTD3_CHECK_ARG(seeds, "null seeds");
  if (bank->n == 0) return 0;
  mt_seed_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, seeds);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_mt_draw_u32(const rtd3_mt_bank* bank, uint32_t* out, int64_t k, void* stream) {
  if (int32_t e = check_bank(bank)) return e;
  RTD3_CHECK_ARG(out && k >= 0, "bad out/k");
  if (bank->n == 0 || k == 0) return 0;
  mt_draw_u32_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, out, k);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_mt_draw_gauss(const rtd3_mt_bank* bank, double* out, int64_t k, void* stream) {
  return rtd3_mt_draw_gauss_where(bank, out, k, nullptr, 0, stream);
}

int32_t rtd3_mt_draw_gauss_where(const rtd3_mt_bank* bank, double* out, int64_t k, const int8_t* where, int32_t equals, void* stream) {
  if (int32_t e = check_bank(bank)) return e;
  RTD3_CHECK_ARG(out && k >= 0, "bad out/k");
  if (bank->n == 0 || k == 0) return 0;
  mt_draw_gauss_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, out, k, where, equals);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_env_init_goal_region(const rtd3_mt_bank* bank, double* goal, double* region, void* stream) {
  if (int32_t e = check_bank(bank)) return e;
  RTD3_CHECK_ARG(goal && region, "null output");
  if (bank->n == 0) return 0;
  init_goal_region_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, goal, region);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_env_reset(const rtd3_mt_bank* bank, const double* region, const uint8_t* mask, int32_t mask_equals, float* x, float* y,
                       double* state64, void* stream) {
  if (int32_t e = check_bank(bank)) return e;
  RTD3_CHECK_ARG(region && x && y, "null argument");
  if (bank->n == 0) return 0;
  env_reset_kernel<<<(int)ceil_div(bank->n, 128), 128, 0, (cudaStream_t)stream>>>(*bank, region, mask, mask_equals, x, y, state64);
  RTD3_LAUNCHED();
  return 0;
}

#ifdef RTD3_ROLLOUT_STAMPS
// Arms the phase stamps of env_rollout_pair_kernel: records go to buf [cap][kStampWords] (device memory, zeroed by the caller) in
// CTA start order.  Not part of the ABI: only the stamped build exports it.
int32_t rtd3_rollout_stamps_arm(void* buf, int64_t cap) {
  unsigned long long* p = (unsigned long long*)buf;
  const unsigned long long zero = 0, c = (unsigned long long)cap;
  RTD3_CUDA(cudaMemcpyToSymbol(g_stamps, &p, sizeof(p)));
  RTD3_CUDA(cudaMemcpyToSymbol(g_stamp_next, &zero, sizeof(zero)));
  RTD3_CUDA(cudaMemcpyToSymbol(g_stamp_cap, &c, sizeof(c)));
  return 0;
}
int32_t rtd3_rollout_stamp_words() { return kStampWords; }
#endif

}  // extern "C"
