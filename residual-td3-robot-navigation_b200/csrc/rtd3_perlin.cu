// The reference's Perlin maps (environment.py:59-95, restated as `perlin_maps` in environment.py of this package) for a list of
// seeds: one CTA per map.  Exactness rules (rtd3.h): the float32 fields before normalisation and `angle` equal the host's bit for
// bit; `speed` follows numpy's float32 operation order with exp evaluated in float64 and rounded once.
//
// What the host computes, per map of seed s:
//   - the gradient of lattice corner (cx, cy) is the first two `uniform(-1, 1)` draws of Python's `random.Random(s * h)`,
//     h = cx + 10 cy + 1.  Over the octaves 5, 10 and 20 h takes the values 1..221, and all four noise instances (speed's three
//     octaves and angle's one) share the seed, so a map needs 221 gradients;
//   - a cell's noise sums, over its four corners in the order (x0,y0), (x0,y1), (x1,y0), (x1,y1), the weight
//     fade(1-|dx|) * fade(1-|dy|) times the dot product g0*dx + g1*dy, in float64 from 0.0, with fade(t) = 6 t^5 - 15 t^4 + 10 t^3
//     and Python's (correctly rounded) powers;
//   - speed's field is n(5) + 0.5 n(10) + 0.25 n(20), angle's n(5), each rounded once to float32; both are min-max normalised in
//     float32 and speed is then stretched by 1 / (1 + exp(-10 (norm - 0.5))).
// Every float64 and float32 step is an explicit _rn intrinsic: nvcc would otherwise contract products and sums into FMAs.
#include "rtd3_common.cuh"
#include "rtd3_mt.cuh"

namespace {

using namespace rtd3;

constexpr int kThreads = 256;
constexpr int kOctaves = 3;                        // 5, 10, 20 (angle uses octave 5 again)
constexpr int kHashes = 221;                       // h = cx + 10 cy + 1 over the lattice corners of octave 20
constexpr int kWarps = kThreads / 32;

bool g_raw_fields = false;                         // rtd3_perlin_set_raw_fields

// ---- Python's random.Random(n).uniform(-1, 1), twice ---------------------------------------------------------------------------
// random.Random(n) seeds MT19937 by init_by_array over the 32-bit words of n (at least one).  The first four outputs, which make
// the two doubles, read state words 0..4 and 397..400 after init_by_array, so the 624-word state is never stored: the key-mixing
// loops run as register recurrences.  The second loop starts from the word 1 that the first loop rewrites after it wraps (that
// value depends on word 623), so the first loop runs once to its end and then again in lockstep with the second.
__device__ __forceinline__ uint32_t init_next(uint32_t prev, uint32_t i) { return 1812433253u * (prev ^ (prev >> 30)) + i; }
__device__ __forceinline__ uint32_t mix1(uint32_t cur, uint32_t prev, uint32_t add) {
  return (cur ^ ((prev ^ (prev >> 30)) * 1664525u)) + add;
}
__device__ __forceinline__ uint32_t mix2(uint32_t cur, uint32_t prev, uint32_t i) {
  return (cur ^ ((prev ^ (prev >> 30)) * 1566083941u)) - i;
}

// The first loop adds key[j] + j with j = iteration % key length (1, 2 or 3): a window of six addends, rotated each iteration,
// serves all three lengths (the compiler renames it away in the unrolled loops).
struct KeyAddends {
  uint32_t a[6];
  __device__ __forceinline__ uint32_t take() {
    const uint32_t v = a[0];
#pragma unroll
    for (int q = 0; q < 5; ++q) a[q] = a[q + 1];
    a[5] = v;
    return v;
  }
};

__device__ __forceinline__ void python_gradient(uint64_t n_lo, uint64_t n_hi, double& g0, double& g1) {
  const uint32_t len = n_hi ? 3u : ((n_lo >> 32) ? 2u : 1u);
  KeyAddends add0;
#pragma unroll
  for (uint32_t q = 0; q < 6; ++q) {
    const uint32_t j = len == 1 ? 0u : len == 2 ? q % 2 : q % 3;   // q % len with q a constant: no division
    add0.a[q] = (j == 0 ? (uint32_t)n_lo : j == 1 ? (uint32_t)(n_lo >> 32) : (uint32_t)n_hi) + j;
  }

  // first loop, once through: i = 1..623, then the wrap (word 0 := word 623) and i = 1 again
  KeyAddends add = add0;
  uint32_t m = 19650218u, a = m;                   // init_genrand word i-1 / first-loop word i-1 (word 0 before the wrap)
  m = init_next(m, 1);
  a = mix1(m, a, add.take());
  const uint32_t m1 = m, a1 = a;                   // init_genrand word 1, first-loop word 1
#pragma unroll 6
  for (uint32_t i = 2; i < RTD3_MT_N; ++i) {
    m = init_next(m, i);
    a = mix1(m, a, add.take());
  }
  const uint32_t a1w = mix1(a1, a, add.take());    // word 1 after the wrap

  // first loop again (i = 2..623, the words the second loop reads) in lockstep with the second loop, which starts at i = 2 from
  // word 1 = a1w; it keeps words 2..4 and 397..400, then wraps (word 0 := word 623) and rewrites word 1
  add = add0;
  add.take();
  m = m1;
  a = a1;
  uint32_t b = a1w;
  uint32_t w[9];                                   // final words 0..4, 397..400
  auto both = [&](uint32_t i) {
    m = init_next(m, i);
    a = mix1(m, a, add.take());
    b = mix2(a, b, i);
  };
#pragma unroll
  for (uint32_t i = 2; i <= 4; ++i) {
    both(i);
    w[i] = b;
  }
#pragma unroll 6
  for (uint32_t i = 5; i < 397; ++i) both(i);
#pragma unroll
  for (uint32_t i = 397; i <= 400; ++i) {
    both(i);
    w[5 + i - 397] = b;
  }
#pragma unroll 6
  for (uint32_t i = 401; i < RTD3_MT_N; ++i) both(i);
  w[1] = mix2(a1w, b, 1);
  w[0] = 0x80000000u;

  // genrand outputs 0..3: the twist of words 0..3 (they pair with words 1..4 and 397..400) and the tempering
  uint32_t out[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t y = (w[k] & 0x80000000u) | (w[k + 1] & 0x7fffffffu);
    out[k] = mt_temper(w[5 + k] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u));
  }
  g0 = __dadd_rn(-1.0, __dmul_rn(2.0, mt_double_from_words(out[0], out[1])));   // uniform(-1, 1) = -1 + 2 * random()
  g1 = __dadd_rn(-1.0, __dmul_rn(2.0, mt_double_from_words(out[2], out[3])));
}

// ---- correctly rounded t^3, t^4, t^5 ---------------------------------------------------------------------------------------------
// Python's `t ** n` is the host's pow, correctly rounded for every fade argument of these maps; CUDA's pow is not.  The powers are
// carried as unevaluated sums hi + lo (each product's rounding error recovered exactly with an FMA) and rounded once at the end;
// the carried error (~2^-100 relative) can only matter within that distance of a rounding boundary, and the tests compare every
// fade argument against the host.
__device__ __forceinline__ void powers345(double t, double& p3, double& p4, double& p5) {
  double hi = __dmul_rn(t, t);
  double lo = __fma_rn(t, t, -hi);
  double q[3];
#pragma unroll
  for (int n = 0; n < 3; ++n) {
    const double h = __dmul_rn(hi, t);
    lo = __dadd_rn(__fma_rn(hi, t, -h), __dmul_rn(lo, t));
    hi = h;
    q[n] = __dadd_rn(hi, lo);
  }
  p3 = q[0];
  p4 = q[1];
  p5 = q[2];
}

__device__ __forceinline__ double fade(double t) {   // 6 * t**5 - 15 * t**4 + 10 * t**3, left to right
  double p3, p4, p5;
  powers345(t, p3, p4, p5);
  return __dadd_rn(__dsub_rn(__dmul_rn(6.0, p5), __dmul_rn(15.0, p4)), __dmul_rn(10.0, p3));
}

// One axis of one octave at grid index c (the same for x and y): p = (c / 100) * octave, lattice corners floor(p) and floor(p + 1),
// offsets p - corner and weights fade(1 - |offset|).
struct Axis {
  double d[2], f[2];
  int c[2];
};

struct Smem {
  double2 grad[kHashes];                           // gradient of hash h at [h - 1]
  Axis axis[kOctaves][kWorld];
  float red[4][kWarps];
};

__device__ __forceinline__ double noise(const Smem& sm, int o, int col, int row) {
  const Axis& X = sm.axis[o][col];
  const Axis& Y = sm.axis[o][row];
  double total = 0.0;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const double2 g = sm.grad[X.c[i] + 10 * Y.c[j]];
      const double dot = __dadd_rn(__dadd_rn(0.0, __dmul_rn(g.x, X.d[i])), __dmul_rn(g.y, Y.d[j]));   // sum() starts at 0
      total = __dadd_rn(total, __dmul_rn(__dmul_rn(X.f[i], Y.f[j]), dot));
    }
  }
  return total;
}

__device__ __forceinline__ void block_min_max(Smem& sm, float v[4]) {   // v: speed min, speed max, angle min, angle max
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    v[0] = fminf(v[0], __shfl_xor_sync(0xffffffffu, v[0], s));
    v[1] = fmaxf(v[1], __shfl_xor_sync(0xffffffffu, v[1], s));
    v[2] = fminf(v[2], __shfl_xor_sync(0xffffffffu, v[2], s));
    v[3] = fmaxf(v[3], __shfl_xor_sync(0xffffffffu, v[3], s));
  }
  if (lane == 0)
#pragma unroll
    for (int q = 0; q < 4; ++q) sm.red[q][warp] = v[q];
  __syncthreads();
#pragma unroll
  for (int q = 0; q < 4; ++q) v[q] = sm.red[q][0];
  for (int w = 1; w < kWarps; ++w) {
    v[0] = fminf(v[0], sm.red[0][w]);
    v[1] = fmaxf(v[1], sm.red[1][w]);
    v[2] = fminf(v[2], sm.red[2][w]);
    v[3] = fmaxf(v[3], sm.red[3][w]);
  }
}

// 4 CTAs per SM: 64 registers and no spills (with the register target ptxas picks for 256 threads alone it spilled 8 bytes)
__global__ void __launch_bounds__(kThreads, 4) perlin_maps_kernel(const int64_t* __restrict__ seeds, float* __restrict__ speed,
                                                               float* __restrict__ angle, int raw) {
  __shared__ Smem sm;
  const int tid = threadIdx.x;
  const uint64_t seed = (uint64_t)seeds[blockIdx.x];
  float* sp = speed + (int64_t)blockIdx.x * kCells;
  float* an = angle + (int64_t)blockIdx.x * kCells;

  if (tid < kHashes) {                             // seed * h < 2^71: a 128-bit product
    const uint64_t h = (uint64_t)(tid + 1);
    double g0, g1;
    python_gradient(seed * h, __umul64hi(seed, h), g0, g1);
    sm.grad[tid] = make_double2(g0, g1);
  }
  for (int e = tid; e < kOctaves * kWorld; e += kThreads) {
    const int o = e / kWorld, c = e - o * kWorld;
    const double p = __dmul_rn(__ddiv_rn((double)c, (double)kWorld), (double)(5 << o));   // (col / W) * octave
    Axis ax;
    ax.c[0] = (int)floor(p);
    ax.c[1] = (int)floor(__dadd_rn(p, 1.0));
#pragma unroll
    for (int i = 0; i < 2; ++i) {
      ax.d[i] = __dsub_rn(p, (double)ax.c[i]);
      ax.f[i] = fade(__dsub_rn(1.0, fabs(ax.d[i])));
    }
    sm.axis[o][c] = ax;
  }
  __syncthreads();

  // the fields before normalisation, stored in place; the same thread reads its cells back after the min-max reduction
  float v[4] = {INFINITY, -INFINITY, INFINITY, -INFINITY};
  for (int cell = tid; cell < kCells; cell += kThreads) {
    const int col = cell / kWorld, row = cell - col * kWorld;
    const double n5 = noise(sm, 0, col, row), n10 = noise(sm, 1, col, row), n20 = noise(sm, 2, col, row);
    const float s = __double2float_rn(__dadd_rn(__dadd_rn(n5, __dmul_rn(0.5, n10)), __dmul_rn(0.25, n20)));
    const float a = __double2float_rn(n5);
    sp[cell] = s;
    an[cell] = a;
    v[0] = fminf(v[0], s);
    v[1] = fmaxf(v[1], s);
    v[2] = fminf(v[2], a);
    v[3] = fmaxf(v[3], a);
  }
  if (raw) return;
  block_min_max(sm, v);
  const float s_range = __fsub_rn(v[1], v[0]), a_range = __fsub_rn(v[3], v[2]);   // 0 for a flat field: NaN cells, as in numpy
  for (int cell = tid; cell < kCells; cell += kThreads) {
    const float norm = __fdiv_rn(__fsub_rn(sp[cell], v[0]), s_range);
    const float x = __fmul_rn(-10.0f, __fsub_rn(norm, 0.5f));
    const float e = __double2float_rn(exp((double)x));
    sp[cell] = __fdiv_rn(1.0f, __fadd_rn(1.0f, e));
    an[cell] = __fdiv_rn(__fsub_rn(an[cell], v[2]), a_range);
  }
}

}  // namespace

extern "C" {

void rtd3_perlin_set_raw_fields(int32_t on) { g_raw_fields = on != 0; }

int32_t rtd3_perlin_maps(const int64_t* seeds, int32_t K, float* speed, float* angle, void* stream) {
  RTD3_CHECK_ARG(seeds && speed && angle, "null argument");
  RTD3_CHECK_ARG(K >= 1 && K <= kMaxMaps, "map count K must be in [1, 65536]");
  perlin_maps_kernel<<<K, kThreads, 0, (cudaStream_t)stream>>>(seeds, speed, angle, g_raw_fields ? 1 : 0);
  RTD3_LAUNCHED();
  return 0;
}

}  // extern "C"
