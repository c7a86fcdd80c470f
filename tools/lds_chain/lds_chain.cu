// Standalone probe: cycles per link of a dependent chain of 8-byte shared-memory gathers (LDS.64) on sm_100, by the number of
// active lanes per warp.  The table is the shape of the rollout pair kernel's halo table (116 x 116 float2 = 107 648 B); every
// lane walks it from its own start, so the lanes of one load hit unrelated cells and share banks as chance has it.
//   lds   : each entry holds the shared-memory address of the next entry (LDS.64 -> LDS.64, no arithmetic in between)
//   lds_nc: the same chain without bank conflicts: entry e links to an entry of the same bank pair (e % 16), and lane l of a
//           half-warp walks bank pair l % 16 - the bare latency of the load, for comparison
//   step  : the fast-path step of env_rollout_pair_kernel (csrc/rtd3_env.cu) - table load, two FFMAs per axis, FADD.RZ, IMADs,
//           the next step's action loaded one step ahead and the trajectory stores - over a random map that fits the halo
// Each configuration runs `warps` chain warps of `lanes` active lanes per CTA, one CTA per SM (the dynamic shared memory is more
// than half the SM's), timed with clock64 by lane 0 of every warp.  warps x lanes = 32 is the arrangement of one 32-env tile.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o lds_chain lds_chain.cu ; run on a B200: ./lds_chain [links]
// Prints one JSON line.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

#define CK(x)                                                                                \
  do {                                                                                       \
    cudaError_t e_ = (x);                                                                    \
    if (e_ != cudaSuccess) {                                                                 \
      fprintf(stderr, "%s:%d %s -> %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_)); \
      exit(1);                                                                               \
    }                                                                                        \
  } while (0)

constexpr int kDim = 116;
constexpr int kEntries = kDim * kDim;
constexpr uint32_t kTableBytes = kEntries * 8;
constexpr uint32_t kRowBytes = kDim * 8;
constexpr int kU = 32;                                   // steps per action tile, as kPairU
constexpr uint32_t kSmem = 160 * 1024;                   // one CTA per SM
constexpr float kClipHi = 98.9999f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float2 lds_f2(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint32_t halo_addr(uint32_t addr_bias, float x, float y) {
  const uint32_t bx = __float_as_uint(__fadd_rz(x, 8388616.0f));
  const uint32_t by = __float_as_uint(__fadd_rz(y, 8388616.0f));
  return bx * kRowBytes + (by * 8u + addr_bias);
}

// table: kEntries float2 (lds: .x = index of the next entry; step: the map's (c, s)); acts: [kU][32] float2 per CTA slot;
// start: per env, the start entry (lds) or state (step).  cycles[blockIdx][warp] = clock64 cycles of `links` links.
template <bool kStep>
__global__ void __launch_bounds__(256, 1)
chain_kernel(const float2* __restrict__ table, const float2* __restrict__ acts, const float2* __restrict__ start, int lanes, int links,
             long long* __restrict__ cycles, float* __restrict__ sink) {
  extern __shared__ __align__(128) unsigned char smem[];
  float2* s_table = reinterpret_cast<float2*>(smem);
  float2* s_act = reinterpret_cast<float2*>(smem + kTableBytes);                   // [kU][32]
  float* s_out = reinterpret_cast<float*>(smem + kTableBytes + kU * 32 * 8);        // [kU*2][32]
  const uint32_t base = smem_u32(s_table);
  for (int i = threadIdx.x; i < kEntries; i += blockDim.x) {
    float2 v = table[i];
    if (!kStep) v.x = __uint_as_float(base + __float_as_uint(v.x) * 8u);
    s_table[i] = v;
  }
  for (int i = threadIdx.x; i < kU * 32; i += blockDim.x) s_act[i] = acts[i];
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane >= lanes) return;
  const int col = warp * lanes + lane;
  const float2 s0 = start[blockIdx.x * 32 + col];
  float sx = s0.x, sy = s0.y;
  long long t0, t1;
  if (!kStep) {
    uint32_t addr = base + __float_as_uint(sx) * 8u;
    float acc = 0.0f;   // keeps the load 8 bytes wide; off the chain
    t0 = clock64();
    for (int k = 0; k < links; k += 8) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float2 v = lds_f2(addr);
        addr = __float_as_uint(v.x);
        acc += v.y;
      }
    }
    t1 = clock64();
    sx = __uint_as_float(addr) + acc;
  } else {
    const uint32_t addr_bias = base - 0x4B000000u * (kRowBytes + 8u);
    const uint32_t tp = smem_u32(s_act + col), tout = smem_u32(s_out + col);
    auto store_state = [&](int u) {
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(tout + (2 * u) * 128u), "f"(sx) : "memory");
      asm volatile("st.shared.f32 [%0], %1;" ::"r"(tout + (2 * u + 1) * 128u), "f"(sy) : "memory");
    };
    t0 = clock64();
    for (int c = 0; c < links / kU; ++c) {
      float2 a = lds_f2(tp);
      uint32_t addr = halo_addr(addr_bias, sx, sy);
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const float2 cs = lds_f2(addr);
        if (u > 0) store_state(u - 1);
        const float2 an = u + 1 < kU ? lds_f2(tp + (u + 1) * 256u) : a;
        const float nx = fmaf(a.x, cs.x, fmaf(-a.y, cs.y, sx));
        const float ny = fmaf(a.x, cs.y, fmaf(a.y, cs.x, sy));
        sx = fminf(fmaxf(nx, 0.0f), kClipHi);
        sy = fminf(fmaxf(ny, 0.0f), kClipHi);
        addr = u == 0 ? halo_addr(addr_bias, sx, sy) : halo_addr(addr_bias, nx, ny);
        a = an;
      }
      store_state(kU - 1);
    }
    t1 = clock64();
  }
  if (lane == 0) cycles[blockIdx.x * 8 + warp] = t1 - t0;
  sink[blockIdx.x * 32 + col] = sx + sy;
}

int main(int argc, char** argv) {
  const int links = argc > 1 ? atoi(argv[1]) : 32768;
  int dev = 0, sms = 0;
  CK(cudaSetDevice(dev));
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  std::mt19937 rng(12345);
  std::uniform_real_distribution<float> u01(0.0f, 1.0f);

  // lds: one random cycle through all entries (Sattolo), so no lane falls into a short loop
  std::vector<int> perm(kEntries);
  for (int i = 0; i < kEntries; ++i) perm[i] = i;
  for (int i = kEntries - 1; i > 0; --i) std::swap(perm[i], perm[std::uniform_int_distribution<int>(0, i - 1)(rng)]);
  std::vector<float2> t_lds(kEntries), t_nc(kEntries), t_step(kEntries), start_lds(sms * 32), start_nc(sms * 32), start_step(sms * 32),
      acts(kU * 32);
  auto as_float = [](uint32_t u) {
    float f;
    memcpy(&f, &u, 4);
    return f;
  };
  // lds_nc: one random cycle through the entries of each bank pair
  for (int r = 0; r < 16; ++r) {
    std::vector<int> cls;
    for (int e = r; e < kEntries; e += 16) cls.push_back(e);
    const int m = (int)cls.size();
    std::vector<int> p(m);
    for (int i = 0; i < m; ++i) p[i] = i;
    for (int i = m - 1; i > 0; --i) std::swap(p[i], p[std::uniform_int_distribution<int>(0, i - 1)(rng)]);
    for (int i = 0; i < m; ++i) t_nc[cls[i]] = make_float2(as_float((uint32_t)cls[p[i]]), 0.0f);
  }
  for (int i = 0; i < kEntries; ++i) {
    t_lds[i] = make_float2(as_float((uint32_t)perm[i]), 0.0f);
    // 5 * (|c| + |s|) <= 7.9 < 8: every step stays inside the halo
    t_step[i] = make_float2(0.79f * (2.0f * u01(rng) - 1.0f), 0.79f * (2.0f * u01(rng) - 1.0f));
  }
  for (int i = 0; i < sms * 32; ++i) {
    start_lds[i] = make_float2(as_float((uint32_t)std::uniform_int_distribution<int>(0, kEntries - 1)(rng)), 0.0f);
    start_nc[i] = make_float2(as_float((uint32_t)(16 * std::uniform_int_distribution<int>(0, kEntries / 16 - 1)(rng) + i % 16)), 0.0f);
    start_step[i] = make_float2(98.9999f * u01(rng), 98.9999f * u01(rng));
  }
  for (int i = 0; i < kU * 32; ++i) acts[i] = make_float2(10.0f * u01(rng) - 5.0f, 10.0f * u01(rng) - 5.0f);

  float2 *d_tl, *d_tn, *d_ts, *d_sl, *d_sn, *d_ss, *d_a;
  long long* d_cyc;
  float* d_sink;
  CK(cudaMalloc(&d_tl, kTableBytes));
  CK(cudaMalloc(&d_tn, kTableBytes));
  CK(cudaMalloc(&d_ts, kTableBytes));
  CK(cudaMalloc(&d_sn, sms * 32 * 8));
  CK(cudaMalloc(&d_sl, sms * 32 * 8));
  CK(cudaMalloc(&d_ss, sms * 32 * 8));
  CK(cudaMalloc(&d_a, kU * 32 * 8));
  CK(cudaMalloc(&d_cyc, sms * 8 * sizeof(long long)));
  CK(cudaMalloc(&d_sink, sms * 32 * 4));
  CK(cudaMemcpy(d_tl, t_lds.data(), kTableBytes, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_tn, t_nc.data(), kTableBytes, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_ts, t_step.data(), kTableBytes, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_sn, start_nc.data(), sms * 32 * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_sl, start_lds.data(), sms * 32 * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_ss, start_step.data(), sms * 32 * 8, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(d_a, acts.data(), kU * 32 * 8, cudaMemcpyHostToDevice));
  CK(cudaFuncSetAttribute(chain_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
  CK(cudaFuncSetAttribute(chain_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));

  struct Cfg { int lanes, warps; };
  const Cfg cfgs[] = {{32, 1}, {16, 1}, {8, 1}, {4, 1}, {16, 2}, {8, 4}, {4, 8}};
  printf("{\"tool\": \"lds_chain\", \"card\": \"%s\", \"sms\": %d, \"links\": %d, \"results\": [", prop.name, sms, links);
  bool first = true;
  const char* names[] = {"lds", "lds_nc", "step"};
  for (int mode = 0; mode < 3; ++mode)
    for (const Cfg& c : cfgs) {
      std::vector<long long> cyc(sms * 8);
      auto run = [&] {
        if (mode == 0) chain_kernel<false><<<sms, c.warps * 32, kSmem>>>(d_tl, d_a, d_sl, c.lanes, links, d_cyc, d_sink);
        else if (mode == 1) chain_kernel<false><<<sms, c.warps * 32, kSmem>>>(d_tn, d_a, d_sn, c.lanes, links, d_cyc, d_sink);
        else chain_kernel<true><<<sms, c.warps * 32, kSmem>>>(d_ts, d_a, d_ss, c.lanes, links, d_cyc, d_sink);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
      };
      run();   // warm-up
      run();
      CK(cudaMemcpy(cyc.data(), d_cyc, sms * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
      std::vector<double> per;
      for (int b = 0; b < sms; ++b)
        for (int w = 0; w < c.warps; ++w) per.push_back((double)cyc[b * 8 + w] / links);
      std::sort(per.begin(), per.end());
      printf("%s{\"chain\": \"%s\", \"lanes\": %d, \"warps\": %d, \"cycles_per_link_median\": %.2f, \"min\": %.2f, \"max\": %.2f}",
             first ? "" : ", ", names[mode], c.lanes, c.warps, per[per.size() / 2], per.front(), per.back());
      first = false;
    }
  printf("]}\n");
  return 0;
}
