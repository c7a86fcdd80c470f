// Shared host/device helpers for librtd3 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/rtd3.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "librtd3 targets sm_100a (B200) only"
#endif

namespace rtd3 {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
// Per-device caches (rtd3_runtime.cu): function attributes and SM counts belong to a device, so they are keyed by the CURRENT
// device and guarded by a mutex (a process may drive several GPUs from several host threads).
cudaError_t ensure_dyn_smem(const void* kernel, size_t bytes);   // cudaFuncAttributeMaxDynamicSharedMemorySize >= bytes on this device
cudaError_t current_num_sms(int* out);                           // multiprocessor count of the current device

#define RTD3_CHECK_ARG(cond, msg)                                   \
  do {                                                              \
    if (!(cond)) {                                                  \
      ::rtd3::set_error("%s: %s", __func__, msg);                   \
      return RTD3_ERR_ARG;                                          \
    }                                                               \
  } while (0)

#define RTD3_CUDA(expr)                                                                   \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      ::rtd3::set_error("%s: %s -> %s", __func__, #expr, cudaGetErrorString(_e));         \
      return (int32_t)_e;                                                                 \
    }                                                                                     \
  } while (0)

// Every launch goes through this so gpu_launches in bench.py is a count, not a guess.
#define RTD3_LAUNCHED()                     \
  do {                                      \
    ::rtd3::count_launch();                 \
    RTD3_CUDA(cudaGetLastError());          \
  } while (0)

// Makes a device current until the end of the scope and then restores the caller's, on every return path.
class DeviceGuard {
 public:
  DeviceGuard() = default;
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
  ~DeviceGuard() {
    if (prev_ >= 0) cudaSetDevice(prev_);
  }
  cudaError_t enter(int device) {
    int cur = 0;
    if (cudaError_t e = cudaGetDevice(&cur)) return e;
    if (cur == device) return cudaSuccess;
    if (cudaError_t e = cudaSetDevice(device)) return e;
    prev_ = cur;
    return cudaSuccess;
  }

 private:
  int prev_ = -1;   // the device to restore, -1 when the guard did not switch
};

constexpr float kMaxAction = 5.0f;                 // constants.py:34
constexpr float kClipHi = 98.9999f;                // float32(WORLD_SIZE - 1.0001), environment.py:117
constexpr int kWorld = RTD3_WORLD_SIZE;
constexpr int kCells = RTD3_MAP_CELLS;
constexpr int kMaxMaps = 65536;                  // maps of a bank (rtd3_env_set_maps) and of one rtd3_perlin_maps call

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// np.clip semantics: NaN passes through (fminf/fmaxf would swallow it).
__device__ __forceinline__ float clip_keep_nan(float v, float lo, float hi) {
  return v < lo ? lo : (v > hi ? hi : v);
}

// ---- mbarrier + bulk-async (TMA) copy primitives, sm_90+/sm_100a PTX ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// Whether the phase of the given parity has completed, without blocking; when it has, the test acquires like mbar_wait.
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// 1-D bulk copy shared -> global, completion tracked by the thread's bulk async-group.
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kN>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kN) : "memory"); }
template <int kN>
__device__ __forceinline__ void bulk_wait() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(kN) : "memory"); }

// Programmatic dependent launch.  launch_dependents lets the next kernel of the stream (launched with
// cudaLaunchAttributeProgrammaticStreamSerialization) start once every CTA of this grid has issued it; grid_dep_wait blocks until
// the grids this one depends on have completed and their memory is visible.  Both are no-ops in a grid launched without the
// attribute.
__device__ __forceinline__ void launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Philox4x32-10 (Salmon et al. 2011), the counter-based generator used for the non-parity index draw.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}

// Two unit normals for (env, tick) from Philox4x32-10 + Box-Muller in float64 (throughput-mode exploration noise: counter-based,
// so a replayed CUDA graph draws fresh noise every tick from the device tick counter).
__device__ __forceinline__ void philox_normal2(uint64_t seed, uint64_t tick, uint64_t env, double& z0, double& z1) {
  const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), (uint32_t)tick, (uint32_t)(tick >> 32)),
                                make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const double u1 = ((double)(r.x >> 5) * 67108864.0 + (double)(r.y >> 6)) / 9007199254740992.0;   // [0,1), 53 bits
  const double u2 = ((double)(r.z >> 5) * 67108864.0 + (double)(r.w >> 6)) / 9007199254740992.0;
  const double rad = sqrt(-2.0 * log(1.0 - u1));                                                  // 1 - u1 in (0,1]
  double s, c;
  sincospi(2.0 * u2, &s, &c);
  z0 = rad * c;
  z1 = rad * s;
}

}  // namespace rtd3
