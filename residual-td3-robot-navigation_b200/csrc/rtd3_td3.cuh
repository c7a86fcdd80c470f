// Types shared by the fp32 learner kernels (rtd3_td3.cu) and the tensor-core learner (rtd3_tc_learner.cu).
#pragma once
#include "rtd3_common.cuh"
#include "rtd3_mlp.cuh"
#include "rtd3_tc.cuh"

namespace rtd3 {

struct ReplayView {
  const float2* s;
  const float2* a;
  const float* r;
  const float2* s2;
  const float* notdone;
};

struct Td3Hyper {
  float gamma, policy_noise, noise_clip, max_action;
  // target-policy smoothing noise (robot.py:338) when no noise tensor is supplied: unit normals from Philox4x32-10 keyed
  // (noise_seed, noise_counter[0] + noise_index, batch row).  The counter lives in device memory (a replayed CUDA graph draws fresh
  // noise); noise_index is the epoch inside one update; rtd3_td3_update advances the counter by `epochs` when it is done.
  unsigned long long noise_seed;
  const unsigned long long* noise_counter;   // nullable: counts as 0
  unsigned long long noise_index;
};

// robot.py:338: the two unit normals of batch row `row` - from the supplied tensor, else generated here
__device__ __forceinline__ float2 target_noise(const float* __restrict__ noise, const Td3Hyper& hp, int row) {
  if (noise) return make_float2(noise[row * 2], noise[row * 2 + 1]);
  double z0, z1;
  philox_normal2(hp.noise_seed, (hp.noise_counter ? hp.noise_counter[0] : 0ull) + hp.noise_index, (uint64_t)row, z0, z1);
  return make_float2((float)z0, (float)z1);
}

// Parameter arena: [actor | critic1 | critic2 | target actor | target critic1 | target critic2], each slot padded to 4 floats.
struct Arena {
  NetShape actor, critic;
  __host__ __device__ int64_t sa() const { return net_stride(actor); }
  __host__ __device__ int64_t sc() const { return net_stride(critic); }
  __host__ __device__ int64_t off(int net) const {   // 0 actor, 1 critic1, 2 critic2, 3..5 targets
    const int64_t a = sa(), c = sc();
    switch (net) {
      case 0: return 0;
      case 1: return a;
      case 2: return a + c;
      case 3: return a + 2 * c;
      case 4: return 2 * a + 2 * c;
      default: return 2 * a + 3 * c;
    }
  }
  __host__ __device__ int64_t online_total() const { return sa() + 2 * sc(); }
  __host__ __device__ int64_t total() const { return 2 * online_total(); }
};

// Tensor-core operand copies of the arena (params_uv = [u | v], each `total()` floats).  Hidden-to-hidden weights W_l [H][H]
// (l = 1..L-1) are stored chunk-major at the offset of W_l and rounded to TF32 (round-to-nearest):
//   u (forward, B operand K-major):            Wu[(k/4)*H + n][k%4] = W[n][k]
//   v (input gradient, B operand K-major of W^T): Wv[(n/4)*H + k][n%4] = W[n][k]
// every other parameter keeps its place and value.
__host__ __device__ inline bool is_hidden_weight(const NetShape& s, int64_t net_off, int64_t i) {
  const int64_t o = i - net_off;
  const int64_t first = (int64_t)s.in * s.hid + s.hid, blk = (int64_t)s.hid * s.hid + s.hid;
  if (o < first) return false;
  const int64_t o2 = o - first;
  const int64_t l = o2 / blk, rem = o2 - l * blk;
  return l < s.layers - 1 && rem < (int64_t)s.hid * s.hid;
}
__host__ __device__ inline int64_t chunk_major_index(const NetShape& s, int64_t net_off, int64_t i) {
  if (!is_hidden_weight(s, net_off, i)) return i;
  const int64_t first = (int64_t)s.in * s.hid + s.hid, blk = (int64_t)s.hid * s.hid + s.hid;
  const int64_t o2 = i - net_off - first;
  const int64_t l = o2 / blk, rem = o2 - l * blk;
  const int64_t n = rem / s.hid, k = rem - n * s.hid;
  return net_off + first + l * blk + ((k >> 2) * s.hid + n) * 4 + (k & 3);
}
__host__ __device__ inline int64_t chunk_major_index_v(const NetShape& s, int64_t net_off, int64_t i) {
  if (!is_hidden_weight(s, net_off, i)) return i;
  const int64_t first = (int64_t)s.in * s.hid + s.hid, blk = (int64_t)s.hid * s.hid + s.hid;
  const int64_t o2 = i - net_off - first;
  const int64_t l = o2 / blk, rem = o2 - l * blk;
  const int64_t n = rem / s.hid, k = rem - n * s.hid;
  return net_off + first + l * blk + ((n >> 2) * s.hid + k) * 4 + (n & 3);
}

// One element of torch.optim.Adam (defaults, robot.py:237-239) in the operation order of torch's CPU kernels, measured against
// torch.optim.Adam in the build container (oracle/td3_oracle.py: adam_step, pinned bit for bit by tests/test_oracle_td3.py):
//   exp_avg.lerp_(grad, 1 - beta1)                       m = fma(g - m, 0.1f, m)
//   exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)     v = fma(0.001f * g, g, v * 0.999f)         (both products rounded)
//   denom = sqrt(v) / sqrt(bc2) + eps;  param.addcdiv_(exp_avg, denom, -step)      p = p + (-step * m) / denom
// Every rounding is spelled out so that the three kernels that apply it (td3_adam_polyak_kernel, the optimiser fused into
// wgrad_kernel, the cooperative kernel) agree bit for bit - left to the compiler, the contraction of a*b + c*d differs between them.
__device__ __forceinline__ void adam_element(float g, float& m, float& v, float& p, float step, float sqrt_bc2) {
  m = __fmaf_rn(__fsub_rn(g, m), 0.1f, m);
  v = __fmaf_rn(__fmul_rn(0.001f, g), g, __fmul_rn(v, 0.999f));
  const float denom = __fadd_rn(__fdiv_rn(sqrtf(v), sqrt_bc2), 1e-8f);
  p = __fadd_rn(p, __fdiv_rn(__fmul_rn(-step, m), denom));
}

// Where arena element o (offset inside its network's slot) sits in the derived copies, decomposed ONCE per element in 32-bit
// arithmetic: the 64-bit divisions of transposed_index / chunk_major_index (five calls per element) made this kernel ~13 us.
struct CopyIndex {
  int t, u, v;          // offsets inside the slot in the transposed / forward chunk-major / input-gradient chunk-major copies
  bool hidden;          // a hidden-to-hidden weight (the only entries that move, and that are TF32-rounded in u / v)
};
__device__ __forceinline__ CopyIndex copy_index(const NetShape& s, int o) {
  CopyIndex c{o, o, o, false};
  const int first = s.in * s.hid + s.hid, blk = s.hid * s.hid + s.hid;
  if (o < first) return c;
  const unsigned o2 = (unsigned)(o - first);
  const unsigned l = o2 / (unsigned)blk, rem = o2 - l * (unsigned)blk;
  if ((int)l >= s.layers - 1 || rem >= (unsigned)(s.hid * s.hid)) return c;
  const unsigned n = rem / (unsigned)s.hid, k = rem - n * (unsigned)s.hid;
  const int base = first + (int)l * blk;
  c.hidden = true;
  c.t = base + (int)(k * s.hid + n);
  c.u = base + (int)((((k >> 2) * s.hid + n) << 2) + (k & 3u));
  c.v = base + (int)((((n >> 2) * s.hid + k) << 2) + (n & 3u));
  return c;
}


// Four consecutive arena elements i .. i+3 of the optimiser pass (i a multiple of 4: network slots, weight matrices and bias vectors all
// start at multiples of 4, so the four are either four neighbours of one row of a hidden weight matrix or four elements that keep
// their place in the derived copies): Adam (when do_adam, with the already scaled gradients g) on the parameters of online network
// `net`, then (when do_polyak) the blend of the matching target parameters, t = t*(1-tau) + p*tau; the transposed copy and the
// tensor-core operand copies (params_uv, nullable) are kept in step.  One round of 16-byte loads per group.  Shared by
// td3_adam_polyak_kernel and the peer-memory all-reduce that applies the optimiser to the sums it forms (rtd3_p2p.cu).
__device__ __forceinline__ void adam_polyak_apply4(const Arena& ar, int i, int net, const float (&g)[4], bool do_adam, bool do_polyak,
                                                   float* __restrict__ params, float* __restrict__ params_t, float* __restrict__ params_uv,
                                                   float* __restrict__ m, float* __restrict__ v, float step, float sqrt_bc2, float tau) {
  const int n_online = (int)ar.online_total(), total = (int)ar.total();
  const int noff = net == 0 ? 0 : (int)ar.off(net);
  const CopyIndex ci = copy_index(net == 0 ? ar.actor : ar.critic, i - noff);      // of element i; hidden: .t stride H, .u contiguous, .v stride 4
  const int H = (net == 0 ? ar.actor : ar.critic).hid;
  const int st = ci.hidden ? H : 1, sv = ci.hidden ? 4 : 1;
  float4 p4 = *reinterpret_cast<const float4*>(params + i);
  float p[4] = {p4.x, p4.y, p4.z, p4.w};
  float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f);
  if (do_polyak) t4 = *reinterpret_cast<const float4*>(params + n_online + i);
  if (do_adam) {
    const float4 m4 = *reinterpret_cast<const float4*>(m + i), v4 = *reinterpret_cast<const float4*>(v + i);
    float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) adam_element(g[e], mm[e], vv[e], p[e], step, sqrt_bc2);
    *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    *reinterpret_cast<float4*>(params + i) = make_float4(p[0], p[1], p[2], p[3]);
#pragma unroll
    for (int e = 0; e < 4; ++e) params_t[noff + ci.t + e * st] = p[e];
    if (params_uv) {
      float pr[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) pr[e] = ci.hidden ? tf32_rn(p[e]) : p[e];
      *reinterpret_cast<float4*>(params_uv + noff + ci.u) = make_float4(pr[0], pr[1], pr[2], pr[3]);
#pragma unroll
      for (int e = 0; e < 4; ++e) params_uv[total + noff + ci.v + e * sv] = pr[e];
    }
  }
  if (do_polyak) {
    const float to[4] = {t4.x, t4.y, t4.z, t4.w};
    float tv[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) tv[e] = __fadd_rn(__fmul_rn(to[e], 1.0f - tau), __fmul_rn(p[e], tau));   // robot.py:309, three roundings
    *reinterpret_cast<float4*>(params + n_online + i) = make_float4(tv[0], tv[1], tv[2], tv[3]);
#pragma unroll
    for (int e = 0; e < 4; ++e) params_t[n_online + noff + ci.t + e * st] = tv[e];
    if (params_uv)
      *reinterpret_cast<float4*>(params_uv + n_online + noff + ci.u) =
          make_float4(ci.hidden ? tf32_rn(tv[0]) : tv[0], ci.hidden ? tf32_rn(tv[1]) : tv[1], ci.hidden ? tf32_rn(tv[2]) : tv[2],
                      ci.hidden ? tf32_rn(tv[3]) : tv[3]);
  }
}

// Adam bookkeeping advanced by the first thread of a step kernel: the step counter and the running powers
// beta1^t, beta2^t (float64, as torch computes the bias corrections in Python floats).  o: 0 actor, 1 critics.
__device__ __forceinline__ void advance_adam_clock(int32_t* steps, double* beta_pows, int o) {
  steps[o] += 1;
  beta_pows[2 * o] *= 0.9;
  beta_pows[2 * o + 1] *= 0.999;
}

}  // namespace rtd3

// launch helpers shared by the public step entry points and rtd3_td3_update (rtd3_td3.cu, rtd3_tc_learner.cu)
struct rtd3_td3;
namespace rtd3 {
int32_t critic_step_launch(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const ReplayView& rp,
                           const int32_t* idx, const float* noise, int32_t batch, const Td3Hyper& hp, float* loss2, float* q_out, float* y_out,
                           int32_t* steps, double* beta_pows, cudaStream_t st);
int32_t advance_noise_counter(uint64_t* counter, uint64_t by, cudaStream_t st);   // counter[0] += by on the stream
int32_t critic_step_tc_launch(rtd3_td3* h, const float* params, const float* params_uv, float* grads, const ReplayView& rp, const int32_t* idx,
                              const float* noise, int32_t batch, const Td3Hyper& hp, float* loss2, float* q_out, float* y_out, int32_t* steps,
                              double* beta_pows, cudaStream_t st);
// small batches on thread-block clusters (rtd3_cluster.cu)
bool cluster_path_ok(const rtd3_td3* h, int batch);
int32_t critic_cluster_launch(rtd3_td3* h, const float* params, const float* params_t, float* scratch, const ReplayView& rp, const int32_t* idx,
                              const float* noise, int32_t batch, const Td3Hyper& hp, float* loss2, float* q_out, float* y_out, int32_t* steps,
                              double* beta_pows, cudaStream_t st);
int32_t actor_cluster_launch(rtd3_td3* h, const float* params, const float* params_t, float* scratch, const ReplayView& rp, const int32_t* idx,
                             int32_t batch, float* loss1, int32_t* steps, double* beta_pows, cudaStream_t st);

// The gradient all-reduce over peer memory with the optimiser applied to the sums (rtd3_p2p.cu): what update_allreduce +
// rtd3_td3_adam_polyak do in two launches and two passes over the arena.  [off, off + count) = the slice of the gradient arena this
// optimiser step reduces; nets / polyak as in rtd3_td3_adam_polyak.
struct P2pAdamArgs {
  Arena ar;
  float* params; float* params_t; float* params_uv; float* m; float* v;
  const double* beta_pows;
  double lr_actor, lr_critic;
  float grad_scale, tau;
  int nets, polyak;
  int64_t off;
};
int32_t p2p_allreduce_adam_launch(const rtd3_p2p_state* p, float* local_grads, int64_t count, const P2pAdamArgs& opt, cudaStream_t st);
}  // namespace rtd3

// the opaque learner handle of the C ABI
constexpr int kNumTiles = 4;
static constexpr int kRowTiles[kNumTiles] = {2, 4, 8, 16};

struct rtd3_td3 {
  rtd3::Arena ar;
  int device;
  int num_sms;
  size_t smem_critic[kNumTiles], smem_actor[kNumTiles], smem_fwd[kNumTiles];
  int cluster_cap;      // clusters of the cluster step kernels the device holds at once (set by rtd3_td3_create; 0: path unavailable)
};

