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

// The optimiser's state: the parameter arena with its derived copies, torch.optim.Adam's moments and clocks (robot.py:237-239) and the
// Polyak rate.  One per update call; every kernel that applies the optimiser takes it.
struct AdamState {
  Arena ar;
  float* params;            // the arena (online | target)
  float* params_t;          // transposed copy
  float* params_uv;         // nullable: the tensor-core operand copies [u | v] are not kept
  float* m;
  float* v;
  double* beta_pows;        // [2][2]: beta1^t, beta2^t of optimiser 0 (actor) and 1 (critics)
  double lr[2];             // 0 actor, 1 critics
  float tau;
};

// torch.optim.Adam's step size lr / (1 - beta1^t) and sqrt(1 - beta2^t), formed in double from the double lr and the running powers
// (as torch forms them in Python floats) and rounded to float once each.
struct AdamStep {
  float step, sqrt_bc2;
};
__device__ __forceinline__ AdamStep adam_step(double lr, double beta1_pow, double beta2_pow) {
  return AdamStep{(float)(lr / (1.0 - beta1_pow)), (float)sqrt(1.0 - beta2_pow)};
}

// One element of torch.optim.Adam (defaults, robot.py:237-239) in the operation order of torch's CPU kernels, measured against
// torch.optim.Adam in the build container (oracle/td3_oracle.py: adam_step, pinned bit for bit by tests/test_oracle_td3.py):
//   exp_avg.lerp_(grad, 1 - beta1)                       m = fma(g - m, 0.1f, m)
//   exp_avg_sq.mul_(beta2).addcmul_(g, g, 1 - beta2)     v = fma(0.001f * g, g, v * 0.999f)         (both products rounded)
//   denom = sqrt(v) / sqrt(bc2) + eps;  param.addcdiv_(exp_avg, denom, -step)      p = p + (-step * m) / denom
// Every rounding is spelled out: its callers, adam_polyak4 and adam_polyak1, are inlined into kernels of different shapes, and left to
// the compiler, the contraction of a*b + c*d would differ between them.
__device__ __forceinline__ void adam_element(float g, float& m, float& v, float& p, float step, float sqrt_bc2) {
  m = __fmaf_rn(__fsub_rn(g, m), 0.1f, m);
  v = __fmaf_rn(__fmul_rn(0.001f, g), g, __fmul_rn(v, 0.999f));
  const float denom = __fadd_rn(__fdiv_rn(sqrtf(v), sqrt_bc2), 1e-8f);
  p = __fadd_rn(p, __fdiv_rn(__fmul_rn(-step, m), denom));
}
// robot.py:309, three roundings
__device__ __forceinline__ float polyak_blend(float t, float p, float tau) { return __fadd_rn(__fmul_rn(t, 1.0f - tau), __fmul_rn(p, tau)); }

// Arena element o (offset inside its network's slot) as a hidden-to-hidden weight W_{l+1}[n][k] (l = 0..L-2), or not one.  32-bit
// arithmetic: a slot of H <= kMaxHidden, L <= kMaxLayers holds well under 2^31 elements (the 64-bit divisions of an earlier per-copy
// index function made the optimiser kernel ~13 us).
struct SlotPos {
  bool hidden;
  unsigned l, n, k;
};
__device__ __forceinline__ SlotPos slot_pos(const NetShape& s, int o) {
  const int first = s.in * s.hid + s.hid, blk = s.hid * s.hid + s.hid;
  if (o < first) return SlotPos{false, 0u, 0u, 0u};
  const unsigned o2 = (unsigned)(o - first);
  const unsigned l = o2 / (unsigned)blk, rem = o2 - l * (unsigned)blk;
  if ((int)l >= s.layers - 1 || rem >= (unsigned)(s.hid * s.hid)) return SlotPos{false, 0u, 0u, 0u};
  const unsigned n = rem / (unsigned)s.hid;
  return SlotPos{true, l, n, rem - n * (unsigned)s.hid};
}

// Where a parameter sits in the derived copies of the arena (offsets inside its network's slot).  Hidden-to-hidden weights W [H][H]
// move; every other parameter keeps its place and value in all three:
//   t  (transposed, forward operand of the fp32 kernels):          Wt[k][n] = W[n][k]
//   u  (tensor cores, forward B operand K-major, TF32-rounded):     Wu[(k/4)*H + n][k%4] = W[n][k]
//   v  (tensor cores, input-gradient B operand K-major of W^T):     Wv[(n/4)*H + k][n%4] = W[n][k]
// params_uv = [u | v], each ar.total() floats.
struct CopyIndex {
  int t, u, v;
  bool hidden;          // a hidden-to-hidden weight (the only entries that move, and that are TF32-rounded in u / v)
};
__device__ __forceinline__ CopyIndex copy_index(const NetShape& s, unsigned l, unsigned n, unsigned k) {   // of W_{l+1}[n][k]
  const int base = s.in * s.hid + s.hid + (int)l * (s.hid * s.hid + s.hid);
  return CopyIndex{base + (int)(k * s.hid + n), base + (int)((((k >> 2) * s.hid + n) << 2) + (k & 3u)),
                   base + (int)((((n >> 2) * s.hid + k) << 2) + (n & 3u)), true};
}
__device__ __forceinline__ CopyIndex copy_index(const NetShape& s, int o) {
  const SlotPos q = slot_pos(s, o);
  return q.hidden ? copy_index(s, q.l, q.n, q.k) : CopyIndex{o, o, o, false};
}

// The optimiser on four consecutive arena elements i .. i+3 of an online network (slot offset noff, ci = copy_index of element i,
// H its hidden width; n_online, total = s.ar.online_total(), s.ar.total()) from operands the caller has loaded: Adam (when do_adam)
// with the already scaled gradients g on the moments m4, v4 and the parameters p4, then (when do_polyak) the blend of the target
// parameters t4, t = t*(1-tau) + p*tau; the results are stored into the arena, the moments and every derived copy.  i is a multiple of 4 (network slots, weight matrices and bias vectors
// all start at multiples of 4), so the four are either four neighbours of one row of a hidden weight matrix (in t a column, stride H;
// in v stride 4) or four elements that keep their place.
__device__ __forceinline__ void adam_polyak4(const AdamState& s, int i, int noff, const CopyIndex& ci, int H, const float (&g)[4], float4 m4,
                                             float4 v4, float4 p4, float4 t4, AdamStep k, bool do_adam, bool do_polyak, int n_online, int total) {
  const int st = ci.hidden ? H : 1, sv = ci.hidden ? 4 : 1;
  float p[4] = {p4.x, p4.y, p4.z, p4.w};
  if (do_adam) {
    float mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) adam_element(g[e], mm[e], vv[e], p[e], k.step, k.sqrt_bc2);
    *reinterpret_cast<float4*>(s.m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(s.v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    *reinterpret_cast<float4*>(s.params + i) = make_float4(p[0], p[1], p[2], p[3]);
#pragma unroll
    for (int e = 0; e < 4; ++e) s.params_t[noff + ci.t + e * st] = p[e];
    if (s.params_uv) {
      float pr[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) pr[e] = ci.hidden ? tf32_rn(p[e]) : p[e];
      *reinterpret_cast<float4*>(s.params_uv + noff + ci.u) = make_float4(pr[0], pr[1], pr[2], pr[3]);
#pragma unroll
      for (int e = 0; e < 4; ++e) s.params_uv[total + noff + ci.v + e * sv] = pr[e];
    }
  }
  if (do_polyak) {
    const float to[4] = {t4.x, t4.y, t4.z, t4.w};
    float tv[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) tv[e] = polyak_blend(to[e], p[e], s.tau);
    *reinterpret_cast<float4*>(s.params + n_online + i) = make_float4(tv[0], tv[1], tv[2], tv[3]);
#pragma unroll
    for (int e = 0; e < 4; ++e) s.params_t[n_online + noff + ci.t + e * st] = tv[e];
    if (s.params_uv)   // the target networks run forward only: their v copy is not kept
      *reinterpret_cast<float4*>(s.params_uv + n_online + noff + ci.u) =
          make_float4(ci.hidden ? tf32_rn(tv[0]) : tv[0], ci.hidden ? tf32_rn(tv[1]) : tv[1], ci.hidden ? tf32_rn(tv[2]) : tv[2],
                      ci.hidden ? tf32_rn(tv[3]) : tv[3]);
  }
}
// The same on one element i.
__device__ __forceinline__ void adam_polyak1(const AdamState& s, int i, int noff, const CopyIndex& ci, float g, float m, float v, float p,
                                             float t, AdamStep k, bool do_adam, bool do_polyak, int n_online, int total) {
  if (do_adam) {
    adam_element(g, m, v, p, k.step, k.sqrt_bc2);
    s.m[i] = m;
    s.v[i] = v;
    s.params[i] = p;
    s.params_t[noff + ci.t] = p;
    if (s.params_uv) {
      const float pr = ci.hidden ? tf32_rn(p) : p;
      s.params_uv[noff + ci.u] = pr;
      s.params_uv[total + noff + ci.v] = pr;
    }
  }
  if (do_polyak) {
    const float tv = polyak_blend(t, p, s.tau);
    s.params[n_online + i] = tv;
    s.params_t[n_online + noff + ci.t] = tv;
    if (s.params_uv) s.params_uv[n_online + noff + ci.u] = ci.hidden ? tf32_rn(tv) : tv;
  }
}

// Load-then-apply form of adam_polyak4 for the kernels that walk the online arena in groups of 4 (td3_adam_polyak_kernel, and the
// peer-memory all-reduce that applies the optimiser to the sums it forms, rtd3_p2p.cu): one round of 16-byte loads per group.
__device__ __forceinline__ void adam_polyak_apply4(const AdamState& s, int i, int net, const float (&g)[4], AdamStep k, bool do_adam, bool do_polyak) {
  const int noff = net == 0 ? 0 : (int)s.ar.off(net);
  const NetShape& sh = net == 0 ? s.ar.actor : s.ar.critic;
  const CopyIndex ci = copy_index(sh, i - noff);
  const float4 p4 = *reinterpret_cast<const float4*>(s.params + i);
  float4 t4 = make_float4(0.f, 0.f, 0.f, 0.f), m4 = t4, v4 = t4;
  if (do_polyak) t4 = *reinterpret_cast<const float4*>(s.params + (int)s.ar.online_total() + i);
  if (do_adam) {
    m4 = *reinterpret_cast<const float4*>(s.m + i);
    v4 = *reinterpret_cast<const float4*>(s.v + i);
  }
  adam_polyak4(s, i, noff, ci, sh.hid, g, m4, v4, p4, t4, k, do_adam, do_polyak, (int)s.ar.online_total(), (int)s.ar.total());
}

// Adam bookkeeping advanced by the first thread of a step kernel: the step counter and the running powers
// beta1^t, beta2^t (float64, as torch computes the bias corrections in Python floats).  o: 0 actor, 1 critics.
__device__ __forceinline__ void advance_adam_clock(int32_t* steps, double* beta_pows, int o) {
  steps[o] += 1;
  beta_pows[2 * o] *= 0.9;
  beta_pows[2 * o + 1] *= 0.999;
}

}  // namespace rtd3

// launch helpers shared by the learner sources
struct rtd3_td3;
namespace rtd3 {
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
  AdamState adam;
  float grad_scale;
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

// the optimiser state of an update call (rtd3_td3_update, rtd3_td3_update_coop)
inline rtd3::AdamState adam_state(const rtd3_td3* h, const rtd3_td3_update_args* a) {
  return rtd3::AdamState{h->ar, a->params, a->params_t, a->params_uv, a->adam_m, a->adam_v, a->beta_pows, {a->lr_actor, a->lr_critic}, a->tau};
}

