// Residual-TD3 learner hot path: replay ring, minibatch gather, twin-critic / actor steps, Adam + Polyak.
// Reference behaviour: /root/reference/robot.py:58-124 (ReplayBuffer), :128-206 (networks), :258-398 (TD3).
#include <cstdlib>

#include "rtd3_common.cuh"
#include "rtd3_mlp.cuh"
#include "rtd3_tc.cuh"
#include "rtd3_p2p.cuh"
#include "rtd3_td3.cuh"

namespace rtd3 {

// ---- critic phase: robot.py:312-366 up to (not including) the optimiser steps ------------------------------------
//   y = r + gamma * min(Q1', Q2')(s2, clip(pi'(s2) + clip(noise*sigma, +-c), +-5)) * notdone
//   L_i = mean((Q_i(s,a) - y)^2); forward + backward of both critics; per-row layer inputs / pre-activation gradients
//   go to the row scratch (slot c = critic c), from which wgrad_kernel forms the parameter gradients.
// One CTA = R batch rows through the whole chain: five network passes driven by ONE loop so that the layer code is
// instantiated once (the fully inlined five-call version was 143 KB of SASS and stalled on instruction fetch).
template <int R>
__global__ void __launch_bounds__(kThreads, 1)
td3_critic_kernel(Arena ar, const float* __restrict__ params, const float* __restrict__ params_t, float* __restrict__ scratch, ReplayView rp, const int32_t* __restrict__ idx,
                  const float* __restrict__ noise /*[B][2] unit normal*/, int B, Td3Hyper hp, float* __restrict__ loss /*[2]*/,
                  float* __restrict__ q_out /*nullable [2][B]*/, float* __restrict__ y_out /*nullable [B]*/, int32_t* __restrict__ steps,
                  double* __restrict__ beta_pows) {
  MlpSmem<R> sm;
  sm.carve(0, ar.critic.hid, ar.critic.layers);
  const int r0 = blockIdx.x * R;
  const int t = threadIdx.x;
  if (blockIdx.x == 0 && t == 0) advance_adam_clock(steps, beta_pows, 1);

  float* S = smem_f + sm.scratch;   // [R][8]: 0 s.x 1 s.y 2 a.x 3 a.y 4 reward 5 notdone 6 y 7 valid
  float* in0 = smem_f + sm.in0;
  float* out = smem_f + sm.out;
  float* dout = smem_f + sm.dout;
  if (t < R) {
    const int row = r0 + t;
    const bool valid = row < B;
    const int j = valid ? idx[row] : 0;
    const float2 s = rp.s[j], a = rp.a[j], s2 = rp.s2[j];
    S[t * 8 + 0] = s.x; S[t * 8 + 1] = s.y; S[t * 8 + 2] = a.x; S[t * 8 + 3] = a.y;
    S[t * 8 + 4] = rp.r[j]; S[t * 8 + 5] = rp.notdone[j]; S[t * 8 + 7] = valid ? 1.f : 0.f;
    in0[t * 4 + 0] = s2.x; in0[t * 4 + 1] = s2.y; in0[t * 4 + 2] = 0.f; in0[t * 4 + 3] = 0.f;
  }
  __syncthreads();

  // pass 0: target actor(s2); 1, 2: target critics(s2, a'); 3, 4: critics(s, a) forward + backward
  for (int pass = 0; pass < 5; ++pass) {
    const int net = pass == 0 ? 3 : (pass == 1 ? 4 : (pass == 2 ? 5 : pass - 2));
    const NetShape shape = pass == 0 ? ar.actor : ar.critic;
    const bool train = pass >= 3;
    const float* P = params + ar.off(net);
    RowScratch rs{scratch + (train ? (pass - 3) : 0) * RowScratch::floats(B, ar.critic.hid, ar.critic.layers), B, ar.critic.hid,
                  ar.critic.layers};
    mlp_forward<R>(P, params_t + ar.off(net), shape, sm, train, train ? &rs : nullptr, r0);
    if (t < R) {
      if (pass == 0) {                                   // smoothing noise and clips (robot.py:338-339)
        const int row = min(r0 + t, B - 1);
        const float2 zn = target_noise(noise, hp, row);
#pragma unroll
        for (int o = 0; o < 2; ++o) {
          float e = (o == 0 ? zn.x : zn.y) * hp.policy_noise;
          e = fminf(fmaxf(e, -hp.noise_clip), hp.noise_clip);
          in0[t * 4 + 2 + o] = fminf(fmaxf(out[t * 2 + o] + e, -hp.max_action), hp.max_action);
        }
      } else if (pass == 1) {
        S[t * 8 + 6] = out[t * 2];
      } else if (pass == 2) {                            // clipped double-Q target (robot.py:342-345)
        const float qmin = fminf(S[t * 8 + 6], out[t * 2]);
        const float y = S[t * 8 + 4] + hp.gamma * qmin * S[t * 8 + 5];
        S[t * 8 + 6] = y;
        if (y_out && r0 + t < B) y_out[r0 + t] = y;
        in0[t * 4 + 0] = S[t * 8 + 0]; in0[t * 4 + 1] = S[t * 8 + 1];
        in0[t * 4 + 2] = S[t * 8 + 2]; in0[t * 4 + 3] = S[t * 8 + 3];
      } else {                                           // MSE loss and its gradient (robot.py:348-353)
        const int c = pass - 3;
        const float valid = S[t * 8 + 7];
        const float q = out[t * 2];
        const float diff = (q - S[t * 8 + 6]) * valid;
        dout[t * 2] = 2.0f * diff / (float)B;
        dout[t * 2 + 1] = 0.f;
        if (q_out && valid != 0.f) q_out[c * B + r0 + t] = q;
        float l = diff * diff / (float)B;                // this row's share of the mean
#pragma unroll
        for (int o = R / 2; o > 0; o >>= 1) l += __shfl_xor_sync((R >= 32) ? 0xffffffffu : ((1u << R) - 1u), l, o);
        if (t == 0) atomicAdd(loss + c, l);
      }
    }
    __syncthreads();
    if (train) {
      mlp_backward<R>(P, shape, sm, &rs, r0, false);
      __syncthreads();
    }
  }
}

// ---- actor phase: robot.py:369-398 up to the optimiser step ---------------------------------------------------------
//   L = -mean(Q1(s, pi(s)));  gradient w.r.t. the actor only (critic-1 parameter gradients are discarded by the reference)
template <int R>
__global__ void __launch_bounds__(kThreads, 1)
td3_actor_kernel(Arena ar, const float* __restrict__ params, const float* __restrict__ params_t, float* __restrict__ scratch, ReplayView rp, const int32_t* __restrict__ idx,
                 int B, float* __restrict__ loss /*[1]*/, int32_t* __restrict__ steps, double* __restrict__ beta_pows) {
  MlpSmem<R> sc;                      // critic pass (activations kept, backward for dQ/da)
  sc.carve(0, ar.critic.hid, ar.critic.layers);
  // the actor pass shares the weight-tile ring and small buffers; only its kept activations and its input are separate
  MlpSmem<R> sa = sc;
  sa.act0 = (int)MlpSmem<R>::floats(ar.critic.hid, ar.critic.layers);
  sa.in0 = sa.act0 + ar.actor.layers * R * sc.ld;
  const int r0 = blockIdx.x * R;
  const int t = threadIdx.x;
  if (blockIdx.x == 0 && t == 0) advance_adam_clock(steps, beta_pows, 0);
  float* S = smem_f + sc.scratch;
  float* actor_in = smem_f + sa.in0;
  RowScratch rs{scratch, B, ar.actor.hid, ar.actor.layers};

  if (t < R) {
    const int row = r0 + t;
    const bool valid = row < B;
    const float2 s = rp.s[valid ? idx[row] : 0];
    actor_in[t * 4 + 0] = s.x; actor_in[t * 4 + 1] = s.y; actor_in[t * 4 + 2] = 0.f; actor_in[t * 4 + 3] = 0.f;
    S[t * 8 + 7] = valid ? 1.f : 0.f;
  }
  __syncthreads();
  // forward: pass 0 a = pi(s) (fed the raw replay state, robot.py:386), pass 1 Q1(s, a)
  for (int pass = 0; pass < 2; ++pass) {
    const MlpSmem<R> sm = pass == 0 ? sa : sc;
    mlp_forward<R>(params + ar.off(pass), params_t + ar.off(pass), pass == 0 ? ar.actor : ar.critic, sm, true, pass == 0 ? &rs : nullptr, r0);
    if (t < R) {
      if (pass == 0) {
        float* cin = smem_f + sc.in0;
        cin[t * 4 + 0] = actor_in[t * 4 + 0]; cin[t * 4 + 1] = actor_in[t * 4 + 1];
        cin[t * 4 + 2] = smem_f[sa.out + t * 2]; cin[t * 4 + 3] = smem_f[sa.out + t * 2 + 1];
      } else {
        const float valid = S[t * 8 + 7];
        smem_f[sc.dout + t * 2] = -valid / (float)B;
        smem_f[sc.dout + t * 2 + 1] = 0.f;
        float l = -smem_f[sc.out + t * 2] * valid / (float)B;
#pragma unroll
        for (int o = R / 2; o > 0; o >>= 1) l += __shfl_xor_sync((R >= 32) ? 0xffffffffu : ((1u << R) - 1u), l, o);
        if (t == 0) atomicAdd(loss, l);
      }
    }
    __syncthreads();
  }
  // backward: pass 0 through critic 1 (only dQ/d(input) is needed), pass 1 through the actor
  for (int pass = 0; pass < 2; ++pass) {
    const MlpSmem<R> sm = pass == 0 ? sc : sa;
    mlp_backward<R>(params + ar.off(1 - pass), pass == 0 ? ar.critic : ar.actor, sm, pass == 0 ? nullptr : &rs, r0, pass == 0);
    if (pass == 0 && t < R) {
      smem_f[sa.dout + t * 2] = smem_f[sc.din + t * 4 + 2];
      smem_f[sa.dout + t * 2 + 1] = smem_f[sc.din + t * 4 + 3];
    }
    __syncthreads();
  }
}

// Optional optimiser fused into the weight-gradient pass (single GPU, batch <= 512: every gradient element is final when its job
// writes it): torch.optim.Adam on the element and, on request, the Polyak blend of the matching target parameter (adam_polyak4 /
// adam_polyak1) - the two separate optimiser launches of an epoch (13 us at B = 256) disappear.
struct AdamFuse {
  AdamState adam;           // adam.params == nullptr: not fused, gradients are stored
  int opt;                  // 0 actor optimiser, 1 critic optimisers (index into lr and beta_pows)
  int polyak;               // blend the target copy of every updated parameter
  int n_online, total;      // adam.ar.online_total() / total(): derived at every use, they made the kernel 8 % longer, B = 256 0.6 % slower
};

// Optional peer-memory exchange fused into the same pass (data parallel, world > 1, with AdamFuse): a job PUSHES the gradient elements
// it has just formed into slot [step parity][rank] of every peer's receive area (remote stores over NVLink, fire and forget), reads the
// peers' contributions to the same elements from its own receive area, adds the W contributions in rank order - the same order on
// every rank, so the replicas stay bit-identical - and applies the optimiser to the sum.  The gradients never go to memory on their
// own rank, and the all-reduce launch of an optimiser step disappears.
// Hand-over WITHOUT a fence: the first version raised a flag per block after a system-scope fence, and the stage stamps
// (RTD3_P2P_PROF, tools/dp_perf.py) showed the fence alone taking 4-17 us per block (MEMBAR.SYS waits for the acknowledgement of
// every remote store in flight) - 10 of the 26 us the kernel then took.  Now every value travels WITH its flag, as in NCCL's LL
// protocol: a 16-byte line is {value, step, value, step}, each 8-byte half is single-copy atomic, and the reader polls its own lines
// until both halves carry this step's number.  Twice the bytes on the link (1 MB per peer and critic step), no fence, no flag hop: the
// hand-over costs one NVLink one-way trip.  A slot is `stride` floats = room for a slice in line form (2 floats per element).
// Why the two parity slots suffice: the steps of a rank are kernel launches in stream order; rank A's step s + 1 kernel starts after its
// step s kernel has ended, i.e. after every block of A has seen B's step s lines, which B pushes only after its step s - 1 kernel has
// ended - so when A overwrites slot [(s + 1) & 1], B has finished reading it.  A reader that sees no line within 20 s traps.
// Stale words: a slot position that a line step last wrote carries an OLDER step number (never this one: the counter only grows, and the
// area starts zeroed while steps start at 1).  The all-reduce kernels of rtd3_p2p.cu (larger batches) share the area and leave raw
// gradient floats there; one of those would have to equal the current step number bit for bit - a denormal of the order of 1e-39 for
// the first billion steps - to be mistaken for a line.
struct P2pFuse {
  float* recv[kP2pMaxWorld];          // rank q's receive area as mapped here
  float* mine;                        // = recv[rank] (a field of its own: indexing the kernel parameter with a run-time rank would
                                      // send the whole struct through local memory)
  int world;                          // 0: no exchange
  int rank;
  unsigned long long* seq_counter;    // last completed step (device memory: a replayed graph counts on by itself)
  unsigned int* block_counter;
  int64_t stride;                     // floats between the [parity][rank] slots of a receive area (>= 2 x the largest slice)
  int64_t slice_off;                  // arena offset of the slice this optimiser step reduces
  float grad_scale;                   // 1 / world
  int mode;                           // 0 all to all, 1 reduce-scatter + all-gather (p2p_exchange4)
  unsigned long long* prof;           // development (RTD3_P2P_PROF=1): %globaltimer stamps [block][2 threads][8 stages], else nullptr
};
__device__ __forceinline__ void p2p_stamp(const P2pFuse& px, int cta, int k) {
  if (px.prof && threadIdx.x < 2) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    px.prof[(cta * 2 + threadIdx.x) * 8 + k] = t;
  }
}
// float offset of element `arena_idx` (line form) in slot [parity][r]
__device__ __forceinline__ int64_t p2p_slot(const P2pFuse& px, unsigned int seq, int r, int64_t arena_idx) {
  return ((int64_t)(seq & 1u) * px.world + r) * px.stride + 2 * (arena_idx - px.slice_off);
}
__device__ __forceinline__ void st_line(float* p, float a, float b, unsigned int f) {
  asm volatile("st.volatile.global.v4.b32 [%0], {%1, %2, %3, %2};" ::"l"(p), "r"(__float_as_uint(a)), "r"(f), "r"(__float_as_uint(b)) : "memory");
}
__device__ __forceinline__ uint4 ld_line(const float* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_half(float* p, float a, unsigned int f) {
  asm volatile("st.volatile.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(a)), "r"(f) : "memory");
}
__device__ __forceinline__ uint2 ld_half(const float* p) {
  uint2 v;
  asm volatile("ld.volatile.global.v2.b32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
// `only` = -1: to every peer; else to that rank alone
__device__ __forceinline__ void p2p_push4(const P2pFuse& px, unsigned int seq, int64_t arena_idx, float4 v, int only) {
  const int64_t at = p2p_slot(px, seq, px.rank, arena_idx);
#pragma unroll
  for (int q = 0; q < kP2pMaxWorld; ++q)
    if (q < px.world && q != px.rank && (only < 0 || q == only)) {
      st_line(px.recv[q] + at, v.x, v.y, seq);
      st_line(px.recv[q] + at + 4, v.z, v.w, seq);
    }
}
__device__ __forceinline__ void p2p_push1(const P2pFuse& px, unsigned int seq, int64_t arena_idx, float v, int only) {
  const int64_t at = p2p_slot(px, seq, px.rank, arena_idx);
#pragma unroll
  for (int q = 0; q < kP2pMaxWorld; ++q)
    if (q < px.world && q != px.rank && (only < 0 || q == only)) st_half(px.recv[q] + at, v, seq);
}
__device__ __forceinline__ void p2p_spin_check(unsigned long long& t0) {
  const unsigned long long now = global_ns();
  if (t0 == 0ull) t0 = now;
  else if (now - t0 > kSpinLimitNs) asm volatile("trap;");
}
// sum over the ranks in rank order (own contribution from registers), times grad_scale.  The lines of ALL peers are requested before
// the first one is examined (one round trip for W - 1 peers when they have arrived, instead of W - 1 dependent ones); a line that does
// not carry `seq` yet is polled.
__device__ __forceinline__ float4 p2p_sum4(const P2pFuse& px, unsigned int seq, int64_t arena_idx, float4 own) {
  const float* mine = px.mine;
  uint4 a[kP2pMaxWorld], b[kP2pMaxWorld];
#pragma unroll
  for (int r = 0; r < kP2pMaxWorld; ++r)
    if (r < px.world && r != px.rank) {
      const float* at = mine + p2p_slot(px, seq, r, arena_idx);
      a[r] = ld_line(at); b[r] = ld_line(at + 4);
    }
  unsigned long long t0 = 0ull;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int r = 0; r < kP2pMaxWorld; ++r) {
    if (r >= px.world) continue;
    float4 v = own;
    if (r != px.rank) {
      const float* at = mine + p2p_slot(px, seq, r, arena_idx);
      while (a[r].y != seq || a[r].w != seq || b[r].y != seq || b[r].w != seq) {
        p2p_spin_check(t0);
        a[r] = ld_line(at); b[r] = ld_line(at + 4);
      }
      v = make_float4(__uint_as_float(a[r].x), __uint_as_float(a[r].z), __uint_as_float(b[r].x), __uint_as_float(b[r].z));
    }
    if (r == 0) acc = v;
    else { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
  }
  return make_float4(acc.x * px.grad_scale, acc.y * px.grad_scale, acc.z * px.grad_scale, acc.w * px.grad_scale);
}
// the same for kN scalars of one thread (slot elements idx[i], live[i] = the thread owns element i): all kN x (W - 1) halves are requested first
template <int kN>
__device__ __forceinline__ void p2p_sum_n(const P2pFuse& px, unsigned int seq, const int64_t (&idx)[kN], const bool (&live)[kN], float (&val)[kN]) {
  const float* mine = px.mine;
  uint2 h[kN][kP2pMaxWorld];
#pragma unroll
  for (int i = 0; i < kN; ++i)
#pragma unroll
    for (int r = 0; r < kP2pMaxWorld; ++r)
      if (live[i] && r < px.world && r != px.rank) h[i][r] = ld_half(mine + p2p_slot(px, seq, r, idx[i]));
  unsigned long long t0 = 0ull;
#pragma unroll
  for (int i = 0; i < kN; ++i) {
    if (!live[i]) continue;
    float acc = 0.f;
#pragma unroll
    for (int r = 0; r < kP2pMaxWorld; ++r) {
      if (r >= px.world) continue;
      float v = val[i];
      if (r != px.rank) {
        const float* at = mine + p2p_slot(px, seq, r, idx[i]);
        while (h[i][r].y != seq) {
          p2p_spin_check(t0);
          h[i][r] = ld_half(at);
        }
        v = __uint_as_float(h[i][r].x);
      }
      acc = r == 0 ? v : acc + v;
    }
    val[i] = acc * px.grad_scale;
  }
}
// the lines rank `from` pushed for this element, as they are
__device__ __forceinline__ float4 p2p_take4(const P2pFuse& px, unsigned int seq, int64_t arena_idx, int from) {
  const float* at = px.mine + p2p_slot(px, seq, from, arena_idx);
  unsigned long long t0 = 0ull;
  uint4 a = ld_line(at), b = ld_line(at + 4);
  while (a.y != seq || a.w != seq || b.y != seq || b.w != seq) {
    p2p_spin_check(t0);
    a = ld_line(at); b = ld_line(at + 4);
  }
  return make_float4(__uint_as_float(a.x), __uint_as_float(a.z), __uint_as_float(b.x), __uint_as_float(b.z));
}
template <int kN>
__device__ __forceinline__ void p2p_take_n(const P2pFuse& px, unsigned int seq, const int64_t (&idx)[kN], const bool (&live)[kN], float (&val)[kN], int from) {
  const float* mine = px.mine;
  uint2 h[kN];
#pragma unroll
  for (int i = 0; i < kN; ++i)
    if (live[i]) h[i] = ld_half(mine + p2p_slot(px, seq, from, idx[i]));
  unsigned long long t0 = 0ull;
#pragma unroll
  for (int i = 0; i < kN; ++i) {
    if (!live[i]) continue;
    while (h[i].y != seq) {
      p2p_spin_check(t0);
      h[i] = ld_half(mine + p2p_slot(px, seq, from, idx[i]));
    }
    val[i] = __uint_as_float(h[i].x);
  }
}
// The exchange of a block's elements.  mode 0 (all to all): push to every peer, add all W contributions - one hop, (W - 1) x the bytes.
// mode 1 (reduce-scatter + all-gather, for W > 2): the block's OWNER rank (block % W) receives the W - 1 partial values, adds them in
// rank order and pushes the finished, scaled sum to every peer; the other ranks push to the owner alone and take the owner's sum as it
// is (bit-identical replicas) - two hops, 2 (W - 1) / W x the bytes per rank instead of (W - 1) x.  The owner's sums travel in slot
// [parity][owner] of the receivers' areas: at those positions nothing else arrives there (partial values only go to the owner's area).
__device__ __forceinline__ float4 p2p_exchange4(const P2pFuse& px, unsigned int seq, int owner, int64_t arena_idx, float4 v) {
  if (px.mode == 0) {
    p2p_push4(px, seq, arena_idx, v, -1);
    return p2p_sum4(px, seq, arena_idx, v);
  }
  if (px.rank == owner) {
    v = p2p_sum4(px, seq, arena_idx, v);
    p2p_push4(px, seq, arena_idx, v, -1);
    return v;
  }
  p2p_push4(px, seq, arena_idx, v, owner);
  return p2p_take4(px, seq, arena_idx, owner);
}
template <int kN>
__device__ __forceinline__ void p2p_exchange_n(const P2pFuse& px, unsigned int seq, int owner, const int64_t (&idx)[kN], const bool (&live)[kN], float (&val)[kN]) {
  const bool reduce_here = px.mode == 0 || px.rank == owner;
  if (px.mode == 0 || !reduce_here) {
#pragma unroll
    for (int i = 0; i < kN; ++i)
      if (live[i]) p2p_push1(px, seq, idx[i], val[i], px.mode == 0 ? -1 : owner);
  }
  if (reduce_here) p2p_sum_n<kN>(px, seq, idx, live, val);
  else p2p_take_n<kN>(px, seq, idx, live, val, owner);
  if (px.mode != 0 && reduce_here) {
#pragma unroll
    for (int i = 0; i < kN; ++i)
      if (live[i]) p2p_push1(px, seq, idx[i], val[i], -1);
  }
}
// bookkeeping of a step, by one thread per block: the last block to come by (every block has read the step number) advances it
__device__ __forceinline__ void p2p_step_done(const P2pFuse& px, unsigned long long seq64, int ncta) {
  if (atomicAdd(px.block_counter, 1u) == (unsigned)ncta - 1u) {
    *px.block_counter = 0u;
    *px.seq_counter = seq64;
  }
}

// ---- weight gradients from the row scratch, reduced over the batch without atomics -----------------------------------
//   hidden layer l (1..L-1):  gW_l[n][k] = sum_b dz_l[b][n] * h_{l-1}[b][k]      32x32 output tiles
//   every hidden layer l:     gb_l[n]    = sum_b dz_l[b][n];   l = 0 also gW_0[n][j] = sum_b dz_0[b][n] * in0[b][j]
//   output layer:             gW_L[o][k] = sum_b dout[b][o] * h_{L-1}[b][k];  gb_L[o] = sum_b dout[b][o]
// blockIdx.x = job, blockIdx.y = network slot, blockIdx.z = batch split (>1 only for large batches: atomicAdd into
// gradients that the optimiser pass left zeroed).  Each of the 8 warps reduces every 8th row; the partial tiles meet in smem.
struct WgradSlots {
  int64_t grad_off[2];      // offset of the slot's network in the gradient arena
  int64_t scratch_off[2];   // offset of the slot's row scratch
};

constexpr int kWgradRows = 256;                                   // batch rows staged per pass
constexpr size_t kWgradSmem = 2 * kWgradRows * 32 * sizeof(float);  // dz slab + layer-input slab (the partial tiles alias them)

__global__ void __launch_bounds__(kThreads, 2)     // two blocks per SM: the whole grid is resident at once (the peer exchange needs it)
wgrad_kernel(NetShape s, const float* __restrict__ scratch, float* __restrict__ grads, WgradSlots slots, int B, int rows_per_split, AdamFuse fz,
             P2pFuse px) {
  __shared__ __align__(16) float red_small[8][32 * 5];
  // peer exchange: this step's number (the last block whose threads have all read it advances it)
  const unsigned long long seq64 = px.world ? *reinterpret_cast<volatile unsigned long long*>(px.seq_counter) + 1ull : 0ull;
  const unsigned int seq = (unsigned int)seq64;                      // the number the lines of this step carry
  const int cta = blockIdx.y * gridDim.x + blockIdx.x, ncta = gridDim.x * gridDim.y;
  p2p_stamp(px, cta, 0);
  if (px.world) {
    __syncthreads();                                                 // every thread of the block has read the step number
    if (threadIdx.x == 32) p2p_step_done(px, seq64, ncta);
  }
  // fused optimiser: the Adam clocks are loaded now, the step size is formed after the batch reduction
  const AdamState& os = fz.adam;
  double bp1 = 0.0, bp2 = 0.0;
  if (os.params) { bp1 = os.beta_pows[2 * fz.opt]; bp2 = os.beta_pows[2 * fz.opt + 1]; }
  const double lr = fz.opt ? os.lr[1] : os.lr[0];   // selected before the reduction: selected after it, it sent the whole AdamFuse to the stack (256 B, spills)
  auto step_size = [&]() { return adam_step(lr, bp1, bp2); };
  // the optimiser's operands of one element, fetched BEFORE the batch reduction (the small jobs' five emits were five dependent
  // chains of two L2 round trips each - the longest blocks of the launch)
  struct OptPre { float m, v, p, t; };
  auto pre_load = [&](int64_t net_off, int64_t o) {
    OptPre q{0.f, 0.f, 0.f, 0.f};
    if (os.params) {
      const int64_t i = net_off + o;
      q.m = os.m[i]; q.v = os.v[i]; q.p = os.params[i];
      if (fz.polyak) q.t = os.params[fz.n_online + i];
    }
    return q;
  };
  auto emit_pre = [&](int64_t net_off, int64_t o, float g, bool atomic_acc, const OptPre& q) {
    if (!os.params) {
      float* dst = grads + net_off + o;
      if (atomic_acc) atomicAdd(dst, g); else *dst = g;
      return;
    }
    adam_polyak1(os, (int)(net_off + o), (int)net_off, copy_index(s, (int)o), g, q.m, q.v, q.p, q.t, step_size(), true, fz.polyak, fz.n_online, fz.total);
  };
  const int H = s.hid, L = s.layers;
  const int nch = (H + 31) / 32;
  const int nT = (L - 1) * nch * nch, nS = L * nch;
  const int job = blockIdx.x;
  const int slot = blockIdx.y;
  const RowScratch rs{const_cast<float*>(scratch) + slots.scratch_off[slot], B, H, L};
  const int64_t G0 = slots.grad_off[slot];
  const bool atomic = gridDim.z > 1;
  const int b_lo = blockIdx.z * rows_per_split, b_hi = min(B, b_lo + rows_per_split);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (job < nT) {
    // 32 x 32 tile of gW_l: both operand slabs ([rows][32] of dz_l and of h_{l-1}) are staged with ONE round of cp.async (the loop of
    // dependent L2 loads it replaces ran at 8 warps per SM: ncu 2.7 long-scoreboard stalls per issue, 15 k of the kernel's 36 k cycles)
    const int l = 1 + job / (nch * nch);
    const int tile = job % (nch * nch);
    const int n0 = (tile / nch) * 32, k0 = (tile % nch) * 32;
    const float* dz = rs.dz(l);
    const float* x = rs.h(l - 1);
    const int ty = lane >> 2, tx = lane & 3;
    float* sz = smem_f;
    float* sx = smem_f + kWgradRows * 32;
    // the optimiser's operands of this thread's 4 consecutive outputs, fetched under the batch reduction
    const int o = threadIdx.x * 4;
    const int gn = n0 + (o >> 5), gk = k0 + (o & 31);
    const bool out_ok = gn < H && gk < H;
    const int64_t off = net_w_off(s, l) + (int64_t)gn * H + gk;
    float4 m4 = make_float4(0.f, 0.f, 0.f, 0.f), v4 = m4, p4 = m4, t4 = m4;
    if (os.params && out_ok) {
      m4 = *reinterpret_cast<const float4*>(os.m + G0 + off);
      v4 = *reinterpret_cast<const float4*>(os.v + G0 + off);
      p4 = *reinterpret_cast<const float4*>(os.params + G0 + off);
      if (fz.polyak) t4 = *reinterpret_cast<const float4*>(os.params + fz.n_online + G0 + off);
    }
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int c0 = b_lo; c0 < b_hi; c0 += kWgradRows) {
      const int rows = min(kWgradRows, b_hi - c0);
      for (int i = threadIdx.x; i < rows * 8; i += kThreads) {
        const int r = i >> 3, q4 = (i & 7) * 4;
        if (n0 + q4 < H) cp_async16(sz + r * 32 + q4, dz + (int64_t)(c0 + r) * H + n0 + q4);
        else *reinterpret_cast<float4*>(sz + r * 32 + q4) = make_float4(0.f, 0.f, 0.f, 0.f);
        if (k0 + q4 < H) cp_async16(sx + r * 32 + q4, x + (int64_t)(c0 + r) * H + k0 + q4);
        else *reinterpret_cast<float4*>(sx + r * 32 + q4) = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      cp_commit();
      cp_wait<0>();
      __syncthreads();
#pragma unroll 4
      for (int b = warp; b < rows; b += 8) {
        const float4 z = *reinterpret_cast<const float4*>(sz + b * 32 + ty * 4);
        const float4 x0 = *reinterpret_cast<const float4*>(sx + b * 32 + tx * 8);
        const float4 x1 = *reinterpret_cast<const float4*>(sx + b * 32 + tx * 8 + 4);
        const float zz[4] = {z.x, z.y, z.z, z.w};
        const float xx[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(zz[i], xx[j], acc[i][j]);
      }
      __syncthreads();
    }
    float* red = smem_f;                      // [8][32 * 32], over the slabs
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float* dst = red + warp * 1024 + (ty * 4 + i) * 32 + tx * 8;
      *reinterpret_cast<float4*>(dst) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
      *reinterpret_cast<float4*>(dst + 4) = make_float4(acc[i][4], acc[i][5], acc[i][6], acc[i][7]);
    }
    __syncthreads();
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const float4 p = *reinterpret_cast<const float4*>(red + w * 1024 + o);
      v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    }
    if (px.world) {
      p2p_stamp(px, cta, 1);
      if (out_ok) v = p2p_exchange4(px, seq, cta % px.world, G0 + off, v);
      p2p_stamp(px, cta, 5);
    }
    if (out_ok) {
      if (!os.params) {
        if (!atomic) *reinterpret_cast<float4*>(grads + G0 + off) = v;
        else { atomicAdd(grads + G0 + off, v.x); atomicAdd(grads + G0 + off + 1, v.y); atomicAdd(grads + G0 + off + 2, v.z); atomicAdd(grads + G0 + off + 3, v.w); }
      } else {                                // W_l[gn][gk..gk+3]
        const float g4[4] = {v.x, v.y, v.z, v.w};
        adam_polyak4(os, (int)(G0 + off), (int)G0, copy_index(s, l - 1, gn, gk), H, g4, m4, v4, p4, t4, step_size(), true, fz.polyak, fz.n_online, fz.total);
      }
    }
    p2p_stamp(px, cta, 6);
  } else if (job < nT + nS) {
    // bias gradients of hidden layer l for 32 units (and, l = 0, the first-layer weights).  After the batch reduction warp q finishes
    // value q of unit n = lane (q = 0 the bias, 1 + j the weight of input j): one optimiser element - and one peer exchange - per
    // thread instead of five dependent ones in warp 0.
    const int l = (job - nT) / nch, n = ((job - nT) % nch) * 32 + lane;
    const float* dz = rs.dz(l);
    const float* in0 = rs.in0();
    float ab = 0.f, aw[4] = {0.f, 0.f, 0.f, 0.f};
    const bool own = warp < 5 && n < H && (warp == 0 || (l == 0 && warp - 1 < s.in));
    const int64_t o = warp == 0 ? net_b_off(s, l) + n : net_w_off(s, 0) + (int64_t)n * s.in + (warp - 1);
    OptPre pre{0.f, 0.f, 0.f, 0.f};
    if (own) pre = pre_load(G0, o);
    if (n < H) {
#pragma unroll 8
      for (int b = b_lo + warp; b < b_hi; b += 8) {
        const float d = __ldg(dz + (int64_t)b * H + n);
        ab += d;
        if (l == 0) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(in0 + (int64_t)b * 4));
          aw[0] = fmaf(d, x.x, aw[0]); aw[1] = fmaf(d, x.y, aw[1]); aw[2] = fmaf(d, x.z, aw[2]); aw[3] = fmaf(d, x.w, aw[3]);
        }
      }
    }
    float* r = &red_small[warp][lane * 5];
    r[0] = ab; r[1] = aw[0]; r[2] = aw[1]; r[3] = aw[2]; r[4] = aw[3];
    __syncthreads();
    float v[1] = {0.f};
    if (own)
      for (int w = 0; w < 8; ++w) v[0] += red_small[w][lane * 5 + warp];
    if (px.world) {
      const int64_t ix[1] = {G0 + o};
      const bool lv[1] = {own};
      p2p_exchange_n<1>(px, seq, cta % px.world, ix, lv, v);
    }
    if (own) emit_pre(G0, o, v[0], atomic, pre);
  } else {
    // output layer: warp o < 2 finishes W_L[o][k] for k = lane of this chunk, warp 2 of chunk 0 the biases
    const int chunk = job - nT - nS, k = chunk * 32 + lane;
    const float* hl = rs.h(L - 1);
    const float* dout = rs.dout();
    float a0 = 0.f, a1 = 0.f, s0 = 0.f, s1 = 0.f;
    const bool own = (warp < 2 && warp < s.out && k < H) || (warp == 2 && chunk == 0 && lane < s.out);
    const int64_t o = warp < 2 ? net_w_off(s, L) + (int64_t)warp * H + k : net_b_off(s, L) + lane;
    const int q = warp < 2 ? warp : 2 + lane;                           // which of the four reduced values
    OptPre pre{0.f, 0.f, 0.f, 0.f};
    if (own) pre = pre_load(G0, o);
#pragma unroll 8
    for (int b = b_lo + warp; b < b_hi; b += 8) {
      const float2 d = __ldg(reinterpret_cast<const float2*>(dout + (int64_t)b * 2));
      const float h = k < H ? __ldg(hl + (int64_t)b * H + k) : 0.f;
      a0 = fmaf(d.x, h, a0); a1 = fmaf(d.y, h, a1);
      s0 += d.x; s1 += d.y;
    }
    float* r = &red_small[warp][lane * 4];
    r[0] = a0; r[1] = a1; r[2] = s0; r[3] = s1;
    __syncthreads();
    float v[1] = {0.f};
    if (own)
      for (int w = 0; w < 8; ++w) v[0] += red_small[w][lane * 4 + q];
    if (px.world) {
      const int64_t ix[1] = {G0 + o};
      const bool lv[1] = {own};
      p2p_exchange_n<1>(px, seq, cta % px.world, ix, lv, v);
    }
    if (own) emit_pre(G0, o, v[0], atomic, pre);
  }
}

// Rebuild the whole transposed arena from the parameters (after weights were written from outside the optimiser).
__global__ void td3_sync_transposed_kernel(Arena ar, const float* __restrict__ params, float* __restrict__ params_t) {
  const int64_t total = ar.total(), n_online = ar.online_total();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i < n_online ? i : i - n_online;
    const int net = j < ar.off(1) ? 0 : (j < ar.off(2) ? 1 : 2);
    const int64_t base = (i < n_online ? 0 : n_online) + ar.off(net);
    params_t[base + copy_index(net == 0 ? ar.actor : ar.critic, (int)(i - base)).t] = params[i];
  }
}

// ---- Adam (torch.optim.Adam defaults, robot.py:237-239) + optional Polyak (robot.py:293-310), one pass --------------
// nets: bit 0 actor, bit 1 critic1, bit 2 critic2 get an Adam step from `grads` (then the gradients are zeroed);
// polyak: same bit layout; afterwards the selected target slots are blended with their (updated) online net:
// t = t*(1-tau) + p*tau.
__global__ void td3_adam_polyak_kernel(AdamState st, float* __restrict__ grads, int nets, float grad_scale, int polyak) {
  __shared__ float s_step[2], s_bc2[2];
  if (threadIdx.x < 2) {                                              // 0: actor optimiser, 1: both critic optimisers
    const AdamStep k = adam_step(threadIdx.x == 0 ? st.lr[0] : st.lr[1], st.beta_pows[2 * threadIdx.x], st.beta_pows[2 * threadIdx.x + 1]);
    s_step[threadIdx.x] = k.step;
    s_bc2[threadIdx.x] = k.sqrt_bc2;
  }
  __syncthreads();
  const int n4 = (int)(st.ar.online_total() >> 2);                  // slots are multiples of 4 floats: a group of 4 never straddles two networks
  for (int i4 = blockIdx.x * blockDim.x + threadIdx.x; i4 < n4; i4 += gridDim.x * blockDim.x) {
    const int i = i4 * 4;
    const int net = i < (int)st.ar.off(1) ? 0 : (i < (int)st.ar.off(2) ? 1 : 2);
    const bool do_adam = (nets >> net) & 1, do_polyak = (polyak >> net) & 1;
    if (!do_adam && !do_polyak) continue;
    float g[4] = {0.f, 0.f, 0.f, 0.f};
    if (do_adam) {
      const float4 g4 = *reinterpret_cast<const float4*>(grads + i);
      g[0] = g4.x * grad_scale; g[1] = g4.y * grad_scale; g[2] = g4.z * grad_scale; g[3] = g4.w * grad_scale;
      *reinterpret_cast<float4*>(grads + i) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int o = net == 0 ? 0 : 1;
    adam_polyak_apply4(st, i, net, g, AdamStep{s_step[o], s_bc2[o]}, do_adam, do_polyak);
  }
}

// ---- plain forward of one network over B rows (actor inference for get_next_action, parity checks of Q-values) ------
template <int R>
__global__ void __launch_bounds__(kThreads, 1)
mlp_forward_kernel(NetShape s, const float* __restrict__ P, const float* __restrict__ Pt, const float* __restrict__ x /*[B][in]*/, float* __restrict__ y /*[B][out]*/,
                   int B) {
  MlpSmem<R> sm;
  sm.carve(0, s.hid, 0);
  const int r0 = blockIdx.x * R, t = threadIdx.x;
  if (t < R * 4) {
    const int r = t >> 2, j = t & 3, row = r0 + r;
    smem_f[sm.in0 + t] = (row < B && j < s.in) ? x[(int64_t)row * s.in + j] : 0.f;
  }
  __syncthreads();
  mlp_forward<R>(P, Pt, s, sm, false, nullptr, r0);
  if (t < R * s.out) {
    const int r = t / s.out, o = t - r * s.out;
    if (r0 + r < B) y[(int64_t)(r0 + r) * s.out + o] = smem_f[sm.out + r * 2 + o];
  }
}

// ---- replay ring (robot.py:79-96): push n rows starting at `position`, wrapping at capacity -------------------------
__global__ void replay_push_kernel(float2* s, float2* a, float* r, float2* s2, float* notdone, int64_t capacity, int64_t position,
                                   const float* __restrict__ sx, const float* __restrict__ sy, const float* __restrict__ ax,
                                   const float* __restrict__ ay, const float* __restrict__ rew, const float* __restrict__ nx,
                                   const float* __restrict__ ny, const uint8_t* __restrict__ done, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t p = (position + i) % capacity;
  s[p] = make_float2(sx[i], sy[i]);
  a[p] = make_float2(ax[i], ay[i]);
  r[p] = rew[i];
  s2[p] = make_float2(nx[i], ny[i]);
  notdone[p] = done[i] ? 0.f : 1.f;
}

// ReplayBuffer.sample's gather (robot.py:113-115): rows idx[b] -> dense minibatch arrays
__global__ void replay_gather_kernel(ReplayView rp, const int32_t* __restrict__ idx, int B, float2* os, float2* oa, float* orw,
                                     float2* os2, float* ond) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int j = idx[b];
  os[b] = rp.s[j]; oa[b] = rp.a[j]; orw[b] = rp.r[j]; os2[b] = rp.s2[j]; ond[b] = rp.notdone[j];
}

static bool shape_ok(const NetShape& s) {
  return s.in >= 1 && s.in <= 4 && s.out >= 1 && s.out <= 2 && s.layers >= 1 && s.layers <= kMaxLayers && s.hid >= 4 &&
         s.hid <= kMaxHidden && s.hid % 4 == 0;
}

}  // namespace rtd3

using namespace rtd3;

// Rows per CTA: few rows while the batch cannot fill the SMs (latency-bound), more rows once it can (every CTA
// re-streams all weights from L2, so larger tiles cut that traffic).
static inline int pick_tile(int64_t B, int num_sms) {
  if (B <= 2 * (int64_t)num_sms) return 0;
  if (B <= 4 * (int64_t)num_sms) return 1;
  if (B <= 16 * (int64_t)num_sms) return 2;
  return 3;
}

static size_t actor_phase_smem(const Arena& ar, int R) {
  return mlp_smem_bytes(R, ar.critic.hid, ar.critic.layers) + ((size_t)ar.actor.layers * R * (ar.critic.hid + 4) + R * 4) * sizeof(float);
}

template <typename K>
static cudaError_t set_smem(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// Every row-tile instantiation a launch can pick, [pick_tile]; rtd3_td3_create sets the shared-memory limit of every entry.
static_assert(kNumTiles == 4 && kRowTiles[0] == 2 && kRowTiles[1] == 4 && kRowTiles[2] == 8 && kRowTiles[3] == 16, "tables follow kRowTiles");
using CriticKernel = decltype(&td3_critic_kernel<2>);
static const CriticKernel kCriticKernels[kNumTiles] = {td3_critic_kernel<2>, td3_critic_kernel<4>, td3_critic_kernel<8>, td3_critic_kernel<16>};
using ActorKernel = decltype(&td3_actor_kernel<2>);
static const ActorKernel kActorKernels[kNumTiles] = {td3_actor_kernel<2>, td3_actor_kernel<4>, td3_actor_kernel<8>, td3_actor_kernel<16>};
using FwdKernel = decltype(&mlp_forward_kernel<2>);
static const FwdKernel kFwdKernels[kNumTiles] = {mlp_forward_kernel<2>, mlp_forward_kernel<4>, mlp_forward_kernel<8>, mlp_forward_kernel<16>};

static unsigned long long* g_p2p_prof = nullptr;   // development: stage stamps of the last fused weight-gradient launch

static int wgrad_jobs(const NetShape& s) {
  const int nch = (s.hid + 31) / 32;
  return (s.layers - 1) * nch * nch + s.layers * nch + nch;
}

static int32_t launch_wgrad(rtd3_td3* h, const NetShape& s, const float* scratch, float* grads, const WgradSlots& slots, int nslots, int B,
                            cudaStream_t st, const AdamFuse& fz = AdamFuse{}, const P2pFuse& px = P2pFuse{}) {
  const int jobs = wgrad_jobs(s);
  const int rows_per_split = 512;
  const int bsplit = (B + rows_per_split - 1) / rows_per_split;
  RTD3_CHECK_ARG(!fz.adam.params || bsplit == 1, "the fused optimiser needs batch <= 512");
  RTD3_CHECK_ARG(!px.world || (fz.adam.params && jobs * nslots <= kP2pBlockFlags), "the fused peer exchange needs the fused optimiser and at most 256 blocks");
  RTD3_CUDA(ensure_dyn_smem((const void*)wgrad_kernel, kWgradSmem));
  static const bool coop_env = !(getenv("RTD3_P2P_COOP") && atoi(getenv("RTD3_P2P_COOP")) == 0);
  if (px.world && coop_env) {
    // every block waits for the same block of its peers: placed as a whole or not at all (see rtd3_p2p_allreduce)
    NetShape s_ = s; WgradSlots sl = slots; AdamFuse fz_ = fz; P2pFuse px_ = px;
    int B_ = B, rps = rows_per_split;
    void* kargs[] = {&s_, &scratch, &grads, &sl, &B_, &rps, &fz_, &px_};
    RTD3_CUDA(cudaLaunchCooperativeKernel((const void*)wgrad_kernel, dim3(jobs, nslots, bsplit), dim3(kThreads), kargs, kWgradSmem, st));
  } else {
    wgrad_kernel<<<dim3(jobs, nslots, bsplit), kThreads, kWgradSmem, st>>>(s, scratch, grads, slots, B, rows_per_split, fz, px);
  }
  RTD3_LAUNCHED();
  return 0;
}

// One critic / actor step of the fp32 kernels: the row tiles or the cluster kernels, then the weight-gradient pass (with the optimiser
// and the peer exchange fused into it on request).
static int32_t critic_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const ReplayView& rp,
                           const int32_t* idx, const float* noise, int32_t batch, const Td3Hyper& hp, float* loss2, float* q_out, float* y_out,
                           int32_t* steps, double* beta_pows, cudaStream_t st, const AdamFuse& fz = AdamFuse{}, const P2pFuse& px = P2pFuse{}) {
  if (cluster_path_ok(h, batch)) {
    const int32_t rc = critic_cluster_launch(h, params, params_t, scratch, rp, idx, noise, batch, hp, loss2, q_out, y_out, steps, beta_pows, st);
    if (rc) return rc;
  } else {
    const int ti = pick_tile(batch, h->num_sms);
    const int R = kRowTiles[ti];
    kCriticKernels[ti]<<<(batch + R - 1) / R, kThreads, h->smem_critic[ti], st>>>(h->ar, params, params_t, scratch, rp, idx, noise, batch, hp, loss2,
                                                                                   q_out, y_out, steps, beta_pows);
    RTD3_LAUNCHED();
  }
  WgradSlots slots;
  const int64_t per = RowScratch::floats(batch, h->ar.critic.hid, h->ar.critic.layers);
  slots.grad_off[0] = h->ar.off(1); slots.grad_off[1] = h->ar.off(2);
  slots.scratch_off[0] = 0; slots.scratch_off[1] = per;
  return launch_wgrad(h, h->ar.critic, scratch, grads, slots, 2, batch, st, fz, px);
}

static int32_t actor_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const float* rp_s,
                          const int32_t* idx, int32_t batch, float* loss1, int32_t* steps, double* beta_pows, void* stream,
                          const AdamFuse& fz = AdamFuse{}, const P2pFuse& px = P2pFuse{}) {
  RTD3_CHECK_ARG(h && params && params_t && grads && scratch && rp_s && idx && loss1 && steps && beta_pows, "null argument");
  RTD3_CHECK_ARG(batch > 0, "batch must be positive");
  ReplayView rp{(const float2*)rp_s, nullptr, nullptr, nullptr, nullptr};
  cudaStream_t st = (cudaStream_t)stream;
  if (cluster_path_ok(h, batch)) {
    const int32_t rc = actor_cluster_launch(h, params, params_t, scratch, rp, idx, batch, loss1, steps, beta_pows, st);
    if (rc) return rc;
  } else {
    const int ti = pick_tile(batch, h->num_sms);
    const int R = kRowTiles[ti];
    kActorKernels[ti]<<<(batch + R - 1) / R, kThreads, h->smem_actor[ti], st>>>(h->ar, params, params_t, scratch, rp, idx, batch, loss1, steps,
                                                                                 beta_pows);
    RTD3_LAUNCHED();
  }
  WgradSlots slots;
  slots.grad_off[0] = h->ar.off(0); slots.grad_off[1] = 0;
  slots.scratch_off[0] = 0; slots.scratch_off[1] = 0;
  return launch_wgrad(h, h->ar.actor, scratch, grads, slots, 1, batch, st, fz, px);
}

extern "C" {

int32_t rtd3_td3_create(rtd3_td3** out, int32_t device, int32_t hidden, int32_t layers) {
  RTD3_CHECK_ARG(out, "out is null");
  rtd3_td3* h = new rtd3_td3();
  h->ar.actor = NetShape{2, hidden, layers, 2};
  h->ar.critic = NetShape{4, hidden, layers, 1};
  if (!shape_ok(h->ar.actor)) {
    delete h;
    rtd3::set_error("rtd3_td3_create: hidden must be a multiple of 4 in [4,%d], layers in [1,%d]", kMaxHidden, kMaxLayers);
    return RTD3_ERR_ARG;
  }
  h->device = device;
  int prev = 0;
  RTD3_CUDA(cudaGetDevice(&prev));
  RTD3_CUDA(cudaSetDevice(device));
  RTD3_CUDA(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device));
  for (int i = 0; i < kNumTiles; ++i) {
    const int R = kRowTiles[i];
    h->smem_critic[i] = mlp_smem_bytes(R, hidden, layers);
    h->smem_actor[i] = actor_phase_smem(h->ar, R);
    h->smem_fwd[i] = mlp_smem_bytes(R, hidden, 0);
    RTD3_CUDA(set_smem(kCriticKernels[i], h->smem_critic[i]));
    RTD3_CUDA(set_smem(kActorKernels[i], h->smem_actor[i]));
    RTD3_CUDA(set_smem(kFwdKernels[i], h->smem_fwd[i]));
  }
  h->cluster_cap = std::max(0, rtd3_td3_cluster_occupancy(h, 256));     // (queried here, never inside a stream capture)
  RTD3_CUDA(cudaSetDevice(prev));
  if (!g_p2p_prof && getenv("RTD3_P2P_PROF") && atoi(getenv("RTD3_P2P_PROF")) == 1) {      // development: stage stamps of the fused exchange
    RTD3_CUDA(cudaMalloc(&g_p2p_prof, kP2pBlockFlags * 16 * sizeof(unsigned long long)));
    RTD3_CUDA(cudaMemset(g_p2p_prof, 0, kP2pBlockFlags * 16 * sizeof(unsigned long long)));
  }
  *out = h;
  return 0;
}

int32_t rtd3_td3_destroy(rtd3_td3* h) {
  delete h;
  return 0;
}

int64_t rtd3_td3_param_count(const rtd3_td3* h, int32_t net) {
  if (!h) return -1;
  return net_param_count(net == 0 || net == 3 ? h->ar.actor : h->ar.critic);
}
int64_t rtd3_td3_param_offset(const rtd3_td3* h, int32_t net) { return h ? h->ar.off(net) : -1; }
int64_t rtd3_td3_arena_floats(const rtd3_td3* h) { return h ? h->ar.total() : -1; }
int64_t rtd3_td3_scratch_floats(const rtd3_td3* h, int32_t batch) {
  return h ? 2 * RowScratch::floats(batch, h->ar.critic.hid, h->ar.critic.layers) : -1;
}

int32_t rtd3_td3_sync_transposed(rtd3_td3* h, const float* params, float* params_t, void* stream) {
  RTD3_CHECK_ARG(h && params && params_t, "null argument");
  td3_sync_transposed_kernel<<<h->num_sms * 2, 256, 0, (cudaStream_t)stream>>>(h->ar, params, params_t);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_td3_critic_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const float* rp_s, const float* rp_a,
                             const float* rp_r, const float* rp_s2, const float* rp_notdone, const int32_t* idx, const float* noise,
                             int32_t batch, float gamma, float policy_noise, float noise_clip, float max_action, float* loss2, float* q_out,
                             float* y_out, int32_t* steps, double* beta_pows, void* stream) {
  RTD3_CHECK_ARG(h && params && params_t && grads && scratch && rp_s && rp_a && rp_r && rp_s2 && rp_notdone && idx && noise && loss2 && steps && beta_pows,
                 "null argument");
  RTD3_CHECK_ARG(batch > 0, "batch must be positive");
  ReplayView rp{(const float2*)rp_s, (const float2*)rp_a, rp_r, (const float2*)rp_s2, rp_notdone};
  Td3Hyper hp{gamma, policy_noise, noise_clip, max_action, 0ull, nullptr, 0ull};
  return critic_step(h, params, params_t, grads, scratch, rp, idx, noise, batch, hp, loss2, q_out, y_out, steps, beta_pows, (cudaStream_t)stream);
}

int32_t rtd3_td3_actor_step(rtd3_td3* h, const float* params, const float* params_t, float* grads, float* scratch, const float* rp_s, const int32_t* idx,
                            int32_t batch, float* loss1, int32_t* steps, double* beta_pows, void* stream) {
  return actor_step(h, params, params_t, grads, scratch, rp_s, idx, batch, loss1, steps, beta_pows, stream);
}

int32_t rtd3_td3_adam_polyak(rtd3_td3* h, float* params, float* params_t, float* params_uv, float* grads, float* adam_m, float* adam_v, const double* beta_pows, int32_t nets,
                             double lr_actor, double lr_critic, float grad_scale, int32_t polyak, float tau, void* stream) {
  RTD3_CHECK_ARG(h && params && params_t && grads && adam_m && adam_v && beta_pows, "null argument");
  const int64_t n = h->ar.online_total();
  const int block = 256;
  const int grid = (int)std::min<int64_t>(ceil_div(n / 4, block), (int64_t)h->num_sms * 8);
  const AdamState opt{h->ar, params, params_t, params_uv, adam_m, adam_v, const_cast<double*>(beta_pows), {lr_actor, lr_critic}, tau};   // clocks read only
  td3_adam_polyak_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(opt, grads, nets, grad_scale, polyak);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_mlp_forward(rtd3_td3* h, int32_t net, const float* params, const float* params_t, const float* x, float* y, int64_t batch,
                         void* stream) {
  RTD3_CHECK_ARG(h && params && params_t && x && y, "null argument");
  RTD3_CHECK_ARG(net >= 0 && net < 6, "net index out of range");
  RTD3_CHECK_ARG(batch >= 0 && batch < (1ll << 31), "bad batch");
  if (batch == 0) return 0;
  const NetShape s = (net == 0 || net == 3) ? h->ar.actor : h->ar.critic;
  const int ti = pick_tile(batch, h->num_sms);
  const int R = kRowTiles[ti];
  const int grid = (int)((batch + R - 1) / R);
  kFwdKernels[ti]<<<grid, kThreads, h->smem_fwd[ti], (cudaStream_t)stream>>>(s, params + h->ar.off(net), params_t + h->ar.off(net), x, y, (int)batch);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_replay_push(float* s, float* a, float* r, float* s2, float* notdone, int64_t capacity, int64_t position, const float* sx,
                         const float* sy, const float* ax, const float* ay, const float* reward, const float* nx, const float* ny,
                         const uint8_t* done, int64_t n, void* stream) {
  RTD3_CHECK_ARG(s && a && r && s2 && notdone && sx && sy && ax && ay && reward && nx && ny && done, "null argument");
  RTD3_CHECK_ARG(capacity > 0 && position >= 0 && position < capacity && n >= 0, "bad capacity/position/n");
  if (n == 0) return 0;
  replay_push_kernel<<<(int)ceil_div(n, 256), 256, 0, (cudaStream_t)stream>>>((float2*)s, (float2*)a, r, (float2*)s2, notdone, capacity,
                                                                              position, sx, sy, ax, ay, reward, nx, ny, done, n);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_replay_gather(const float* s, const float* a, const float* r, const float* s2, const float* notdone, const int32_t* idx,
                           int32_t batch, float* out_s, float* out_a, float* out_r, float* out_s2, float* out_notdone, void* stream) {
  RTD3_CHECK_ARG(s && a && r && s2 && notdone && idx && out_s && out_a && out_r && out_s2 && out_notdone, "null argument");
  RTD3_CHECK_ARG(batch >= 0, "negative batch");
  if (batch == 0) return 0;
  ReplayView rp{(const float2*)s, (const float2*)a, r, (const float2*)s2, notdone};
  replay_gather_kernel<<<(batch + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rp, idx, batch, (float2*)out_s, (float2*)out_a, out_r,
                                                                              (float2*)out_s2, out_notdone);
  RTD3_LAUNCHED();
  return 0;
}


// ---- TD3.td3_update (robot.py:258-285) as ONE call: the epoch loop, the gradient all-reduce of the data-parallel learner and the
// optimiser / Polyak steps issued on `stream` (plain launches: the whole call can be captured in a CUDA graph, the NCCL node included).
__global__ void advance_counter_kernel(unsigned long long* counter, unsigned long long by) { counter[0] += by; }

}  // extern "C"
int32_t rtd3::advance_noise_counter(uint64_t* counter, uint64_t by, cudaStream_t st) {
  advance_counter_kernel<<<1, 1, 0, st>>>((unsigned long long*)counter, (unsigned long long)by);
  RTD3_LAUNCHED();
  return 0;
}
extern "C" {

__global__ void target_noise_kernel(Td3Hyper hp, float2* __restrict__ out, int64_t rows) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows) out[i] = target_noise(nullptr, hp, (int)i);
}

static int32_t update_allreduce(const rtd3_td3_update_args* a, int64_t off, int64_t count, cudaStream_t st) {
  if (a->world <= 1) return 0;
  if (a->p2p) {
    const rtd3_p2p_state* p = a->p2p;
    return rtd3_p2p_allreduce(p->peer_recv, p->peer_flags, p->rank, p->world, p->seq_counter, p->sum + off, a->grads + off, count, p->slot_floats,
                              p->block_counter, st);
  }
  return rtd3_allreduce_grads(a->comm, a->grads + off, count, st);
}

int32_t rtd3_td3_target_noise(uint64_t seed, uint64_t counter, float* out, int64_t rows, void* stream) {
  RTD3_CHECK_ARG(out && rows >= 0 && rows < (1ll << 31), "bad argument");
  if (rows == 0) return 0;
  // the generator of the critic kernels (rtd3_td3.cuh: target_noise), evaluated for rows 0..rows-1 of step `counter`
  const Td3Hyper hp{0.f, 0.f, 0.f, 0.f, (unsigned long long)seed, nullptr, (unsigned long long)counter};
  target_noise_kernel<<<(int)ceil_div(rows, 256), 256, 0, (cudaStream_t)stream>>>(hp, (float2*)out, rows);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3_td3_update(rtd3_td3* h, const rtd3_td3_update_args* a, void* stream) {
  RTD3_CHECK_ARG(h && a, "null argument");
  RTD3_CHECK_ARG(a->params && a->params_t && a->grads && a->adam_m && a->adam_v && a->steps && a->beta_pows, "null learner state");
  RTD3_CHECK_ARG(a->rp_s && a->rp_a && a->rp_r && a->rp_s2 && a->rp_notdone && a->idx, "null replay ring / index sets");
  RTD3_CHECK_ARG(a->batch > 0 && a->epochs >= 0 && a->policy_update_delay >= 1, "bad batch / epochs / policy_update_delay");
  RTD3_CHECK_ARG(a->critic_losses && a->actor_losses, "null loss outputs");
  RTD3_CHECK_ARG(a->noise || a->noise_counter, "either a noise tensor or the device noise counter is required");
  RTD3_CHECK_ARG(a->world >= 1 && (a->world == 1 || a->comm || a->p2p), "world > 1 needs a communicator (rtd3_comm) or a peer-memory state");
  RTD3_CHECK_ARG(!a->p2p || (a->p2p->world == a->world && a->p2p->sum), "peer-memory state of another world size");
  const bool tc = a->tf32 != 0;
  RTD3_CHECK_ARG(!tc || (a->params_uv && rtd3_td3_tf32_supported(h)), "tf32 needs params_uv and a 2 x 128 / 2 x 256 learner");
  RTD3_CHECK_ARG(tc || a->scratch, "the fp32 steps need the row scratch");
  cudaStream_t st = (cudaStream_t)stream;
  const int E = a->epochs, B = a->batch, delay = a->policy_update_delay;
  if (E == 0) return 0;
  const int n_actor = (E + delay - 1) / delay;
  RTD3_CUDA(cudaMemsetAsync(a->critic_losses, 0, sizeof(float) * 2 * (size_t)E, st));
  RTD3_CUDA(cudaMemsetAsync(a->actor_losses, 0, sizeof(float) * (size_t)n_actor, st));
  const ReplayView rp{(const float2*)a->rp_s, (const float2*)a->rp_a, a->rp_r, (const float2*)a->rp_s2, a->rp_notdone};
  Td3Hyper hp{a->gamma, a->policy_noise, a->noise_clip, a->max_action, (unsigned long long)a->noise_seed,
              (const unsigned long long*)a->noise_counter, 0ull};
  float* opt_grads = (a->world > 1 && a->p2p) ? a->p2p->sum : a->grads;      // what the optimiser consumes
  const float scale = 1.0f / (float)a->world;
  const int64_t off_c = h->ar.off(1), n_online = h->ar.online_total();
  // Single GPU, fp32 step kernels, batch <= 512 (no split weight-gradient pass): the optimiser - and on actor epochs the Polyak
  // blends - run inside the weight-gradient kernels; the critics' targets are blended right after the critics' Adam step of the
  // same epoch (the actor step in between reads neither the targets nor changes the critics: robot.py:278-285 gives the same values)
  // Data parallel over peer memory, same conditions: the weight-gradient kernels also exchange their gradient tiles with the peers
  // before they apply the optimiser (P2pFuse) - no all-reduce launch at all.  RTD3_P2P_FUSE: 2 (default) this form, 1 the all-reduce
  // kernel that applies the optimiser (p2p_allreduce_adam_kernel), 0 all-reduce and optimiser as two kernels (development)
  static const int p2p_fuse_env = getenv("RTD3_P2P_FUSE") ? atoi(getenv("RTD3_P2P_FUSE")) : 2;
  static const int p2p_mode_env = getenv("RTD3_P2P_MODE") ? atoi(getenv("RTD3_P2P_MODE")) : -1;   // development: force the exchange pattern
  const bool fuse_wg = a->world > 1 && a->p2p && p2p_fuse_env >= 2 && !tc && B <= 512 && 2 * wgrad_jobs(h->ar.critic) <= kP2pBlockFlags &&
                       wgrad_jobs(h->ar.actor) <= kP2pBlockFlags && a->p2p->slot_floats >= 2 * std::max(off_c, n_online - off_c);
  const bool fuse = (a->world == 1 || fuse_wg) && !tc && B <= 512;
  auto px_for = [&](bool actor) {
    P2pFuse px{};
    if (!fuse_wg) return px;
    px.prof = g_p2p_prof;
    for (int r = 0; r < a->world; ++r) {
      px.recv[r] = a->p2p->peer_recv[r];
    }
    px.mine = a->p2p->peer_recv[a->p2p->rank];
    px.world = a->world; px.rank = a->p2p->rank;
    px.seq_counter = (unsigned long long*)a->p2p->seq_counter; px.block_counter = a->p2p->block_counter;
    px.stride = a->p2p->slot_floats; px.slice_off = actor ? 0 : off_c; px.grad_scale = scale;
    px.mode = p2p_mode_env >= 0 ? p2p_mode_env : (a->world > 2 ? 1 : 0);
    return px;
  };
  const AdamState opt = adam_state(h, a);
  auto fuse_for = [&](bool actor, bool polyak) { return AdamFuse{opt, actor ? 0 : 1, polyak ? 1 : 0, (int)n_online, (int)h->ar.total()}; };
  // Data parallel over peer memory: the all-reduce kernel applies the optimiser to the sums it forms (one launch and one pass over the
  // arena less per optimiser step); RTD3_P2P_FUSE=0 keeps the two-kernel form (development)
  const bool fuse_p2p = a->world > 1 && a->p2p && p2p_fuse_env >= 1 && !fuse_wg;
  auto p2p_opt = [&](int nets, int polyak, int64_t off) { return P2pAdamArgs{opt, scale, nets, polyak, off}; };
  int64_t k = 0, ka = 0;
  int32_t rc = 0;
  for (int e = 0; e < E; ++e) {
    hp.noise_index = (unsigned long long)e;
    const float* nz = a->noise ? a->noise + (int64_t)e * B * 2 : nullptr;
    const int32_t* ix = a->idx + k * B;
    ++k;
    if (tc)
      rc = critic_step_tc_launch(h, a->params, a->params_uv, a->grads, rp, ix, nz, B, hp, a->critic_losses + 2 * e, nullptr, nullptr, a->steps,
                                 a->beta_pows, st);
    else
      rc = critic_step(h, a->params, a->params_t, a->grads, a->scratch, rp, ix, nz, B, hp, a->critic_losses + 2 * e, nullptr, nullptr, a->steps,
                       a->beta_pows, st, fuse ? fuse_for(false, e % delay == 0) : AdamFuse{}, px_for(false));
    if (rc) return rc;
    if (fuse_p2p) {
      if ((rc = p2p_allreduce_adam_launch(a->p2p, a->grads, n_online - off_c, p2p_opt(0b110, 0, off_c), st))) return rc;
    } else if (!fuse) {
      if ((rc = update_allreduce(a, off_c, n_online - off_c, st))) return rc;
      if ((rc = rtd3_td3_adam_polyak(h, a->params, a->params_t, a->params_uv, opt_grads, a->adam_m, a->adam_v, a->beta_pows, 0b110, a->lr_actor,
                                     a->lr_critic, scale, 0, a->tau, st)))
        return rc;
    }
    if (e % delay == 0) {
      const int32_t* ixa = a->idx + k * B;
      ++k;
      if (tc)
        rc = rtd3_td3_actor_step_tf32(h, a->params, a->params_uv, a->grads, a->rp_s, ixa, B, a->actor_losses + ka, a->steps, a->beta_pows, st);
      else
        rc = actor_step(h, a->params, a->params_t, a->grads, a->scratch, a->rp_s, ixa, B, a->actor_losses + ka, a->steps, a->beta_pows, st,
                        fuse ? fuse_for(true, true) : AdamFuse{}, px_for(true));
      ++ka;
      if (rc) return rc;
      if (fuse_p2p) {
        if ((rc = p2p_allreduce_adam_launch(a->p2p, a->grads, off_c, p2p_opt(0b001, 0b111, 0), st))) return rc;
      } else if (!fuse) {
        if ((rc = update_allreduce(a, 0, off_c, st))) return rc;
        if ((rc = rtd3_td3_adam_polyak(h, a->params, a->params_t, a->params_uv, opt_grads, a->adam_m, a->adam_v, a->beta_pows, 0b001, a->lr_actor,
                                       a->lr_critic, scale, 0b111, a->tau, st)))
          return rc;
      }
    }
  }
  if (!a->noise) return advance_noise_counter(a->noise_counter, (uint64_t)E, st);
  return 0;
}

/* development: copies the stage stamps of the last fused weight-gradient + peer-exchange launch ([256 blocks][2 threads][8 stages]
 * uint64 nanoseconds) to the host; returns 0 when RTD3_P2P_PROF=1 was not set */
int32_t rtd3_debug_p2p_prof(uint64_t* out_host) {
  if (!g_p2p_prof || !out_host) return 0;
  RTD3_CUDA(cudaMemcpy(out_host, g_p2p_prof, kP2pBlockFlags * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return 1;
}

}  // extern "C"
