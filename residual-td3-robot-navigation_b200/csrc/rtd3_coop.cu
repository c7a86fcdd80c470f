// Small-batch residual-TD3 learner as ONE persistent cooperative kernel per update (robot.py:258-398; SURVEY.md 7 step 5a).
//
// Why: at B <= 512 a critic / actor step is a chain of small dense layers.  The row-tiled kernels of rtd3_td3.cu give every CTA a
// few batch rows and make it stream the weights of five networks from L2 (240 MB per critic step against 3.2 MB of parameters,
// VERDICT r1) in four launches per step.  Here one CTA per SM stays resident for the whole update, every H x H product is cut into
// 32 x 64 (or 32 x 32) output tiles over ALL SMs - a tile reads its 32 activation rows and 64 weight columns once, 6 MB per product
// instead of 33 MB - and the layers of the chain are separated by grid-wide barriers instead of kernel boundaries.  The optimiser and
// the Polyak updates are stages of the same kernel, and so is the gradient all-reduce of the data-parallel learner: every CTA pushes
// its slice of the gradients into the peers' receive slots over NVLink, one flag hop, and the Adam stage sums the slots in rank
// order (the protocol of rtd3_p2p.cu, without a kernel of its own).
//
// Stage plan of a critic step (L hidden layers; "|" = grid barrier):
//   fwd layer 1..L-1 of {target actor(s2), critic1(s,a), critic2(s,a)}   [first layer generated on the fly from the replay rows]
//   | a' = clip(target actor out + clip(noise))                                                     (robot.py:338-339)
//   | fwd layer 1..L-1 of {target critic1, target critic2}(s2, a')
//   | y = r + gamma min(Q1', Q2') notdone; Q_i; loss_i; dout_i                                      (robot.py:342-353)
//   | per hidden layer, top down: dX and dW products of both critics (+ output-layer gradients)
//   | first-layer gradients | [push to peers |] Adam on both critics                                (robot.py:356-363)
// and of an actor step: actor fwd | a = actor out | critic1 fwd | critic1 dX (dout = -1/B) | dQ/da | actor dX + dW | first-layer
// gradients | [push |] Adam on the actor + the three Polyak updates (robot.py:369-398, 283-285).
//
// Everything another CTA produced inside the launch (activations, gradients, the parameters themselves) is read through L2
// (ld.global.cg / cp.async.cg): L1 is not coherent across SMs.
#include <algorithm>

#include "rtd3_common.cuh"
#include "rtd3_mlp.cuh"
#include "rtd3_td3.cuh"

namespace rtd3 {

constexpr int kCT = 256;                 // threads per CTA
constexpr int CTM = 32, CTK = 256;       // tile rows; reduction PANEL: the whole K of a hidden layer (<= 256) is staged at once
constexpr int kAld = CTK + 4;            // row stride of the A tile in shared memory (16 B aligned rows, skewed banks)
constexpr int kCoopMaxWorld = RTD3_P2P_MAX_WORLD;

__device__ __forceinline__ float ldcg(const float* p) { return __ldcg(p); }
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gsrc, bool valid) {
  const int bytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes) : "memory");
}

// ---- grid barrier (all CTAs are co-resident: cooperative launch) ---------------------------------------------------------------
// Arrival: one counter.  Release: kBarLines generation words in DIFFERENT 128 B lines; CTA b polls line b % kBarLines with a back-off.
// (With every idle CTA polling ONE word in a tight loop, the L2 slice that owns it saturates - a hundred pollers against a slice
// that serves about one request per clock - and every load of the working CTAs that maps to that slice queues behind them: all
// stages of the kernel ran ~4x slower than their instruction counts explain, ncu r2a.)
constexpr int kBarLines = 16;
constexpr int kBarWords = 32 * (1 + kBarLines);          // floats of scratch header: counter line + generation lines
struct GridBarrier {
  unsigned int* count;
  volatile unsigned int* gen;                            // gen[32 * g], g < kBarLines
};
__device__ int g_prof_slot;
__device__ long long* g_tile_prof;          // development: phase stamps of block 0's tiles (second half of the prof buffer)
__device__ int g_tile_slot;
__device__ __forceinline__ void tile_stamp() {
  if (g_tile_prof && blockIdx.x == 0 && threadIdx.x == 0) {
    long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    const int s = g_tile_slot;
    if (s < 120) { g_tile_prof[s] = now; g_tile_slot = s + 1; }
  }
}
__device__ __forceinline__ void prof_stamp(long long* prof) {
  long long now;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
  const int s = g_prof_slot;
  if (s < 126) { prof[s] = now; g_prof_slot = s + 1; }
}
__device__ __forceinline__ void grid_sync(const GridBarrier& b, long long* prof = nullptr) {
  __syncthreads();
  if (threadIdx.x == 0) {
    if (prof && blockIdx.x == 0) prof_stamp(prof);       // block 0 ARRIVES: its own work of the stage is done
    volatile unsigned int* mine = b.gen + 32 * (blockIdx.x % kBarLines);
    const unsigned int g = *mine;
    __threadfence();
    if (atomicAdd(b.count, 1u) == gridDim.x - 1) {
      *b.count = 0u;
      __threadfence();
#pragma unroll
      for (int l = 0; l < kBarLines; ++l) b.gen[32 * l] = g + 1u;
    } else {
      while (*mine == g) __nanosleep(32);
    }
    __threadfence();
    if (prof && blockIdx.x == 0) prof_stamp(prof);       // ... and is released
  }
  __syncthreads();
}

// ---- arguments -----------------------------------------------------------------------------------------------------------------
struct CoopPeers {
  float* recv[kCoopMaxWorld];
  unsigned long long* flags[kCoopMaxWorld];
};

struct CoopArgs {
  long long* prof;           // nullable (development): block 0 stamps %globaltimer at every stage boundary of the last epoch
  AdamState adam;            // adam.params_uv is not used: this kernel keeps no tensor-core copies
  float* grads;
  int32_t* steps;
  ReplayView rp;
  const int32_t* idx;
  const float* noise;        // nullable [E][B][2]
  Td3Hyper hp;
  int B, E, delay;
  float* critic_losses;      // [E][2]
  float* actor_losses;       // [ceil(E/delay)]
  float* scratch;            // coop_scratch_floats()
  GridBarrier bar;
  // data parallel (world > 1): peer-memory all-reduce inside the kernel
  int world, rank;
  CoopPeers peers;
  unsigned long long* seq_counter;
  long long slot_floats;
};

// Activation slots: 0 target actor / actor, 1 target critic 1 / critic 1 (actor step), 2 target critic 2, 3 critic 1, 4 critic 2.
// Per slot: H_l [B][Hd] for l = 0..L-1, dZ_l [B][Hd] for l = 0..L-2 (the top one is generated from dout), then small per-row arrays.
struct Scratch {
  float* base;
  int Bp, Hd, L;
  __host__ __device__ int64_t slot_floats() const { return (int64_t)(2 * L - 1) * Bp * Hd; }
  __host__ __device__ float* H(int slot, int l) const { return base + slot * slot_floats() + (int64_t)l * Bp * Hd; }
  __host__ __device__ float* dZ(int slot, int l) const { return base + slot * slot_floats() + (int64_t)(L + l) * Bp * Hd; }
  __host__ __device__ float* small_base() const { return base + 5 * slot_floats(); }
  __host__ __device__ float* in4(int slot) const { return small_base() + (int64_t)slot * Bp * 4; }          // net input rows [B][4]
  __host__ __device__ float* dout(int slot) const { return small_base() + (int64_t)(5 + slot) * Bp * 4; }   // [B][2] (stride 2)
  __host__ __device__ float* rowval(int k) const { return small_base() + (int64_t)40 * Bp + (int64_t)k * Bp; }   // k < 8: per-row scalars
  __host__ __device__ static int64_t floats(int B, int Hd, int L) {
    const int64_t Bp = (B + 31) / 32 * 32;
    return 5 * (int64_t)(2 * L - 1) * Bp * Hd + 48 * Bp;
  }
};

// ---- one output tile of C = A * B ------------------------------------------------------------------------------------------------
// A [M][Kred]: loaded (A_GLOBAL), generated from the net input and the first layer (A_GEN_FIRST), generated from dout and the
// output layer (A_GEN_DOUT: the gradient w.r.t. the last hidden layer's pre-activation), or the TRANSPOSE of such a [Kred][M] array
// (AT_GLOBAL / AT_GEN_DOUT: weight gradients, whose reduction runs over the batch).  B [Kred][N] row-major, always loaded.
enum { A_GLOBAL = 0, A_GEN_FIRST, A_GEN_DOUT, AT_GLOBAL, AT_GEN_DOUT };
enum { E_RELU_BIAS = 0, E_MASK, E_GRAD };

struct TileOp {
  int akind, ekind;
  int M, N, Kred;
  const float* A; int lda;
  const float* Bm; int ldb;
  // generators
  const float* gen_in;        // [rows][4] net input (A_GEN_FIRST)
  const float* W0; const float* b0; int in_dim;
  float* H0_store;            // nullable: the generated first-layer output goes here as well (n-tile 0 stores it)
  const float* Hmask;         // [rows][Hd] output of the last hidden layer (A*_GEN_DOUT)
  const float* dout;          // [rows][2]
  const float* Wout; int out_dim; int Hd;
  // epilogue
  const float* bias;          // E_RELU_BIAS
  const float* mask_src; int ldmask;   // E_MASK: C = mask_src > 0 ? acc : 0
  float* C; int ldc;
  float* bias_grad;           // E_GRAD, nullable: row sums of A (n-tile 0 writes them)
};

// B panel: rows k0..k0+kload-1 of B [Kred][N], columns n0..n0+TN-1 -> Bs[kk][TN]  (bulk of the tile's traffic: cp.async, L2 only)
template <int TN>
__device__ __forceinline__ void load_b_panel(const TileOp& op, float* Bs, int k0, int kload, int n0) {
  const int F4 = kload * (TN / 4);
  for (int q = threadIdx.x; q < F4; q += kCT) {
    const int kk = q / (TN / 4), nq = q - kk * (TN / 4);
    const int k = k0 + kk, n = n0 + nq * 4;
    const bool ok = k < op.Kred && n < op.N;
    cp_async16_zfill(Bs + kk * TN + nq * 4, op.Bm + (int64_t)(ok ? k : 0) * op.ldb + (ok ? n : 0), ok);
  }
}

// A panel: rows m0..m0+31, reduction k0..k0+kload-1 -> As[r][kk]
__device__ __forceinline__ void load_a_panel(const TileOp& op, float* As, const float* in_s, const float* w_s, int m0, int k0, int kload) {
  const int kq_n = kload >> 2;                           // float4 per row
  if (op.akind == A_GLOBAL) {
    for (int q = threadIdx.x; q < CTM * kq_n; q += kCT) {
      const int r = q / kq_n, kq = q - r * kq_n;
      const int m = m0 + r, k = k0 + kq * 4;
      const bool ok = m < op.M && k < op.Kred;
      cp_async16_zfill(As + r * kAld + kq * 4, op.A + (int64_t)(ok ? m : 0) * op.lda + (ok ? k : 0), ok);
    }
  } else if (op.akind == A_GEN_FIRST) {
    // h0[m][k] = relu(b0[k] + sum_j in[m][j] W0[k][j]); 4 consecutive k of one row per item
    for (int q = threadIdx.x; q < CTM * kq_n; q += kCT) {
      const int r = q / kq_n, kq = q - r * kq_n;
      const int m = m0 + r;
      float vv[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int k = k0 + kq * 4 + i;
        if (m < op.M && k < op.Kred) {
          float s = w_s[4 * kMaxHidden + k];
          for (int j = 0; j < op.in_dim; ++j) s = fmaf(in_s[r * 4 + j], w_s[k * op.in_dim + j], s);
          vv[i] = fmaxf(s, 0.f);
        }
      }
      const float4 v = make_float4(vv[0], vv[1], vv[2], vv[3]);
      *reinterpret_cast<float4*>(As + r * kAld + kq * 4) = v;
      if (op.H0_store && m < op.M && k0 + kq * 4 < op.Kred) *reinterpret_cast<float4*>(op.H0_store + (int64_t)m * op.Hd + k0 + kq * 4) = v;
    }
  } else if (op.akind == A_GEN_DOUT) {
    // dz[m][k] = h[m][k] > 0 ? sum_o dout[m][o] Wout[o][k] : 0     (in_s holds dout of the tile's rows)
    for (int q = threadIdx.x; q < CTM * kq_n; q += kCT) {
      const int r = q / kq_n, kq = q - r * kq_n;
      const int m = m0 + r, k = k0 + kq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m < op.M && k < op.Kred) {
        const float4 h = ldcg4(op.Hmask + (int64_t)m * op.Hd + k);
        const float4 w0 = *reinterpret_cast<const float4*>(w_s + k);
        float4 w1 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (op.out_dim > 1) w1 = *reinterpret_cast<const float4*>(w_s + op.Hd + k);
        const float d0 = in_s[r * 4], d1 = in_s[r * 4 + 1];
        v.x = h.x > 0.f ? fmaf(d0, w0.x, d1 * w1.x) : 0.f;
        v.y = h.y > 0.f ? fmaf(d0, w0.y, d1 * w1.y) : 0.f;
        v.z = h.z > 0.f ? fmaf(d0, w0.z, d1 * w1.z) : 0.f;
        v.w = h.w > 0.f ? fmaf(d0, w0.w, d1 * w1.w) : 0.f;
      }
      *reinterpret_cast<float4*>(As + r * kAld + kq * 4) = v;
    }
  } else {
    // transposed: As[r = output row (a hidden unit n)][kk = batch row]; source [batch][Hd], 4 consecutive units of one batch row per item
    for (int q = threadIdx.x; q < kload * (CTM / 4); q += kCT) {
      const int bb = q >> 3, nq = q & 7;                 // CTM / 4 == 8 float4 of units per batch row
      const int b = k0 + bb, n = m0 + nq * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (b < op.Kred && n < op.M) {
        if (op.akind == AT_GLOBAL) {
          v = ldcg4(op.A + (int64_t)b * op.lda + n);
        } else {
          const float4 h = ldcg4(op.Hmask + (int64_t)b * op.Hd + n);
          const float4 w0 = *reinterpret_cast<const float4*>(w_s + n);
          float4 w1 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (op.out_dim > 1) w1 = *reinterpret_cast<const float4*>(w_s + op.Hd + n);
          const float d0 = ldcg(op.dout + (int64_t)b * 2), d1 = ldcg(op.dout + (int64_t)b * 2 + 1);
          v.x = h.x > 0.f ? fmaf(d0, w0.x, d1 * w1.x) : 0.f;
          v.y = h.y > 0.f ? fmaf(d0, w0.y, d1 * w1.y) : 0.f;
          v.z = h.z > 0.f ? fmaf(d0, w0.z, d1 * w1.z) : 0.f;
          v.w = h.w > 0.f ? fmaf(d0, w0.w, d1 * w1.w) : 0.f;
        }
      }
      As[(nq * 4 + 0) * kAld + bb] = v.x;
      As[(nq * 4 + 1) * kAld + bb] = v.y;
      As[(nq * 4 + 2) * kAld + bb] = v.z;
      As[(nq * 4 + 3) * kAld + bb] = v.w;
    }
  }
}

// (not inlined: the stages call it from a dozen places, and a fully inlined kernel was 560 KB of SASS)
template <int TN>
__device__ __noinline__ void gemm_tile(const TileOp& op_in, int tm, int tn, float* smem) {
  constexpr int NT = TN / 16;                            // outputs per thread along n (4 or 2)
  float* As = smem;                                      // [CTM][kAld]
  float* Bs = smem + CTM * kAld;                         // [CTK][64]
  float* in_s = Bs + CTK * 64;                           // [CTM][4]
  float* w_s = in_s + CTM * 4;                           // [5][kMaxHidden]: first layer (W0 | b0) or output layer weights of the generators
  const TileOp& op = op_in;                              // lives in shared memory (see stage_ops)
  const int t = threadIdx.x, ty = t >> 4, tx = t & 15;
  tile_stamp();
  __syncthreads();                                       // the previous tile's readers are done with the shared buffers
  const int m0 = tm * CTM, n0 = tn * TN;
  float acc[2][NT];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < NT; ++j) acc[i][j] = 0.f;
  float my_rsum = 0.f;
  const bool want_rsum = op.ekind == E_GRAD && op.bias_grad && tn == 0;

  if (op.akind == A_GEN_FIRST) {
    if (t < CTM * 4) {
      const int r = t >> 2, j = t & 3;
      in_s[t] = (m0 + r < op.M && j < op.in_dim) ? ldcg(op.gen_in + (int64_t)(m0 + r) * 4 + j) : 0.f;
    }
    for (int q = t; q < op.Hd * op.in_dim; q += kCT) w_s[q] = ldcg(op.W0 + q);          // W0 [Hd][in]
    for (int q = t; q < op.Hd; q += kCT) w_s[4 * kMaxHidden + q] = ldcg(op.b0 + q);
  } else if (op.akind == A_GEN_DOUT || op.akind == AT_GEN_DOUT) {
    if (op.akind == A_GEN_DOUT && t < CTM * 2) {
      const int r = t >> 1, o = t & 1;
      in_s[r * 4 + o] = (m0 + r < op.M) ? ldcg(op.dout + (int64_t)(m0 + r) * 2 + o) : 0.f;
    }
    for (int q = t; q < op.Hd * op.out_dim; q += kCT) w_s[q] = ldcg(op.Wout + q);        // Wout [out][Hd]
  }
  __syncthreads();

  // The whole reduction range of a hidden layer (K <= 256) is staged in ONE go - one L2 round trip per tile instead of one per
  // 32-wide chunk (the tile is a chain of dependent L2 accesses otherwise: with eight chunks it took 15-19 us, stage stamps r2) -
  // and weight gradients, whose reduction runs over the batch, walk it in panels of 256 rows.
  for (int k0 = 0; k0 < op.Kred; k0 += CTK) {
    const int kp = min(CTK, op.Kred - k0);
    const int kload = (kp + 31) & ~31;                   // zero-filled up to a multiple of 32
    if (k0 > 0) __syncthreads();                         // the previous panel's readers are done
    tile_stamp();
    load_b_panel<TN>(op, Bs, k0, kload, n0);
    tile_stamp();
    load_a_panel(op, As, in_s, w_s, m0, k0, kload);
    tile_stamp();
    cp_commit();
    cp_wait<0>();
    __syncthreads();
    tile_stamp();
#pragma unroll 2
    for (int kk = 0; kk < kload; kk += 4) {
      const float4 a0 = *reinterpret_cast<const float4*>(As + ty * kAld + kk);
      const float4 a1 = *reinterpret_cast<const float4*>(As + (ty + 16) * kAld + kk);
      const float av0[4] = {a0.x, a0.y, a0.z, a0.w}, av1[4] = {a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float bv[NT];
        if (NT == 4) {
          const float4 q = *reinterpret_cast<const float4*>(Bs + (kk + i) * TN + tx * 4);
          bv[0] = q.x; bv[1] = q.y; bv[2] = q.z; bv[NT - 1] = q.w;
        } else {
          const float2 q = *reinterpret_cast<const float2*>(Bs + (kk + i) * TN + tx * 2);
          bv[0] = q.x; bv[1] = q.y;
        }
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          acc[0][j] = fmaf(av0[i], bv[j], acc[0][j]);
          acc[1][j] = fmaf(av1[i], bv[j], acc[1][j]);
        }
      }
    }
    if (want_rsum && t < CTM) {
#pragma unroll 8
      for (int kk = 0; kk < kload; ++kk) my_rsum += As[t * kAld + kk];
    }
  }

  tile_stamp();
  // epilogue
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int m = m0 + ty + 16 * i;
    if (m >= op.M) continue;
    const int n = n0 + tx * NT;
    if (n >= op.N) continue;
    float v[NT];
#pragma unroll
    for (int j = 0; j < NT; ++j) v[j] = acc[i][j];
    if (op.ekind == E_RELU_BIAS) {
#pragma unroll
      for (int j = 0; j < NT; ++j) v[j] = fmaxf(v[j] + ldcg(op.bias + n + j), 0.f);
    } else if (op.ekind == E_MASK) {
#pragma unroll
      for (int j = 0; j < NT; ++j) v[j] = ldcg(op.mask_src + (int64_t)m * op.ldmask + n + j) > 0.f ? v[j] : 0.f;
    }
    float* dst = op.C + (int64_t)m * op.ldc + n;
    if (NT == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[NT - 1]);
    else *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
  }
  if (want_rsum && t < CTM && m0 + t < op.M) op.bias_grad[m0 + t] = my_rsum;
  tile_stamp();
}

// ---- operation builders -----------------------------------------------------------------------------------------------------------
struct NetRef {
  NetShape s;
  const float* P;      // torch-layout parameters
  const float* Pt;     // transposed hidden weights
  float* G;            // gradient slot (trained nets)
  int slot;            // activation slot
};

__device__ __forceinline__ NetRef net_ref(const CoopArgs& a, int net, int slot) {
  NetRef r;
  r.s = (net == 0 || net == 3) ? a.adam.ar.actor : a.adam.ar.critic;
  r.P = a.adam.params + a.adam.ar.off(net);
  r.Pt = a.adam.params_t + a.adam.ar.off(net);
  r.G = net < 3 ? a.grads + a.adam.ar.off(net) : nullptr;
  r.slot = slot;
  return r;
}

// forward of hidden layer l (1..L-1): H_l = relu(H_{l-1} Wt_l + b_l)
__device__ __forceinline__ TileOp fwd_op(const CoopArgs& a, const Scratch& sc, const NetRef& nr, int l, bool keep_h0) {
  TileOp op{};
  const int Hd = nr.s.hid;
  op.ekind = E_RELU_BIAS;
  op.M = a.B; op.N = Hd; op.Kred = Hd; op.Hd = Hd;
  op.Bm = nr.Pt + net_w_off(nr.s, l); op.ldb = Hd;
  op.bias = nr.P + net_b_off(nr.s, l);
  op.C = sc.H(nr.slot, l); op.ldc = Hd;
  if (l == 1) {
    op.akind = A_GEN_FIRST;
    op.gen_in = sc.in4(nr.slot);
    op.W0 = nr.P + net_w_off(nr.s, 0); op.b0 = nr.P + net_b_off(nr.s, 0); op.in_dim = nr.s.in;
    op.H0_store = keep_h0 ? sc.H(nr.slot, 0) : nullptr;
  } else {
    op.akind = A_GLOBAL;
    op.A = sc.H(nr.slot, l - 1); op.lda = Hd;
  }
  return op;
}

// input gradient through hidden layer l (L-1..1): dZ_{l-1} = relu'(H_{l-1}) * (dZ_l W_l)
__device__ __forceinline__ TileOp dx_op(const CoopArgs& a, const Scratch& sc, const NetRef& nr, int l) {
  TileOp op{};
  const int Hd = nr.s.hid, L = nr.s.layers;
  op.ekind = E_MASK;
  op.M = a.B; op.N = Hd; op.Kred = Hd; op.Hd = Hd;
  op.Bm = nr.P + net_w_off(nr.s, l); op.ldb = Hd;                    // W_l [n][k]: reduction index n is the row
  op.mask_src = sc.H(nr.slot, l - 1); op.ldmask = Hd;
  op.C = sc.dZ(nr.slot, l - 1); op.ldc = Hd;
  if (l == L - 1) {
    op.akind = A_GEN_DOUT;
    op.Hmask = sc.H(nr.slot, L - 1); op.dout = sc.dout(nr.slot);
    op.Wout = nr.P + net_w_off(nr.s, L); op.out_dim = nr.s.out;
  } else {
    op.akind = A_GLOBAL;
    op.A = sc.dZ(nr.slot, l); op.lda = Hd;
  }
  return op;
}

// weight gradient of hidden layer l (1..L-1): gW_l[n][k] = sum_b dZ_l[b][n] H_{l-1}[b][k]; gb_l[n] = sum_b dZ_l[b][n]
__device__ __forceinline__ TileOp dw_op(const CoopArgs& a, const Scratch& sc, const NetRef& nr, int l) {
  TileOp op{};
  const int Hd = nr.s.hid, L = nr.s.layers;
  op.ekind = E_GRAD;
  op.M = Hd; op.N = Hd; op.Kred = a.B; op.Hd = Hd;
  op.Bm = sc.H(nr.slot, l - 1); op.ldb = Hd;
  op.C = nr.G + net_w_off(nr.s, l); op.ldc = Hd;
  op.bias_grad = nr.G + net_b_off(nr.s, l);
  if (l == L - 1) {
    op.akind = AT_GEN_DOUT;
    op.Hmask = sc.H(nr.slot, L - 1); op.dout = sc.dout(nr.slot);
    op.Wout = nr.P + net_w_off(nr.s, L); op.out_dim = nr.s.out;
  } else {
    op.akind = AT_GLOBAL;
    op.A = sc.dZ(nr.slot, l); op.lda = Hd;
  }
  return op;
}

__device__ __forceinline__ int tiles_of(const TileOp& op, int TN) { return ((op.M + CTM - 1) / CTM) * ((op.N + TN - 1) / TN); }

// Run `nops` tile operations as one stage: the tiles of all of them are dealt round-robin to the CTAs.  Narrow tiles when the wide
// ones would leave most SMs idle.
__device__ __noinline__ void run_gemm_stage(const TileOp* ops, int nops, float* smem) {
  int total64 = 0;
  for (int i = 0; i < nops; ++i) total64 += tiles_of(ops[i], 64);
  const bool narrow = 2 * total64 <= (int)gridDim.x;
  const int TN = narrow ? 32 : 64;
  int total = 0;
  for (int i = 0; i < nops; ++i) total += tiles_of(ops[i], TN);
  for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
    int rem = tile, i = 0;
    while (rem >= tiles_of(ops[i], TN)) { rem -= tiles_of(ops[i], TN); ++i; }
    const int ntn = (ops[i].N + TN - 1) / TN;
    const int tm = rem / ntn, tn = rem - tm * ntn;
    if (narrow) gemm_tile<32>(ops[i], tm, tn, smem);
    else gemm_tile<64>(ops[i], tm, tn, smem);
  }
}

// ---- small stages -----------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int global_warp() { return (int)blockIdx.x * (kCT / 32) + (int)(threadIdx.x >> 5); }
__device__ __forceinline__ int total_warps() { return (int)gridDim.x * (kCT / 32); }

// out[o] = bout[o] + sum_k H[row][k] Wout[o][k]   (one warp; float4 per lane, all loads of the row issued before the first use)
__device__ __forceinline__ void out_layer_row(const NetRef& nr, const float* __restrict__ Hrow, float& o0, float& o1) {
  const int Hd = nr.s.hid, lane = threadIdx.x & 31;
  const float* W = nr.P + net_w_off(nr.s, nr.s.layers);
  const bool two = nr.s.out > 1;
  float4 h[2], w0[2], w1[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {                          // Hd <= 256: at most two float4 per lane
    const int k = (u * 32 + lane) * 4;
    const bool ok = k < Hd;
    h[u] = ok ? ldcg4(Hrow + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    w0[u] = ok ? ldcg4(W + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    w1[u] = (ok && two) ? ldcg4(W + Hd + k) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  float v0 = 0.f, v1 = 0.f;
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    v0 = fmaf(h[u].x, w0[u].x, v0); v0 = fmaf(h[u].y, w0[u].y, v0); v0 = fmaf(h[u].z, w0[u].z, v0); v0 = fmaf(h[u].w, w0[u].w, v0);
    v1 = fmaf(h[u].x, w1[u].x, v1); v1 = fmaf(h[u].y, w1[u].y, v1); v1 = fmaf(h[u].z, w1[u].z, v1); v1 = fmaf(h[u].w, w1[u].w, v1);
  }
  v0 = warp_sum(v0);
  v1 = warp_sum(v1);
  const float* bo = nr.P + net_b_off(nr.s, nr.s.layers);
  o0 = v0 + ldcg(bo);
  o1 = two ? v1 + ldcg(bo + 1) : 0.f;
}

// Batch reductions of the small gradients, one job = one network x 32 consecutive hidden units, dealt to the CTAs from
// `first_block` on: the 8 warps of a CTA take every 8th batch row (lanes = the 32 units: one coalesced 128 B load per row, eight
// rows in flight per warp), the partial sums meet in shared memory.
//   kind 0: gWout[o][k] = sum_b dout[b][o] H_{L-1}[b][k], gbout[o] = sum_b dout[b][o]
//   kind 1: gW0[n][j]   = sum_b dZ0[b][n] in[b][j],        gb0[n]   = sum_b dZ0[b][n]
__device__ __noinline__ void small_grads(const CoopArgs& a, const Scratch& sc, const NetRef* nets, int nnets, int kind, int first_block, float* smem) {
  const int Hd = nets[0].s.hid;
  const int nch = (Hd + 31) / 32;
  const int jobs = nnets * nch;
  const int nb = (int)gridDim.x;
  const int vb = ((int)blockIdx.x - first_block % nb + nb) % nb;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* red = smem;                                     // [8 warps][32 lanes][6]
  for (int job = vb; job < jobs; job += nb) {
    const int ni = job / nch, u = (job - ni * nch) * 32 + lane;     // this lane's hidden unit
    const NetRef& nr = nets[ni];
    const float* X = kind == 0 ? sc.H(nr.slot, nr.s.layers - 1) : sc.dZ(nr.slot, 0);
    const float* d = sc.dout(nr.slot);
    const float* in = sc.in4(nr.slot);
    float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    __syncthreads();                                     // the previous job's / stage's readers of `red` are done
#pragma unroll 8
    for (int b = warp; b < a.B; b += 8) {
      const float x = u < Hd ? ldcg(X + (int64_t)b * Hd + u) : 0.f;
      if (kind == 0) {
        const float d0 = ldcg(d + 2 * b), d1 = ldcg(d + 2 * b + 1);
        acc[0] = fmaf(d0, x, acc[0]); acc[1] = fmaf(d1, x, acc[1]);
        acc[2] += d0; acc[3] += d1;
      } else {
        const float4 q = ldcg4(in + (int64_t)b * 4);
        acc[0] = fmaf(x, q.x, acc[0]); acc[1] = fmaf(x, q.y, acc[1]); acc[2] = fmaf(x, q.z, acc[2]); acc[3] = fmaf(x, q.w, acc[3]);
        acc[4] += x;
      }
    }
#pragma unroll
    for (int q = 0; q < 6; ++q) red[(warp * 32 + lane) * 6 + q] = acc[q];
    __syncthreads();
    if (warp == 0 && u < Hd) {
      float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int w = 0; w < 8; ++w)
#pragma unroll
        for (int q = 0; q < 6; ++q) v[q] += red[(w * 32 + lane) * 6 + q];
      if (kind == 0) {
        float* gw = nr.G + net_w_off(nr.s, nr.s.layers);
        gw[u] = v[0];
        if (nr.s.out > 1) gw[Hd + u] = v[1];
        if (u == 0) {
          float* gb = nr.G + net_b_off(nr.s, nr.s.layers);
          gb[0] = v[2];
          if (nr.s.out > 1) gb[1] = v[3];
        }
      } else {
        nr.G[net_b_off(nr.s, 0) + u] = v[4];
        for (int jj = 0; jj < nr.s.in; ++jj) nr.G[net_w_off(nr.s, 0) + u * nr.s.in + jj] = v[jj];
      }
    }
  }
  __syncthreads();
}

// The one-hidden-layer case has no dZ_0 array (the top gradient is generated): L >= 2 is required by the launcher.

__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ float ld_volatile_f32(const float* p) {
  float v;
  asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// Adam (torch defaults, robot.py:237-239) on the nets of `nets` (bit 0 actor, 1 critic1, 2 critic2), then Polyak on `polyak`.
// World > 1: the gradients are first pushed to every rank's receive slot, one flag per rank is raised after a grid barrier, and the
// optimiser sums the `world` slots of this rank's area in rank order (bit-identical replicas).
__device__ __noinline__ void adam_stage(const CoopArgs& a, int nets, int polyak, unsigned long long seq) {
  AdamState os = a.adam;
  os.params_uv = nullptr;            // the tensor-core copies are not kept (learner.py marks them stale after a cooperative update)
  const int n_online = (int)os.ar.online_total();
  const int off1 = (int)os.ar.off(1), off2 = (int)os.ar.off(2);
  const int lo = (nets & 1) ? 0 : off1, hi = (nets & 6) ? n_online : off1;      // range of gradients this step produced
  const int gtid = (int)blockIdx.x * kCT + (int)threadIdx.x, gthreads = (int)gridDim.x * kCT;
  const float* slots = nullptr;
  if (a.world > 1) {
    const long long slot = ((long long)(seq & 1ull) * a.world + a.rank) * a.slot_floats;
    for (int i = lo + gtid; i < hi; i += gthreads) {
      const float g = ldcg(a.grads + i);
      for (int q = 0; q < a.world; ++q) a.peers.recv[q][slot + i] = g;
    }
    __threadfence_system();
    grid_sync(a.bar);
    if (blockIdx.x == 0 && (int)threadIdx.x < a.world) {
      __threadfence_system();
      st_release_sys_u64(a.peers.flags[threadIdx.x] + a.rank, seq);
    }
    if ((int)threadIdx.x < a.world) {
      const unsigned long long* f = a.peers.flags[a.rank] + threadIdx.x;
      unsigned long long t0 = 0;
      while (ld_acquire_sys_u64(f) < seq) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
        if (!t0) t0 = now;
        if (now - t0 > 20ull * 1000 * 1000 * 1000) asm volatile("trap;");
      }
    }
    __syncthreads();
    slots = a.peers.recv[a.rank] + (long long)(seq & 1ull) * a.world * a.slot_floats;
  }
  __shared__ float s_step[2], s_bc2[2];
  if (threadIdx.x < 2) {
    const AdamStep k = adam_step(threadIdx.x == 0 ? os.lr[0] : os.lr[1], os.beta_pows[2 * threadIdx.x], os.beta_pows[2 * threadIdx.x + 1]);
    s_step[threadIdx.x] = k.step;
    s_bc2[threadIdx.x] = k.sqrt_bc2;
  }
  __syncthreads();
  const float scale = 1.0f / (float)a.world;
  for (int i = gtid; i < n_online; i += gthreads) {
    const int net = i < off1 ? 0 : (i < off2 ? 1 : 2);
    const bool do_adam = (nets >> net) & 1, do_polyak = (polyak >> net) & 1;
    if (!do_adam && !do_polyak) continue;
    const int noff = net == 0 ? 0 : (net == 1 ? off1 : off2);
    const NetShape s = net == 0 ? os.ar.actor : os.ar.critic;
    if (i - noff >= (int)net_param_count(s)) continue;                        // slot padding
    const float p = ldcg(os.params + i);
    float g = 0.f, m = 0.f, v = 0.f, t = 0.f;
    if (do_adam) {
      if (a.world > 1) {
        for (int r = 0; r < a.world; ++r) g += ld_volatile_f32(slots + (long long)r * a.slot_floats + i);
      } else {
        g = ldcg(a.grads + i);
      }
      g *= scale;
      m = os.m[i];
      v = os.v[i];
    }
    if (do_polyak) t = ldcg(os.params + n_online + i);
    const int o = net == 0 ? 0 : 1;
    adam_polyak1(os, i, noff, copy_index(s, i - noff), g, m, v, p, t, AdamStep{s_step[o], s_bc2[o]}, do_adam, do_polyak, n_online,
                 (int)os.ar.total());
  }
}

// deterministic sum of a per-row array (block 0, warp 0)
__device__ __forceinline__ void reduce_rows_to(const float* rows, int B, float* out) {
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += 32) s += ldcg(rows + b);
    s = warp_sum(s);
    if (threadIdx.x == 0) *out = s;
  }
}

// ---- the kernel ---------------------------------------------------------------------------------------------------------------------
// The tile operations of the current stage.  Built by ONE thread into shared memory: as per-thread local arrays they cost every
// thread of every CTA ~100 local stores per stage (30 MB of L2 write traffic per stage over the grid - it made every stage, and
// every L2 access of the kernel, several times slower; ncu r2a: 554 k local store instructions for two epochs).
__shared__ TileOp s_ops[4];
__shared__ NetRef s_nets[2];

__global__ void __launch_bounds__(kCT, 1) td3_update_coop_kernel(CoopArgs a) {
  extern __shared__ __align__(16) float coop_smem[];
  const Scratch sc{a.scratch, (a.B + 31) / 32 * 32, a.adam.ar.critic.hid, a.adam.ar.critic.layers};
  const int L = a.adam.ar.critic.layers, B = a.B;
  const int lane = threadIdx.x & 31;
  unsigned long long seq = a.world > 1 ? *reinterpret_cast<volatile unsigned long long*>(a.seq_counter) : 0ull;
  int k_idx = 0, ka = 0;

  if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) { g_prof_slot = 0; g_tile_slot = 0; g_tile_prof = nullptr; }
  for (int e = 0; e < a.E; ++e) {
    long long* prof = (e == a.E - 1) ? a.prof : nullptr;
    if (prof && blockIdx.x == 0 && threadIdx.x == 0) g_tile_prof = a.prof + 128;
    // =============================================================== critic step (robot.py:312-366)
    {
      const int32_t* idx = a.idx + (int64_t)k_idx * B;
      ++k_idx;
      const NetRef ta = net_ref(a, 3, 0), tc1 = net_ref(a, 4, 1), tc2 = net_ref(a, 5, 2), c1 = net_ref(a, 1, 3), c2 = net_ref(a, 2, 4);
      if (blockIdx.x == 0 && threadIdx.x == 0) advance_adam_clock(a.steps, a.adam.beta_pows, 1);
      // gather: net inputs of the target actor (s2) and of both critics (s, a)
      for (int b = (int)blockIdx.x * kCT + (int)threadIdx.x; b < B; b += (int)gridDim.x * kCT) {
        const int j = idx[b];
        const float2 s = a.rp.s[j], ac = a.rp.a[j], s2 = a.rp.s2[j];
        *reinterpret_cast<float4*>(sc.in4(0) + 4 * b) = make_float4(s2.x, s2.y, 0.f, 0.f);
        const float4 sa = make_float4(s.x, s.y, ac.x, ac.y);
        *reinterpret_cast<float4*>(sc.in4(3) + 4 * b) = sa;
        *reinterpret_cast<float4*>(sc.in4(4) + 4 * b) = sa;
        sc.rowval(0)[b] = a.rp.r[j];
        sc.rowval(1)[b] = a.rp.notdone[j];
      }
      grid_sync(a.bar, prof);
      for (int l = 1; l < L; ++l) {
        if (threadIdx.x == 0) { s_ops[0] = fwd_op(a, sc, ta, l, false); s_ops[1] = fwd_op(a, sc, c1, l, true); s_ops[2] = fwd_op(a, sc, c2, l, true); }
        __syncthreads();
        run_gemm_stage(s_ops, 3, coop_smem);
        grid_sync(a.bar, prof);
      }
      // a' = clip(pi'(s2) + clip(noise * sigma, +-c), +-max_action)        robot.py:338-339
      for (int b = global_warp(); b < B; b += total_warps()) {
        float o0, o1;
        out_layer_row(ta, sc.H(0, L - 1) + (int64_t)b * ta.s.hid, o0, o1);
        if (lane == 0) {
          Td3Hyper hp = a.hp;
          hp.noise_index = (unsigned long long)e;
          const float2 z = target_noise(a.noise ? a.noise + (int64_t)e * B * 2 : nullptr, hp, b);
          const float e0 = fminf(fmaxf(z.x * a.hp.policy_noise, -a.hp.noise_clip), a.hp.noise_clip);
          const float e1 = fminf(fmaxf(z.y * a.hp.policy_noise, -a.hp.noise_clip), a.hp.noise_clip);
          const float a0 = fminf(fmaxf(o0 + e0, -a.hp.max_action), a.hp.max_action);
          const float a1 = fminf(fmaxf(o1 + e1, -a.hp.max_action), a.hp.max_action);
          const float s2x = ldcg(sc.in4(0) + 4 * b), s2y = ldcg(sc.in4(0) + 4 * b + 1);
          const float4 in = make_float4(s2x, s2y, a0, a1);
          *reinterpret_cast<float4*>(sc.in4(1) + 4 * b) = in;
          *reinterpret_cast<float4*>(sc.in4(2) + 4 * b) = in;
        }
      }
      grid_sync(a.bar, prof);
      for (int l = 1; l < L; ++l) {
        if (threadIdx.x == 0) { s_ops[0] = fwd_op(a, sc, tc1, l, false); s_ops[1] = fwd_op(a, sc, tc2, l, false); }
        __syncthreads();
        run_gemm_stage(s_ops, 2, coop_smem);
        grid_sync(a.bar, prof);
      }
      // y, Q, losses, dout                                               robot.py:342-353
      for (int b = global_warp(); b < B; b += total_warps()) {
        float q1t, q2t, q1, q2, dummy;
        out_layer_row(tc1, sc.H(1, L - 1) + (int64_t)b * tc1.s.hid, q1t, dummy);
        out_layer_row(tc2, sc.H(2, L - 1) + (int64_t)b * tc2.s.hid, q2t, dummy);
        out_layer_row(c1, sc.H(3, L - 1) + (int64_t)b * c1.s.hid, q1, dummy);
        out_layer_row(c2, sc.H(4, L - 1) + (int64_t)b * c2.s.hid, q2, dummy);
        if (lane == 0) {
          const float y = ldcg(sc.rowval(0) + b) + a.hp.gamma * fminf(q1t, q2t) * ldcg(sc.rowval(1) + b);
          const float d1 = q1 - y, d2 = q2 - y;
          *reinterpret_cast<float2*>(sc.dout(3) + 2 * b) = make_float2(2.0f * d1 / (float)B, 0.f);
          *reinterpret_cast<float2*>(sc.dout(4) + 2 * b) = make_float2(2.0f * d2 / (float)B, 0.f);
          sc.rowval(2)[b] = d1 * d1 / (float)B;
          sc.rowval(3)[b] = d2 * d2 / (float)B;
        }
      }
      grid_sync(a.bar, prof);
      reduce_rows_to(sc.rowval(2), B, a.critic_losses + 2 * e);
      if (blockIdx.x == 0 && threadIdx.x >= 32 && threadIdx.x < 64) {           // second loss by warp 1 of block 0
        float s = 0.f;
        for (int b = lane; b < B; b += 32) s += ldcg(sc.rowval(3) + b);
        s = warp_sum(s);
        if (lane == 0) a.critic_losses[2 * e + 1] = s;
      }
      // backward through the hidden layers, top down; the output-layer gradients ride along in the first of these stages
      if (threadIdx.x == 0) { s_nets[0] = c1; s_nets[1] = c2; }
      for (int l = L - 1; l >= 1; --l) {
        if (threadIdx.x == 0) { s_ops[0] = dx_op(a, sc, c1, l); s_ops[1] = dx_op(a, sc, c2, l); s_ops[2] = dw_op(a, sc, c1, l); s_ops[3] = dw_op(a, sc, c2, l); }
        __syncthreads();
        run_gemm_stage(s_ops, 4, coop_smem);
        if (l == L - 1) small_grads(a, sc, s_nets, 2, 0, 4 * tiles_of(s_ops[0], 64), coop_smem);
        grid_sync(a.bar, prof);
      }
      small_grads(a, sc, s_nets, 2, 1, 0, coop_smem);
      grid_sync(a.bar, prof);
      if (a.world > 1) ++seq;
      adam_stage(a, 0b110, 0, seq);
      grid_sync(a.bar, prof);
    }
    // =============================================================== actor step (robot.py:369-398) + Polyak (robot.py:283-285)
    if (e % a.delay == 0) {
      const int32_t* idx = a.idx + (int64_t)k_idx * B;
      ++k_idx;
      const NetRef ac = net_ref(a, 0, 0), c1 = net_ref(a, 1, 1);
      if (blockIdx.x == 0 && threadIdx.x == 0) advance_adam_clock(a.steps, a.adam.beta_pows, 0);
      for (int b = (int)blockIdx.x * kCT + (int)threadIdx.x; b < B; b += (int)gridDim.x * kCT) {
        const float2 s = a.rp.s[idx[b]];
        *reinterpret_cast<float4*>(sc.in4(0) + 4 * b) = make_float4(s.x, s.y, 0.f, 0.f);   // the actor is fed the raw state, robot.py:386
      }
      grid_sync(a.bar, prof);
      for (int l = 1; l < L; ++l) {
        if (threadIdx.x == 0) s_ops[0] = fwd_op(a, sc, ac, l, true);
        __syncthreads();
        run_gemm_stage(s_ops, 1, coop_smem);
        grid_sync(a.bar, prof);
      }
      for (int b = global_warp(); b < B; b += total_warps()) {
        float o0, o1;
        out_layer_row(ac, sc.H(0, L - 1) + (int64_t)b * ac.s.hid, o0, o1);
        if (lane == 0) {
          const float sx = ldcg(sc.in4(0) + 4 * b), sy = ldcg(sc.in4(0) + 4 * b + 1);
          *reinterpret_cast<float4*>(sc.in4(1) + 4 * b) = make_float4(sx, sy, o0, o1);
          *reinterpret_cast<float2*>(sc.dout(1) + 2 * b) = make_float2(-1.0f / (float)B, 0.f);   // d(-mean Q)/dQ
        }
      }
      grid_sync(a.bar, prof);
      for (int l = 1; l < L; ++l) {
        if (threadIdx.x == 0) s_ops[0] = fwd_op(a, sc, c1, l, true);
        __syncthreads();
        run_gemm_stage(s_ops, 1, coop_smem);
        grid_sync(a.bar, prof);
      }
      // loss = -mean Q1(s, pi(s)) (per-row terms, summed after the next barrier); then critic-1 backward for dQ/d(input)
      for (int b = global_warp(); b < B; b += total_warps()) {
        float q, dummy;
        out_layer_row(c1, sc.H(1, L - 1) + (int64_t)b * c1.s.hid, q, dummy);
        if (lane == 0) sc.rowval(4)[b] = -q / (float)B;
      }
      for (int l = L - 1; l >= 1; --l) {
        if (threadIdx.x == 0) s_ops[0] = dx_op(a, sc, c1, l);
        __syncthreads();
        run_gemm_stage(s_ops, 1, coop_smem);
        grid_sync(a.bar, prof);
      }
      reduce_rows_to(sc.rowval(4), B, a.actor_losses + ka);
      ++ka;
      // dQ/da[b][j] = sum_k dZ0[b][k] W0c[k][2 + j]  -> the actor's dout
      for (int b = global_warp(); b < B; b += total_warps()) {
        const int Hd = c1.s.hid;
        const float* dz = sc.dZ(1, 0) + (int64_t)b * Hd;
        const float* W0 = c1.P + net_w_off(c1.s, 0);
        float g0 = 0.f, g1 = 0.f;
        for (int k = lane; k < Hd; k += 32) {
          const float d = ldcg(dz + k);
          g0 = fmaf(d, ldcg(W0 + k * 4 + 2), g0);
          g1 = fmaf(d, ldcg(W0 + k * 4 + 3), g1);
        }
        g0 = warp_sum(g0);
        g1 = warp_sum(g1);
        if (lane == 0) *reinterpret_cast<float2*>(sc.dout(0) + 2 * b) = make_float2(g0, g1);
      }
      grid_sync(a.bar, prof);
      if (threadIdx.x == 0) s_nets[0] = ac;
      for (int l = L - 1; l >= 1; --l) {
        if (threadIdx.x == 0) { s_ops[0] = dx_op(a, sc, ac, l); s_ops[1] = dw_op(a, sc, ac, l); }
        __syncthreads();
        run_gemm_stage(s_ops, 2, coop_smem);
        if (l == L - 1) small_grads(a, sc, s_nets, 1, 0, 2 * tiles_of(s_ops[0], 64), coop_smem);
        grid_sync(a.bar, prof);
      }
      small_grads(a, sc, s_nets, 1, 1, 0, coop_smem);
      grid_sync(a.bar, prof);
      if (a.world > 1) ++seq;
      adam_stage(a, 0b001, 0b111, seq);
      grid_sync(a.bar, prof);
    }
  }
  if (a.prof && blockIdx.x == 0 && threadIdx.x == 0) g_tile_prof = nullptr;
  if (a.world > 1 && blockIdx.x == 0 && threadIdx.x == 0) *a.seq_counter = seq;
}

constexpr size_t kCoopSmemBytes = (CTM * kAld + CTK * 64 + CTM * 4 + 5 * kMaxHidden) * sizeof(float);

}  // namespace rtd3

using namespace rtd3;

extern "C" {

int32_t rtd3_td3_coop_supported(const rtd3_td3* h, int32_t batch) {
  if (!h) return 0;
  const NetShape& s = h->ar.critic;
  return (s.layers >= 2 && s.hid % 4 == 0 && batch >= 1 && batch <= 4096) ? 1 : 0;
}

int64_t rtd3_td3_coop_scratch_floats(const rtd3_td3* h, int32_t batch) {
  if (!h) return -1;
  return Scratch::floats(batch, h->ar.critic.hid, h->ar.critic.layers) + kBarWords;    // + the barrier words
}

static long long* g_coop_prof = nullptr;
/* Development aid: DEVICE buffer of 256 int64 that the next cooperative updates stamp with %globaltimer at every stage boundary of
 * their last epoch (arrival of block 0 at the barrier, release from it); NULL switches it off. */
int32_t rtd3_debug_coop_prof(long long* device_buf) {
  g_coop_prof = device_buf;
  return 0;
}

int32_t rtd3_td3_update_coop(rtd3_td3* h, const rtd3_td3_update_args* a, float* coop_scratch, void* stream) {
  RTD3_CHECK_ARG(h && a && coop_scratch, "null argument");
  RTD3_CHECK_ARG(a->params && a->params_t && a->grads && a->adam_m && a->adam_v && a->steps && a->beta_pows, "null learner state");
  RTD3_CHECK_ARG(a->rp_s && a->rp_a && a->rp_r && a->rp_s2 && a->rp_notdone && a->idx, "null replay ring / index sets");
  RTD3_CHECK_ARG(a->batch > 0 && a->epochs >= 0 && a->policy_update_delay >= 1, "bad batch / epochs / policy_update_delay");
  RTD3_CHECK_ARG(a->critic_losses && a->actor_losses, "null loss outputs");
  RTD3_CHECK_ARG(a->noise || a->noise_counter, "either a noise tensor or the device noise counter is required");
  RTD3_CHECK_ARG(rtd3_td3_coop_supported(h, a->batch), "the cooperative learner needs layers >= 2 and batch <= 4096");
  RTD3_CHECK_ARG(a->world >= 1 && (a->world == 1 || a->p2p), "world > 1 needs the peer-memory state (the NCCL path uses rtd3_td3_update)");
  RTD3_CHECK_ARG(!a->tf32, "the cooperative learner is the fp32 path");
  RTD3_CHECK_ARG((uintptr_t)coop_scratch % 16 == 0, "coop_scratch must be 16 B aligned");
  if (a->epochs == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  CoopArgs c{};
  c.prof = g_coop_prof;
  c.adam = adam_state(h, a);
  c.grads = a->grads; c.steps = a->steps;
  c.rp = ReplayView{(const float2*)a->rp_s, (const float2*)a->rp_a, a->rp_r, (const float2*)a->rp_s2, a->rp_notdone};
  c.idx = a->idx; c.noise = a->noise;
  c.hp = Td3Hyper{a->gamma, a->policy_noise, a->noise_clip, a->max_action, (unsigned long long)a->noise_seed,
                  (const unsigned long long*)a->noise_counter, 0ull};
  c.B = a->batch; c.E = a->epochs; c.delay = a->policy_update_delay;
  c.critic_losses = a->critic_losses; c.actor_losses = a->actor_losses;
  // the first kBarWords floats of the scratch hold the barrier words (zero-initialised by the caller once; the barrier leaves them zero /
  // monotone), the rest is the activation scratch
  c.bar = GridBarrier{reinterpret_cast<unsigned int*>(coop_scratch), reinterpret_cast<volatile unsigned int*>(coop_scratch) + 32};
  c.scratch = coop_scratch + kBarWords;
  c.world = a->world;
  if (a->world > 1) {
    const rtd3_p2p_state* p = a->p2p;
    RTD3_CHECK_ARG(p->world == a->world && p->world <= kCoopMaxWorld && p->rank >= 0 && p->rank < p->world, "bad peer-memory state");
    RTD3_CHECK_ARG(p->slot_floats >= h->ar.online_total(), "receive slots smaller than the gradient buffer");
    c.rank = p->rank;
    for (int r = 0; r < p->world; ++r) {
      c.peers.recv[r] = p->peer_recv[r];
      c.peers.flags[r] = (unsigned long long*)p->peer_flags[r];
    }
    c.seq_counter = (unsigned long long*)p->seq_counter;
    c.slot_floats = p->slot_floats;
  }
  RTD3_CUDA(ensure_dyn_smem((const void*)td3_update_coop_kernel, kCoopSmemBytes));
  int per_sm = 0;
  RTD3_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, td3_update_coop_kernel, kCT, kCoopSmemBytes));
  RTD3_CHECK_ARG(per_sm >= 1, "the cooperative kernel does not fit on an SM");
  const int grid = h->num_sms;                           // one CTA per SM
  void* kargs[] = {&c};
  RTD3_CUDA(cudaLaunchCooperativeKernel((const void*)td3_update_coop_kernel, dim3(grid), dim3(kCT), kargs, kCoopSmemBytes, st));
  count_launch();
  if (!a->noise) return advance_noise_counter(a->noise_counter, (uint64_t)a->epochs, st);   // as rtd3_td3_update does
  return 0;
}

}  // extern "C"
