// Large-batch network forward on the 5th-generation tensor cores (tcgen05 + TMEM), TF32 operands, fp32 accumulate.
// Opt-in throughput mode (TD3.precision = "tf32"): the north star asks for tensor cores "only where the shapes
// justify it" - a 128-row batch tile against an H x H hidden layer (M=128, N=H<=256, K=H) does, the 4..16-row tiles of
// the small-batch learner do not.  fp32 FFMA (rtd3_mlp.cuh) stays the parity path; this one is checked against it
// at TF32 tolerance (tests/test_tc_gpu.py).
//
// One CTA = 128 batch rows through the whole network (robot.py:153-159 / 193-200):
//   first layer (in <= 4) and output layer (out <= 2): FFMA by the 128 row threads;
//   every hidden H x H layer: D[128 x H] (TMEM, fp32) = X[128 x H] * W^T, issued as H/8 tcgen05.mma.kind::tf32 by ONE
//   thread, operands in shared memory in the no-swizzle K-major canonical layout (16 B k-chunks, 8-row core matrices):
//       X : chunk-major [H/4][128 rows][4]   (LBO = 2048 B between k-chunks, SBO = 128 B between 8-row groups)
//       W : chunk-major [H/4][H rows n][4]   (LBO = 16*H B,                  SBO = 128 B) - kept in exactly this order in a
//           third parameter arena (params_u), so a 32-wide K slab is ONE contiguous cp.async.bulk (TMA) per stage;
//   epilogue: the row threads read their TMEM lane with tcgen05.ld (32 columns at a time), add bias, ReLU, and write the
//   next layer's X straight back in the chunk layout (16 B per 4 columns, consecutive rows -> conflict-free).
#include <cstdlib>
#include <cuda_fp16.h>

#include "rtd3_common.cuh"
#include "rtd3_mlp.cuh"
#include "rtd3_tc.cuh"
#include "rtd3_tc_f16.cuh"
#include "rtd3_td3.cuh"

namespace rtd3 {

constexpr int kTcRows = 128;          // batch rows per CTA = UMMA M
constexpr int kTcRowWarps = 16;       // four per TMEM sub-partition: warp w serves rows 32*(w%4).. and column quarter w/4 (H % 128 == 0),
constexpr int kTcColParts = kTcRowWarps / 4;   // else two active per sub-partition with column halves (H % 64 == 0)
constexpr int kTcThreads = (kTcRowWarps + 2) * 32;   // warps 0-15: row threads / epilogue, warp 16: TMA producer, warp 17: MMA issuer
constexpr int kTcKSlab = 32;          // K per pipeline stage = 4 MMAs of K=8
constexpr int kTcStages = 2;

// Shared-memory plan (bytes): X [H/4][128][4] | W stages [2][8][H][4] | small params | barriers | tmem base
__host__ __device__ inline size_t tc_smem_bytes(int hid, int layers) {
  return (size_t)hid * 512 + (size_t)kTcStages * hid * 128 + ((size_t)hid * 4 + hid + (size_t)(layers - 1) * hid + 2 * hid + 4) * 4 + 64 + kTcColParts * kTcRows * 2 * 4;
}

__global__ void __launch_bounds__(kTcThreads, 1)
mlp_forward_tc_kernel(NetShape s, const float* __restrict__ P /*torch layout*/, const float* __restrict__ Pu /*chunk-major hidden weights*/,
                      const float* __restrict__ x /*[B][in]*/, float* __restrict__ y /*[B][out]*/, int B) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int H = s.hid, L = s.layers;
  float* Xs = reinterpret_cast<float*>(smem_raw);                                   // [H/4][128][4]
  float* Ws = Xs + (size_t)H * 128;                                                 // [2][8][H][4]
  float* small = Ws + (size_t)kTcStages * H * 32;
  float* W1 = small;                    // [H][4] (zero-padded input dim)
  float* b1 = W1 + H * 4;               // [H]
  float* bh = b1 + H;                   // [L-1][H]
  float* Wo = bh + (L - 1) * H;         // [2][H]
  float* bo = Wo + 2 * H;               // [2] (+2 pad)
  uint64_t* bars = reinterpret_cast<uint64_t*>(bo + 4);                             // full[2], empty[2], acc_ready
  uint64_t* full = bars, *empty = bars + kTcStages, *acc_ready = bars + 2 * kTcStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kTcStages + 1);
  float* part = reinterpret_cast<float*>(bars + 2 * kTcStages + 2);                 // [column parts][128 rows][2] output-layer partial sums

  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int rt = (warp & 3) * 32 + lane;            // row threads: tile row (= TMEM lane) ...
  // ... and column part of this thread: quarters when every quarter is a whole number of 32-column TMEM loads, else halves or
  // the whole row (the surplus warps of each sub-partition then idle through the barriers with an empty column range)
  const int parts = (H % (32 * kTcColParts) == 0) ? kTcColParts : ((H % 64 == 0) ? 2 : 1);
  const int cpart = warp >> 2;
  const int c_lo = cpart < parts ? cpart * (H / parts) : 0, c_hi = cpart < parts ? c_lo + H / parts : 0;
  const int tiles = (B + kTcRows - 1) / kTcRows;

  // ---- setup (once per CTA: the kernel is persistent over its tiles): small parameters, barriers, TMEM allocation -----
  for (int i = t; i < H * 4; i += kTcThreads) {
    const int c = i >> 2, j = i & 3;
    W1[i] = j < s.in ? __ldg(P + net_w_off(s, 0) + c * s.in + j) : 0.f;
  }
  for (int i = t; i < H; i += kTcThreads) b1[i] = __ldg(P + net_b_off(s, 0) + i);
  for (int l = 1; l < L; ++l)
    for (int i = t; i < H; i += kTcThreads) bh[(l - 1) * H + i] = __ldg(P + net_b_off(s, l) + i);
  for (int i = t; i < 2 * H; i += kTcThreads) Wo[i] = (i / H) < s.out ? __ldg(P + net_w_off(s, L) + i) : 0.f;
  if (t < 2) bo[t] = t < s.out ? __ldg(P + net_b_off(s, L) + t) : 0.f;
  if (t == 0) {
    for (int i = 0; i < kTcStages; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
    mbar_init(acc_ready, 1);
    fence_mbar_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // instruction descriptor: D = F32, A = B = TF32, both K-major, N = H, M = 128
  const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)(kTcRows >> 4) << 24);
  const int slabs = H / kTcKSlab;
  const uint32_t stage_bytes = (uint32_t)H * (kTcKSlab / 4) * 16;      // 8 chunks x H rows x 16 B
  constexpr int kRowMma = (kTcRowWarps + 1) * 32;                      // named barrier 2: row warps + the MMA warp

  if (warp == kTcRowWarps) {
    // ===== TMA producer: free-running over (tile, layer, K slab); one contiguous bulk copy per slab.  It is throttled only by the
    // stage ring, so the first slabs of the next tile arrive while the row warps still work on the current one.
    if (lane == 0) {
      uint32_t it_p = 0;
      for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x)
        for (int l = 1; l < L; ++l) {
          const float* Wu = Pu + net_w_off(s, l);
          for (int ks = 0; ks < slabs; ++ks, ++it_p) {
            const int st = it_p % kTcStages;
            mbar_wait(empty + st, ((it_p / kTcStages) & 1) ^ 1);
            mbar_arrive_expect_tx(full + st, stage_bytes);
            bulk_g2s(Ws + (size_t)st * H * 32, Wu + (size_t)ks * H * 32, stage_bytes, full + st);
          }
        }
    }
  } else if (warp == kTcRowWarps + 1) {
    // ===== MMA issuer =====
    uint32_t it_c = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x)
      for (int l = 1; l < L; ++l) {
        bar_sync(2, kRowMma);                         // X of this layer is in shared memory, the accumulator has been drained
        if (lane == 0) {
          tc_fence_after();
          for (int ks = 0; ks < slabs; ++ks, ++it_c) {
            const int st = it_c % kTcStages;
            mbar_wait(full + st, (it_c / kTcStages) & 1);
            tc_fence_after();
#pragma unroll
            for (int k4 = 0; k4 < kTcKSlab / 8; ++k4) {
              const uint64_t ad = umma_desc_kmajor(smem_u32(Xs + (size_t)(ks * 8 + k4 * 2) * (kTcRows * 4)), kTcRows * 16, 128);
              const uint64_t bd = umma_desc_kmajor(smem_u32(Ws + (size_t)st * H * 32 + (size_t)(k4 * 2) * H * 4), (uint32_t)H * 16, 128);
              umma_tf32(tmem, ad, bd, idesc, (ks | k4) != 0 ? 1u : 0u);
            }
            umma_commit(empty + st);                  // frees the weight stage once these MMAs have read it
          }
          umma_commit(acc_ready);                     // accumulator complete (commits track all prior MMAs)
        }
        __syncwarp();
      }
  } else {
    // ===== row warps: first layer, epilogues, output layer =====
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
      const int r0 = tile * kTcRows;
      const int row = r0 + rt;
      float x0[4] = {0.f, 0.f, 0.f, 0.f};
      if (row < B)
        for (int j = 0; j < s.in; ++j) x0[j] = x[(int64_t)row * s.in + j];
      // first layer: X = relu(b1 + x0 W1^T) in the chunk layout (the previous tile's readers of X are past their last barrier)
      for (int c = c_lo; c < c_hi; c += 4) {
        float4 h;
        float* hp = &h.x;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 w = *reinterpret_cast<const float4*>(W1 + (c + q) * 4);
          float v = b1[c + q];
          v = fmaf(x0[0], w.x, v); v = fmaf(x0[1], w.y, v); v = fmaf(x0[2], w.z, v); v = fmaf(x0[3], w.w, v);
          hp[q] = fmaxf(v, 0.f);
        }
        *reinterpret_cast<float4*>(Xs + (size_t)(c >> 2) * (kTcRows * 4) + rt * 4) = h;
      }
      for (int l = 1; l < L; ++l) {
        fence_proxy_async();                          // generic-proxy writes of X -> visible to the tensor core (async proxy)
        tc_fence_before();
        bar_sync(2, kRowMma);
        // epilogue: TMEM -> registers -> bias + ReLU -> next X (in place: every MMA that read X has completed)
        mbar_wait(acc_ready, acc_phase);
        acc_phase ^= 1;
        tc_fence_after();
        const float* bias = bh + (l - 1) * H;
        for (int cb = c_lo; cb < c_hi; cb += 32) {
          float v[32];
          tmem_ld32(tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)cb, v);
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float4 h;
            h.x = fmaxf(v[4 * q + 0] + bias[cb + 4 * q + 0], 0.f);
            h.y = fmaxf(v[4 * q + 1] + bias[cb + 4 * q + 1], 0.f);
            h.z = fmaxf(v[4 * q + 2] + bias[cb + 4 * q + 2], 0.f);
            h.w = fmaxf(v[4 * q + 3] + bias[cb + 4 * q + 3], 0.f);
            *reinterpret_cast<float4*>(Xs + (size_t)((cb >> 2) + q) * (kTcRows * 4) + rt * 4) = h;
          }
        }
        tc_fence_before();
      }
      bar_sync(1, kTcRowWarps * 32);                  // all column parts of every row are written
      // output layer: each thread sums its column half, the halves meet in shared memory
      float o0 = 0.f, o1 = 0.f;
      for (int c = c_lo; c < c_hi; c += 4) {
        const float4 h = *reinterpret_cast<const float4*>(Xs + (size_t)(c >> 2) * (kTcRows * 4) + rt * 4);
        const float4 w0 = *reinterpret_cast<const float4*>(Wo + c), w1 = *reinterpret_cast<const float4*>(Wo + H + c);
        o0 = fmaf(h.x, w0.x, o0); o0 = fmaf(h.y, w0.y, o0); o0 = fmaf(h.z, w0.z, o0); o0 = fmaf(h.w, w0.w, o0);
        o1 = fmaf(h.x, w1.x, o1); o1 = fmaf(h.y, w1.y, o1); o1 = fmaf(h.z, w1.z, o1); o1 = fmaf(h.w, w1.w, o1);
      }
      part[(cpart * kTcRows + rt) * 2] = o0;        // warps without columns contribute zeros
      part[(cpart * kTcRows + rt) * 2 + 1] = o1;
      bar_sync(1, kTcRowWarps * 32);
      if (warp < 4 && row < B) {
        float y0 = bo[0], y1 = bo[1];
#pragma unroll
        for (int c = 0; c < kTcColParts; ++c) { y0 += part[(c * kTcRows + rt) * 2]; y1 += part[(c * kTcRows + rt) * 2 + 1]; }
        y[(int64_t)row * s.out] = y0;
        if (s.out > 1) y[(int64_t)row * s.out + 1] = y1;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(256) : "memory");
}

// ---- f16 forward with the hidden weights RESIDENT in shared memory (layers == 2) ---------------------------------------------
// The TF32 kernel above streams the 256 KB of W2 (H = 256) from L2 for every 128-row tile: its 64 KB of stage ring holds what
// one TMA latency delivers, so the tile time is the weight stream, not the tensor core (12 us per tile against 2 us of MMAs).
// fp16 operands carry the same 11-bit significand as TF32 in half the bytes: W2 is 128 KB and stays in shared memory for the
// whole launch next to a 64 KB X tile, the MMAs run at the 16-bit rate (K = 16 per instruction), and nothing is streamed.
// (Range: |W| <= sqrt(6/fan_in), post-ReLU first-layer activations are bounded by |state - goal| * |W1| < 400 << 65504; the
// conversion saturates.)  With two accumulator buffers in TMEM the epilogue of tile i (bias, ReLU and the fused output layer,
// straight from the accumulator: X is never written back) overlaps the MMAs of tile i+1:
//   row warps : wait acc(i) -> first layer of tile i+1 into X -> barrier -> epilogue + output layer of tile i
//   MMA warp  : barrier -> H/16 tcgen05.mma.kind::f16 into acc((i+1) & 1) -> commit
// The per-tile pieces live in rtd3_tc_f16.cuh (the multi-tick kernel of rtd3_tick.cu runs the same code).
__global__ void __launch_bounds__(kHfThreads, 1)
mlp_forward_f16_kernel(NetShape s, const float* __restrict__ P /*torch layout*/, const uint16_t* __restrict__ Wh /*[H/8][H][8] half*/,
                       const float* __restrict__ x /*[B][in]*/, float* __restrict__ y /*[B][out]*/, int B, uint32_t tmem_cols) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int H = s.hid;
  const HfSmem m = hf_carve(smem_raw, H);
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int rt = (warp & 3) * 32 + lane, cpart = warp >> 2;
  int c_lo, c_hi;
  hf_columns(H, cpart, c_lo, c_hi);
  const int tiles = (B + kHfRows - 1) / kHfRows;
  const bool in2 = s.in <= 2;
  const uint32_t tmem = hf_setup(m, s, P, Wh, tmem_cols);
  const uint32_t idesc = hf_idesc(H);

  if (warp == kHfRowWarps) {
    // ===== MMA issuer =====
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      bar_sync(2, kHfRowMma);                         // X of this tile is in shared memory; accumulator (it & 1) has been drained
      if (lane == 0) {
        if (it == 0) mbar_wait(m.w_full, 0);
        hf_issue_tile(m, H, tmem + (it & 1u) * (uint32_t)H, idesc, m.acc_ready + (it & 1u));
      }
      __syncwarp();
    }
  } else {
    // ===== row warps =====
    auto load_x = [&](int tile, float (&x0)[4]) {   // this thread's input row of `tile`
      const int row = tile * kHfRows + rt;
#pragma unroll
      for (int j = 0; j < 4; ++j) x0[j] = (row < B && j < s.in) ? __ldg(x + (int64_t)row * s.in + j) : 0.f;
    };
    float xn[4];
    if ((int)blockIdx.x < tiles) {
      load_x(blockIdx.x, xn);
      hf_first_layer(m, xn, in2, rt, c_lo, c_hi);
      bar_sync(2, kHfRowMma);
    }
    uint32_t it = 0, phase0 = 0, phase1 = 0;
    for (int tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++it) {
      const int row = tile * kHfRows + rt;
      const bool more = tile + (int)gridDim.x < tiles;
      if (more) load_x(tile + gridDim.x, xn);         // in flight while this tile's products finish
      if (it & 1u) { mbar_wait(m.acc_ready + 1, phase1); phase1 ^= 1; }
      else { mbar_wait(m.acc_ready, phase0); phase0 ^= 1; }
      tc_fence_after();
      // the MMAs of this tile have read X: the next tile's first layer may overwrite it, and its MMAs then run under the epilogue below
      if (more) {
        hf_first_layer(m, xn, in2, rt, c_lo, c_hi);
        bar_sync(2, kHfRowMma);
      }
      // two part buffers: tile i+1 writes the other one, and the barrier of tile i+1 orders tile i+2's writes after tile i's reads
      hf_epilogue(m, tmem + (it & 1u) * (uint32_t)H + ((uint32_t)((warp & 3) * 32) << 16), rt, cpart, c_lo, c_hi, (int)(it & 1u));
      bar_sync(1, kHfRowThreads);
      if (warp < 4 && row < B) {
        const float2 o = hf_output(m, rt, (int)(it & 1u));
        y[(int64_t)row * s.out] = o.x;
        if (s.out > 1) y[(int64_t)row * s.out + 1] = o.y;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(tmem_cols) : "memory");
}

// fp16 arena: six slots of (L-1) hidden-to-hidden weights, nothing else: params_h[(net*(L-1) + l-1)*H*H + ((k/8)*H + n)*8 + k%8] =
// half(W_l[n][k]) (every matrix 16 B aligned, which the torch-order slots of the fp32 arena are not)
__global__ void sync_half_kernel(Arena ar, const float* __restrict__ params, uint16_t* __restrict__ params_h) {
  const int64_t total = ar.total();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int net = 5;
    while (net > 0 && i < ar.off(net)) --net;
    const NetShape& s = (net % 3 == 0) ? ar.actor : ar.critic;
    const SlotPos q = slot_pos(s, (int)(i - ar.off(net)));
    if (!q.hidden) continue;
    const int64_t hh = (int64_t)s.hid * s.hid, l = q.l, n = q.n, k = q.k;
    params_h[((int64_t)net * (s.layers - 1) + l) * hh + ((k >> 3) * s.hid + n) * 8 + (k & 7)] =
        __half_as_ushort(__float2half_rn(fminf(fmaxf(params[i], -65504.f), 65504.f)));
  }
}

// Rebuild both chunk-major copies of the whole arena (u: forward operand order, v: input-gradient operand order).
__global__ void sync_chunk_major_kernel(NetShape actor, NetShape critic, int64_t sa, int64_t sc, const float* __restrict__ params,
                                        float* __restrict__ params_uv) {
  const int64_t n_online = sa + 2 * sc, total = 2 * n_online;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i < n_online ? i : i - n_online;
    const int net = j < sa ? 0 : (j < sa + sc ? 1 : 2);
    const int64_t off = (i < n_online ? 0 : n_online) + (net == 0 ? 0 : (net == 1 ? sa : sa + sc));
    const CopyIndex c = copy_index(net == 0 ? actor : critic, (int)(i - off));
    const float p = c.hidden ? tf32_rn(params[i]) : params[i];
    params_uv[off + c.u] = p;
    params_uv[total + off + c.v] = p;
  }
}

}  // namespace rtd3

using namespace rtd3;

extern "C" {

/* Rebuild the chunk-major (UMMA operand order) copy of all hidden-layer weights from the torch-layout arena. */
int32_t rtd3_tc_sync_weights(int32_t hidden, int32_t layers, const float* params, float* params_uv, void* stream) {
  RTD3_CHECK_ARG(params && params_uv && hidden >= 4 && hidden <= kMaxHidden && layers >= 1 && layers <= kMaxLayers, "bad argument");
  const NetShape a{2, hidden, layers, 2}, c{4, hidden, layers, 1};
  sync_chunk_major_kernel<<<296, 256, 0, (cudaStream_t)stream>>>(a, c, net_stride(a), net_stride(c), params, params_uv);
  RTD3_LAUNCHED();
  return 0;
}

/* Network forward on tcgen05 tensor cores (TF32 operands, fp32 accumulate) for batch tiles of 128 rows.
 * net: 0/3 actor (2->H..->2), else critic (4->H..->1); param_off: offset of the network's slot in both arenas.
 * Requires hidden % 32 == 0, 64 <= hidden <= 256. */
int32_t rtd3_mlp_forward_tf32(int32_t hidden, int32_t layers, int32_t is_actor, int64_t param_off, const float* params, const float* params_u,
                              const float* x, float* y, int64_t batch, void* stream) {
  RTD3_CHECK_ARG(params && params_u && x && y, "null argument");
  RTD3_CHECK_ARG(hidden % 32 == 0 && hidden >= 64 && hidden <= 256 && layers >= 2 && layers <= kMaxLayers,
                 "tf32 path needs hidden in {64..256} divisible by 32 and at least one hidden-to-hidden layer");
  RTD3_CHECK_ARG(batch >= 0 && batch < (1ll << 31), "bad batch");
  if (batch == 0) return 0;
  const NetShape s = is_actor ? NetShape{2, hidden, layers, 2} : NetShape{4, hidden, layers, 1};
  const size_t smem = tc_smem_bytes(hidden, layers);
  RTD3_CUDA(ensure_dyn_smem((const void*)mlp_forward_tc_kernel, smem));
  // persistent: one CTA per SM (193 KB of shared memory each) walking its tiles; setup and TMEM allocation happen once per CTA
  const int tiles = (int)ceil_div(batch, kTcRows);
  int num_sms = 0;
  RTD3_CUDA(current_num_sms(&num_sms));
  const int grid = tiles < num_sms ? tiles : num_sms;
  mlp_forward_tc_kernel<<<grid, kTcThreads, smem, (cudaStream_t)stream>>>(s, params + param_off, params_u + param_off, x, y, (int)batch);
  RTD3_LAUNCHED();
  return 0;
}

/* fp16 chunk-major copies of the hidden-to-hidden weights of all six networks (see mlp_forward_f16_kernel). */
int32_t rtd3_tc_sync_weights_f16(int32_t hidden, int32_t layers, const float* params, uint16_t* params_h, void* stream) {
  RTD3_CHECK_ARG(params && params_h && hidden >= 4 && hidden <= kMaxHidden && layers >= 1 && layers <= kMaxLayers, "bad argument");
  const Arena ar{NetShape{2, hidden, layers, 2}, NetShape{4, hidden, layers, 1}};
  sync_half_kernel<<<296, 256, 0, (cudaStream_t)stream>>>(ar, params, params_h);
  RTD3_LAUNCHED();
  return 0;
}

/* Network forward with fp16 operands on the tcgen05 tensor cores, hidden weight resident in shared memory (layers == 2). */
int32_t rtd3_mlp_forward_f16(int32_t hidden, int32_t layers, int32_t net, const float* params, const uint16_t* params_h, const float* x,
                             float* y, int64_t batch, void* stream) {
  RTD3_CHECK_ARG(params && params_h && x && y, "null argument");
  RTD3_CHECK_ARG(hidden % 32 == 0 && hidden >= 64 && hidden <= 256 && layers == 2, "f16 path needs layers == 2 and hidden in {64..256} divisible by 32");
  RTD3_CHECK_ARG(net >= 0 && net < 6, "net must be 0..5");
  RTD3_CHECK_ARG(batch >= 0 && batch < (1ll << 31), "bad batch");
  if (batch == 0) return 0;
  const Arena ar{NetShape{2, hidden, layers, 2}, NetShape{4, hidden, layers, 1}};
  const NetShape s = net % 3 == 0 ? ar.actor : ar.critic;
  const int64_t param_off = ar.off(net);
  const uint16_t* wh = params_h + (int64_t)net * (layers - 1) * hidden * hidden;
  const size_t smem = hf_smem_bytes(hidden);
  RTD3_CUDA(ensure_dyn_smem((const void*)mlp_forward_f16_kernel, smem));
  const int tiles = (int)ceil_div(batch, kHfRows);
  int num_sms = 0;
  RTD3_CUDA(current_num_sms(&num_sms));
  uint32_t cols = 32;
  while (cols < 2u * (uint32_t)hidden) cols <<= 1;      // two accumulator buffers, a power of two of TMEM columns
  const int grid = tiles < num_sms ? tiles : num_sms;
  mlp_forward_f16_kernel<<<grid, kHfThreads, smem, (cudaStream_t)stream>>>(s, params + param_off, wh, x, y, (int)batch, cols);
  RTD3_LAUNCHED();
  return 0;
}

}  // extern "C"
