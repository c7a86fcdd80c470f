// Small-batch residual-TD3 steps on thread-block clusters (fp32, the parity path): robot.py:312-366 (train_critic) and
// robot.py:369-398 (train_actor) up to the optimiser steps, for batches that cannot fill the GPU row by row.
//
// The row-tile kernels of rtd3_td3.cu give every CTA 2-16 batch rows and let it stream the weights of all five networks from L2:
// at B = 256 that is 128 CTAs x 1.8 MB = 240 MB of L2 reads for 3.2 MB of parameters, and the step runs at the L2 bandwidth.  Here a
// CLUSTER of CS CTAs owns R batch rows and splits the COLUMNS of every layer: CTA c computes output columns [c*Wc, (c+1)*Wc) of each
// layer for all R rows, so it needs 1/CS of every weight matrix (a [H][Wc] column slice, staged by cp.async through a ring that runs
// ahead of the arithmetic - the weights do not depend on the activations), and pushes its slice of the layer output into the shared
// memory of all CTAs of the cluster so that each of them holds the full-width input of the next layer.  The pushes are st.async
// stores that complete transaction bytes on an mbarrier of the RECEIVING CTA: a CTA goes on as soon as ITS input is complete - no
// cluster-wide barrier per layer (measured: barrier.cluster after a push costs 1 300-2 900 cycles, the products 1 500).  Two
// mbarriers alternate by stage; consecutive stages write different tiles, and a CTA can only be one stage ahead of the slowest CTA
// of its cluster (it needs that CTA's output to go on), which is what makes the reuse of tiles and barriers two stages later safe.
// What is NOT exchanged: the first layer (2-4 inputs) is evaluated for all H columns by every CTA, and the last hidden layer's
// output stays with its CTA - only its contribution to the 1-2 head outputs (R x out partial sums) is pushed.  So a forward pass of
// a 2-hidden-layer network costs one tiny exchange, a backward pass one full one.  A ninth warp does nothing but issue the weight
// copies (an issue costs ~100 cycles per bulk copy, 16 per tile).  The per-row layer inputs / pre-activation gradients go to the same
// row scratch as before; wgrad_kernel (+ fused Adam) consumes them.
#include <algorithm>

#include "rtd3_common.cuh"
#include "rtd3_mlp.cuh"
#include "rtd3_td3.cuh"

namespace rtd3 {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t map_to_rank(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// 16 / 8 bytes into the shared memory of a CTA of the cluster; the bytes are counted on that CTA's mbarrier when they have landed
__device__ __forceinline__ void st_async4(uint32_t addr, const float4& v, uint32_t bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.f32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(addr), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void st_async2(uint32_t addr, float a, float b, uint32_t bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(addr), "f"(a), "f"(b), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// (default semantics, acquire at CTA scope: the bytes counted on the barrier are visible to whoever observes the phase - the pattern
// of every TMA / st.async consumer.  With .acquire.cluster ptxas adds CCTL.IVALL, an L1 invalidate, to EVERY wait of every warp:
// 12 % of the kernel's stall samples.)
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAITC_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONEC_%=;\n"
      "bra WAITC_%=;\n"
      "DONEC_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}


constexpr int kCT = kThreads;            // compute threads; one more warp issues the weight copies
constexpr int kClBlock = kCT + 32;
__device__ __forceinline__ void cta_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kCT) : "memory"); }   // the compute threads only

// Shared-memory plan of one CTA (offsets in floats into smem_f), its place in the cluster and the running stage state.
struct Cl {
  int ring;          // [ns][Wc / 4][4 H + 4] weight slices: groups of 4 rows, row n = the H weights that feed own output column n
  int red;           // [KG][R][Wc] partial sums of the reduction groups
  int small;         // per network: W0 [H][in] b0 [H] (one copy) | pad to 5 H | b_l [L-1][H] | head [out][H] + head bias (one copy)
  int act0;          // kept activations, nkeep full-width [R][ld] tiles
  int xl;            // first-layer output of a network whose activations are not kept (written locally only)
  int dz0, dz1;      // full-width tiles that receive pushed slices (they alternate; one tile when there is one push per pass)
  int in0, out, dout, din, S;         // [R][4], [R][2], [R][2], [R][4], [R][8]
  int hpart;         // [R][Wc / 4][2] head contributions of the column groups
  int hp, dinp;      // [CS][R][2] each: head / input-gradient partial sums of the CTAs of the cluster
  int bar;           // mbarriers (uint64): [0,1] stages, [2..4] ring slot full, [5..7] ring slot empty, [8] small parameters
  int ld, Wc, H, L, ns, tile_floats, small_stride;
  int ncg_sh;        // log2 of the column groups a reduction group spans (>= Wc / 4)
  int kgn, part;     // reduction groups and their length
  int rank, c_lo, ncols;
  int started;       // 0 until this thread has waited for the start barrier (it does so right before the cluster's first push)
  int stg;           // stages completed so far (the same number in every thread of the cluster)
  int dsel;          // which dz tile the next pushed output goes to
  long long* prof;   // development: stage stamps of thread 0 of CTA 0 ((code << 48) | clock64), nullptr = off
  int pn;
};
__device__ __forceinline__ void stamp(Cl& c, int code) {
  if (c.prof && threadIdx.x == 0 && c.pn < 254) c.prof[1 + c.pn++] = ((long long)code << 48) | (clock64() & 0xffffffffffffll);
}

struct ClPlan {      // host side of the same plan
  int ns;
  size_t bytes;
};

__host__ __device__ inline int cl_wc(int H, int CS) { return ((H + 4 * CS - 1) / (4 * CS)) * 4; }
__host__ __device__ inline int cl_ncg_sh(int Wc) {
  int sh = 0;
  while ((4 << sh) < Wc) ++sh;
  return sh;
}
constexpr size_t kClSmemLimit = 226 * 1024;

static ClPlan make_plan(int R, int CS, int H, int L, int nets, int nkeep) {
  const int Wc = cl_wc(H, CS), ld = H + 4;
  const int kgn = kCT / ((1 << cl_ncg_sh(Wc)) * (R / 4));
  const size_t tile = (size_t)(Wc / 4) * (4 * H + 4);
  const size_t small_stride = (size_t)(6 + L) * H + 4;
  const size_t fixed = (size_t)kgn * R * Wc + nets * small_stride + (size_t)(nkeep + (L >= 3 ? 3 : 2)) * R * ld + R * (4 + 2 + 2 + 4 + 8) +
                       (size_t)R * (Wc / 4) * 2 + (size_t)2 * CS * R * 2 + 24;
  ClPlan p;
  p.ns = 3;
  p.bytes = (fixed + p.ns * tile) * sizeof(float);
  if (p.bytes > kClSmemLimit) {
    p.ns = 2;
    p.bytes = (fixed + p.ns * tile) * sizeof(float);
  }
  return p;
}

__device__ __forceinline__ void cl_carve(Cl& c, int R, int CS, int H, int L, int ns, int nets, int nkeep) {
  c.H = H; c.L = L; c.ns = ns;
  c.Wc = cl_wc(H, CS);
  c.ld = H + 4;
  c.tile_floats = (c.Wc / 4) * (4 * H + 4);
  c.small_stride = (6 + L) * H + 4;
  c.ncg_sh = cl_ncg_sh(c.Wc);
  c.kgn = kCT / ((1 << c.ncg_sh) * (R / 4));
  c.part = ((H + 4 * c.kgn - 1) / (4 * c.kgn)) * 4;
  int p = 0;
  c.ring = p; p += ns * c.tile_floats;
  c.red = p; p += c.kgn * R * c.Wc;
  c.small = p; p += nets * c.small_stride;
  c.act0 = p; p += nkeep * R * c.ld;
  c.xl = p; p += R * c.ld;
  c.dz0 = p; p += R * c.ld;
  c.dz1 = c.dz0;
  if (L >= 3) { c.dz1 = p; p += R * c.ld; }
  c.in0 = p; p += R * 4;
  c.out = p; p += R * 2;
  c.dout = p; p += R * 2;
  c.din = p; p += R * 4;
  c.S = p; p += R * 8;
  c.hpart = p; p += R * (c.Wc / 4) * 2;
  c.hp = p; p += CS * R * 2;
  c.dinp = p; p += CS * R * 2;
  c.bar = p;
  c.rank = (int)cluster_ctarank();
  c.c_lo = c.rank * c.Wc;
  c.ncols = max(0, min(c.Wc, H - c.c_lo));
  c.stg = 0; c.dsel = 0; c.started = 0;
  c.prof = nullptr; c.pn = 0;
}

// ---- weight ring ------------------------------------------------------------------------------------------------------------------
// tile = the rows of one H x H matrix that produce the own output columns: forward W_l[n][:] (torch layout, n = own column),
// backward Wt_l[k][:] (the transposed copy, k = own column) - Wc contiguous rows of H floats, fetched in groups of 4 rows (one bulk
// copy of 16 H bytes per group: per-row copies made the issue, ~100 cycles per copy, the longest part of a stage) into groups of
// pitch 4 H + 4 floats: the product's lane cl reads the rows of group cl, and the skew keeps the lanes on different banks.
// The producer warp (threads kCT..) issues tile after tile as the ring's slots are released.
__device__ __forceinline__ uint64_t* cl_bar(const Cl& c, int i) { return reinterpret_cast<uint64_t*>(smem_f + c.bar) + i; }
__device__ __forceinline__ void cl_producer(const Cl& c, const float* const* tiles, int first, int ntiles) {
  const int lane = threadIdx.x - kCT;
  for (int i = first; i < ntiles; ++i) {
    const int slot = i % c.ns;
    if (i >= c.ns) mbar_wait(cl_bar(c, 5 + slot), (uint32_t)((i / c.ns - 1) & 1));
    if (c.ncols > 0) {
      uint64_t* bar = cl_bar(c, 2 + slot);
      if (lane == 0) mbar_arrive_expect_tx(bar, (uint32_t)(c.ncols * c.H * 4));
      __syncwarp();
      if (lane < (c.ncols >> 2))
        bulk_g2s(smem_f + c.ring + slot * c.tile_floats + lane * (4 * c.H + 4), tiles[i] + (int64_t)(c.c_lo + 4 * lane) * c.H, (uint32_t)(16 * c.H),
                 bar);
    }
  }
}
// make tile i resident (compute threads)
__device__ __forceinline__ int tile_acquire(const Cl& c, int i) {
  cta_sync();          // the previous epilogue has left the partial sums (the stage waits in between are not CTA barriers)
  if (c.ncols > 0) mbar_wait(cl_bar(c, 2 + i % c.ns), (uint32_t)((i / c.ns) & 1));
  return c.ring + (i % c.ns) * c.tile_floats;
}
// all compute threads have left the product of tile i: its slot may be refilled
__device__ __forceinline__ void tile_release(const Cl& c, int i) {
  if (threadIdx.x == 0) mbar_arrive(cl_bar(c, 5 + i % c.ns));
}

// small parameters: per network three kinds of bulk copies, issued by the lanes of the producer warp at kernel start onto mbarrier 8 -
// W0 and b0 (adjacent in the arena), every further bias vector, the head with its bias.  (Loads by the compute threads, LDGSTS or
// LDG + STS, kept the prologue at 8-9 k cycles: ten loads per thread behind an index decode.)
__device__ __forceinline__ uint32_t small_bytes(const Cl& c, const NetShape& s) {
  return (uint32_t)((c.H * s.in + c.H + (s.layers - 1) * c.H + s.out * c.H + 4) * 4);
}
__device__ __forceinline__ void small_issue(const Cl& c, int slot, const float* __restrict__ P, const NetShape& s, int item) {
  float* sp = smem_f + c.small + slot * c.small_stride;
  uint64_t* bar = cl_bar(c, 8);
  if (item == 0) bulk_g2s(sp, P, (uint32_t)((c.H * s.in + c.H) * 4), bar);
  else if (item < s.layers) bulk_g2s(sp + (4 + item) * c.H, P + net_b_off(s, item), (uint32_t)(c.H * 4), bar);
  else if (item == s.layers) bulk_g2s(sp + (4 + s.layers) * c.H, P + net_w_off(s, s.layers), (uint32_t)((s.out * c.H + 4) * 4), bar);
}
__device__ __forceinline__ int sp_w0(const Cl& c, int slot) { return c.small + slot * c.small_stride; }
__device__ __forceinline__ int sp_b0(const Cl& c, int slot, int in_dim) { return c.small + slot * c.small_stride + in_dim * c.H; }
// own slice of b_l, l >= 1
__device__ __forceinline__ int sp_bias(const Cl& c, int slot, int l) { return c.small + slot * c.small_stride + (4 + l) * c.H + c.c_lo; }
// head [out][H], its bias right behind it
__device__ __forceinline__ int sp_head(const Cl& c, int slot) { return c.small + slot * c.small_stride + (4 + c.L) * c.H; }

// the dz tile the next pushed output goes to (they alternate: consecutive stages never write the same tile)
__device__ __forceinline__ int next_dz(Cl& c) {
  const int r = c.dsel ? c.dz1 : c.dz0;
  c.dsel ^= 1;
  return r;
}

// The start barrier (every CTA of the cluster runs and has initialised its mbarriers) is only needed before the first store into a
// peer's shared memory: the threads arrive at kernel start and wait here, a first layer and a product later.
__device__ __forceinline__ void ensure_started(Cl& c) {
  if (!c.started) {
    cluster_wait();
    c.started = 1;
  }
}

// ---- stages ------------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t stage_bar(const Cl& c) { return smem_u32(smem_f + c.bar) + 8u * (uint32_t)(c.stg & 1); }
// four own values (columns c_lo + cc .. +3 of row r) into tile Y of every CTA of the cluster
template <int CS>
__device__ __forceinline__ void push4(const Cl& c, int off, const float4& v) {
  const uint32_t own = smem_u32(smem_f + off), bar = stage_bar(c);
#pragma unroll
  for (int k = 0; k < CS; ++k) st_async4(map_to_rank(own, (uint32_t)k), v, map_to_rank(bar, (uint32_t)k));
}
template <int CS>
__device__ __forceinline__ void push2(const Cl& c, int off, float a, float b) {
  const uint32_t own = smem_u32(smem_f + off), bar = stage_bar(c);
#pragma unroll
  for (int k = 0; k < CS; ++k) st_async2(map_to_rank(own, (uint32_t)k), a, b, map_to_rank(bar, (uint32_t)k));
}
// wait until the `bytes` all CTAs push to this one in the current stage have landed
__device__ __forceinline__ void stage_wait(Cl& c, uint32_t bytes) {
  const uint32_t bar = stage_bar(c);
  if (threadIdx.x == 0) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
  mbar_wait_cluster(bar, (uint32_t)((c.stg >> 1) & 1));
  c.stg += 1;
}
// [R][2] partial sums of every CTA -> all CTAs (slot [rank]), summed in rank order into dst[r * dstride + {0,1}] (+ bias).
// exchange_finish: the pushes of this CTA (push2 into buf + (rank * R + r) * 2) have been issued by whichever threads held the sums.
template <int R, int CS>
__device__ __forceinline__ void exchange_finish(Cl& c, int buf, int dst, int dstride, float bias0, float bias1) {
  const int t = threadIdx.x;
  stage_wait(c, (uint32_t)(CS * R * 8));
  if (t < R) {
    float x = 0.f, y = 0.f;
#pragma unroll
    for (int k = 0; k < CS; ++k) { x += smem_f[buf + (k * R + t) * 2]; y += smem_f[buf + (k * R + t) * 2 + 1]; }
    smem_f[dst + t * dstride] = x + bias0;
    smem_f[dst + t * dstride + 1] = y + bias1;
  }
  cta_sync();
}
template <int R, int CS>
__device__ __forceinline__ void exchange_pairs(Cl& c, int buf, float a, float b, int dst, int dstride, float bias0, float bias1) {
  if (threadIdx.x < R) push2<CS>(c, buf + (c.rank * R + threadIdx.x) * 2, a, b);
  exchange_finish<R, CS>(c, buf, dst, dstride, bias0, bias1);
}

// ---- first layer, ALL columns, every CTA: h[r][c] = relu(b[c] + sum_j in0[r][j] * W0[c][j]) -------------------------------------------
template <int R>
__device__ __forceinline__ void cl_first(Cl& c, int slot, int in_dim, int Y, float* __restrict__ gh /*nullable [B][H]*/, int r0, int B) {
  const int w0 = sp_w0(c, slot), bb = sp_b0(c, slot, in_dim);
  for (int col = threadIdx.x; col < c.H; col += kCT) {
    float w[4] = {0.f, 0.f, 0.f, 0.f};
    if (in_dim == 4) {
      const float4 q = lds4(w0 + col * 4);
      w[0] = q.x; w[1] = q.y; w[2] = q.z; w[3] = q.w;
    } else {
      const float2 q = *reinterpret_cast<const float2*>(smem_f + w0 + col * 2);
      w[0] = q.x; w[1] = q.y;
    }
    const float bias = smem_f[bb + col];
    const bool own = gh && col >= c.c_lo && col < c.c_lo + c.ncols;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const float4 x = lds4(c.in0 + r * 4);
      float v = bias;
      v = fmaf(x.x, w[0], v); v = fmaf(x.y, w[1], v); v = fmaf(x.z, w[2], v); v = fmaf(x.w, w[3], v);
      v = fmaxf(v, 0.f);
      smem_f[Y + r * c.ld + col] = v;
      if (own && r0 + r < B) gh[(int64_t)(r0 + r) * c.H + col] = v;
    }
  }
  stamp(c, 10);
}

// ---- hidden product, own columns: red[g][r][c] = sum_{j in group g} X[r][j] * T[c][j] ------------------------------------------------
// thread = (reduction group, row group rg, column group cl); it owns rows rg, rg + RG, rg + 2 RG, rg + 3 RG (neighbouring row groups
// read neighbouring rows: with ld = H + 4 their float4 fall into different banks) and the 4 columns of tile group cl
// (inlined into the forward and the backward pass: one shared __noinline__ copy was measured - 15 % of the kernel's stall samples are
// instruction fetches - and was slower, 2.9-3.5 k cycles per product against 2.5 k)
template <int R>
__device__ __forceinline__ void cl_product_impl(int T, int X, int H, int ld, int Wc, int ncols, int ncg_sh, int part, int red) {
  constexpr int RG = R / 4;
  const int t = threadIdx.x;
  const int cl = t & ((1 << ncg_sh) - 1);
  const int rg = (t >> ncg_sh) % RG;
  const int kg = (t >> ncg_sh) / RG;
  const int jlo = kg * part, jhi = min(H, jlo + part);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { acc[i][0] = 0.f; acc[i][1] = 0.f; acc[i][2] = 0.f; acc[i][3] = 0.f; }
  if (4 * cl < ncols) {
    const int tw = T + cl * (4 * H + 4), xr = X + rg * ld;
#pragma unroll 2
    for (int j = jlo; j < jhi; j += 4) {
      float4 w[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) w[e] = lds4(tw + e * H + j);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 x = lds4(xr + i * RG * ld + j);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          acc[i][e] = fmaf(x.x, w[e].x, acc[i][e]); acc[i][e] = fmaf(x.y, w[e].y, acc[i][e]);
          acc[i][e] = fmaf(x.z, w[e].z, acc[i][e]); acc[i][e] = fmaf(x.w, w[e].w, acc[i][e]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(smem_f + red + (kg * R + rg + i * RG) * Wc + 4 * cl) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
  cta_sync();
}
template <int R>
__device__ __forceinline__ void cl_product(const Cl& c, int T, int X) {
  cl_product_impl<R>(T, X, c.H, c.ld, c.Wc, c.ncols, c.ncg_sh, c.part, c.red);
}

// sum of the partials of the four values (r, cc..cc+3)
template <int R>
__device__ __forceinline__ float4 cl_reduce4(const Cl& c, int r, int cc) {
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int g = 0; g < c.kgn; ++g) {
    const float4 p = lds4(c.red + (g * R + r) * c.Wc + cc);
    v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
  }
  return v;
}

// ---- hidden layer forward: Y[r][c] = relu(b[c] + sum_k X[r][k] * Wt[k][c]), own columns ------------------------------------------------
// not the last hidden layer: the slice is pushed into tile Y of the whole cluster (the next product reduces over all columns).
// The last one: kept locally when `Ykeep` >= 0 (the backward pass masks with it), and its contribution to the head goes out instead:
// out[r][o] = b[o] + sum over the CTAs (in rank order) of sum_{c own} h[r][c] * Wout[o][c].
template <int R, int CS>
__device__ __forceinline__ void cl_fwd_hidden(Cl& c, int ti, int T, int slot, int l, bool last, int X, int Y, int out_dim, float* __restrict__ gh, int r0,
                                              int B) {
  stamp(c, 20);
  cl_product<R>(c, T, X);
  tile_release(c, ti);
  stamp(c, 21);
  ensure_started(c);
  const int q = c.ncols >> 2, bb = sp_bias(c, slot, l), hd = sp_head(c, slot);
  // 16 column groups and all rows in one sweep: the 16 threads of a row are half a warp and add their head contributions by shuffles
  const bool fast = last && q == 16 && R * 16 <= kCT;
  for (int idx = threadIdx.x; idx < R * q; idx += kCT) {
    const int r = idx / q, cg = idx - r * q, cc = cg * 4;
    const float4 p = cl_reduce4<R>(c, r, cc);
    const float4 b = lds4(bb + cc);
    const float4 o = make_float4(fmaxf(b.x + p.x, 0.f), fmaxf(b.y + p.y, 0.f), fmaxf(b.z + p.z, 0.f), fmaxf(b.w + p.w, 0.f));
    if (!last) push4<CS>(c, Y + r * c.ld + c.c_lo + cc, o);
    else {
      if (Y >= 0) *reinterpret_cast<float4*>(smem_f + Y + r * c.ld + c.c_lo + cc) = o;
      const float4 wa = lds4(hd + c.c_lo + cc);
      float h0 = o.x * wa.x;
      h0 = fmaf(o.y, wa.y, h0); h0 = fmaf(o.z, wa.z, h0); h0 = fmaf(o.w, wa.w, h0);
      float h1 = 0.f;
      if (out_dim > 1) {
        const float4 wb = lds4(hd + c.H + c.c_lo + cc);
        h1 = o.x * wb.x;
        h1 = fmaf(o.y, wb.y, h1); h1 = fmaf(o.z, wb.z, h1); h1 = fmaf(o.w, wb.w, h1);
      }
      if (fast) {                                            // (whole warps run this branch: idx < R * 16 is a multiple of 32)
#pragma unroll
        for (int sft = 8; sft > 0; sft >>= 1) {
          h0 += __shfl_xor_sync(0xffffffffu, h0, sft);
          h1 += __shfl_xor_sync(0xffffffffu, h1, sft);
        }
        if (cg == 0) push2<CS>(c, c.hp + (c.rank * R + r) * 2, h0, h1);
      } else {
        *reinterpret_cast<float2*>(smem_f + c.hpart + idx * 2) = make_float2(h0, h1);
      }
    }
    if (gh && r0 + r < B) *reinterpret_cast<float4*>(gh + (int64_t)(r0 + r) * c.H + c.c_lo + cc) = o;
  }
  stamp(c, 22);
  if (!last) {
    stage_wait(c, (uint32_t)(R * c.H * 4));
    stamp(c, 23);
  } else {
    const float bias0 = smem_f[hd + out_dim * c.H], bias1 = out_dim > 1 ? smem_f[hd + out_dim * c.H + 1] : 0.f;
    if (!fast) {
      cta_sync();
      float a = 0.f, b2 = 0.f;
      if (threadIdx.x < R) {
        for (int g = 0; g < q; ++g) {
          const float2 v = *reinterpret_cast<const float2*>(smem_f + c.hpart + (threadIdx.x * q + g) * 2);
          a += v.x; b2 += v.y;
        }
        push2<CS>(c, c.hp + (c.rank * R + threadIdx.x) * 2, a, b2);
      }
    }
    exchange_finish<R, CS>(c, c.hp, c.out, 2, bias0, bias1);
    stamp(c, 30);
  }
}

// forward pass of one network.  keep: activations stay in act(keep0 + l) for the backward pass.
template <int R, int CS>
__device__ __forceinline__ void cl_forward(Cl& c, int slot, const NetShape& s, bool keep, int keep0, const RowScratch* rs, int r0, int& ti) {
  const int B = rs ? rs->B : 0;
  int x = keep ? c.act0 + keep0 * R * c.ld : c.xl;
  cl_first<R>(c, slot, s.in, x, rs ? rs->h(0) : nullptr, r0, B);
  if (s.layers == 1) {
    // the head straight from the first layer (every CTA holds all of it): own columns' contribution, exchanged like any other
    cta_sync();
    const int hd = sp_head(c, slot);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int p = warp; p < R * 2; p += kCT / 32) {
      const int r = p >> 1, o = p & 1;
      float v = 0.f;
      if (o < s.out)
        for (int cc = lane; cc < c.ncols; cc += 32) v = fmaf(smem_f[x + r * c.ld + c.c_lo + cc], smem_f[hd + o * c.H + c.c_lo + cc], v);
      v = warp_sum(v);
      if (lane == 0) smem_f[c.din + r * 4 + o] = v;          // din doubles as scratch here (the backward pass writes it later)
    }
    cta_sync();
    ensure_started(c);
    const float a = threadIdx.x < R ? smem_f[c.din + threadIdx.x * 4] : 0.f, b2 = threadIdx.x < R ? smem_f[c.din + threadIdx.x * 4 + 1] : 0.f;
    exchange_pairs<R, CS>(c, c.hp, a, b2, c.out, 2, smem_f[hd + s.out * c.H], s.out > 1 ? smem_f[hd + s.out * c.H + 1] : 0.f);
    return;
  }
  for (int l = 1; l < s.layers; ++l) {
    const bool last = l == s.layers - 1;
    const int y = keep ? c.act0 + (keep0 + l) * R * c.ld : (last ? -1 : next_dz(c));
    const int T = tile_acquire(c, ti);
    cl_fwd_hidden<R, CS>(c, ti, T, slot, l, last, x, y, s.out, rs ? rs->h(l) : nullptr, r0, B);
    ++ti;
    x = y;
  }
}

// ---- backward (pre-activation gradients; the parameter gradients are wgrad_kernel's) ---------------------------------------------
// dz_{L-1}[r][k] = relu'(h_{L-1}[r][k]) * sum_o dout[r][o] * Wout[o][k], own columns -> all CTAs (the next product reduces over it)
// dz_{l-1}[r][k] = relu'(h_{l-1}[r][k]) * sum_n dz_l[r][n] * W_l[n][k]
// want_din: din[r][j] = sum_c dz_0[r][c] * W0[c][j] (partials over own columns, summed over the cluster in rank order)
template <int R, int CS>
__device__ __forceinline__ void cl_backward(Cl& c, int slot, const NetShape& s, int keep0, const RowScratch* rs, int r0, bool want_din, int& ti) {
  const int L = s.layers, B = rs ? rs->B : 0;
  const int t = threadIdx.x;
  if (rs && c.rank == 0 && t < R && r0 + t < B) {
    *reinterpret_cast<float4*>(rs->in0() + (int64_t)(r0 + t) * 4) = lds4(c.in0 + t * 4);
    *reinterpret_cast<float2*>(rs->dout() + (int64_t)(r0 + t) * 2) = *reinterpret_cast<const float2*>(smem_f + c.dout + t * 2);
  }
  const int q = c.ncols >> 2;
  int cur = L > 1 ? next_dz(c) : c.xl;                 // a single hidden layer: dz_0 is only read back by this CTA (want_din)
  {
    const bool push = L > 1;                          // a product reduces over it
    const int hd = sp_head(c, slot), Hl = c.act0 + (keep0 + L - 1) * R * c.ld;
    float* g = rs ? rs->dz(L - 1) : nullptr;
    for (int idx = t; idx < R * q; idx += kCT) {
      const int r = idx / q, cc = (idx - r * q) * 4, k = c.c_lo + cc;
      const float d0 = smem_f[c.dout + r * 2], d1 = smem_f[c.dout + r * 2 + 1];
      const float4 wa = lds4(hd + k), h = lds4(Hl + r * c.ld + k);
      const float4 wb = s.out > 1 ? lds4(hd + c.H + k) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 o;
      o.x = h.x > 0.f ? fmaf(d0, wa.x, d1 * wb.x) : 0.f;
      o.y = h.y > 0.f ? fmaf(d0, wa.y, d1 * wb.y) : 0.f;
      o.z = h.z > 0.f ? fmaf(d0, wa.z, d1 * wb.z) : 0.f;
      o.w = h.w > 0.f ? fmaf(d0, wa.w, d1 * wb.w) : 0.f;
      if (push) push4<CS>(c, cur + r * c.ld + k, o);
      else *reinterpret_cast<float4*>(smem_f + cur + r * c.ld + k) = o;
      if (g && r0 + r < B) *reinterpret_cast<float4*>(g + (int64_t)(r0 + r) * c.H + k) = o;
    }
    stamp(c, 40);
    if (push) stage_wait(c, (uint32_t)(R * c.H * 4)); else cta_sync();
    stamp(c, 41);
  }
  for (int l = L - 1; l >= 1; --l) {
    const int T = tile_acquire(c, ti);
    stamp(c, 50);
    cl_product<R>(c, T, cur);
    tile_release(c, ti);
    ++ti;
    stamp(c, 51);
    const bool push = l - 1 >= 1;                    // another product follows
    const int nxt = push ? next_dz(c) : c.xl;
    const int Hp = c.act0 + (keep0 + l - 1) * R * c.ld;
    float* g = rs ? rs->dz(l - 1) : nullptr;
    for (int idx = t; idx < R * q; idx += kCT) {
      const int r = idx / q, cc = (idx - r * q) * 4, k = c.c_lo + cc;
      const float4 p = cl_reduce4<R>(c, r, cc);
      const float4 h = lds4(Hp + r * c.ld + k);
      const float4 o = make_float4(h.x > 0.f ? p.x : 0.f, h.y > 0.f ? p.y : 0.f, h.z > 0.f ? p.z : 0.f, h.w > 0.f ? p.w : 0.f);
      if (push) push4<CS>(c, nxt + r * c.ld + k, o);
      else if (want_din) *reinterpret_cast<float4*>(smem_f + nxt + r * c.ld + k) = o;
      if (g && r0 + r < B) *reinterpret_cast<float4*>(g + (int64_t)(r0 + r) * c.H + k) = o;
    }
    stamp(c, 52);
    if (push) stage_wait(c, (uint32_t)(R * c.H * 4)); else cta_sync();
    stamp(c, 53);
    cur = nxt;
  }
  if (want_din) {
    // partial over own columns: one warp per (r, j); only the action components j = 2, 3 are used (robot.py:386-391)
    const int warp = t >> 5, lane = t & 31;
    const int w0 = sp_w0(c, slot);
    for (int p = warp; p < R * 2; p += kCT / 32) {
      const int r = p >> 1, j = 2 + (p & 1);
      float v = 0.f;
      for (int cc = lane; cc < c.ncols; cc += 32) v = fmaf(smem_f[cur + r * c.ld + c.c_lo + cc], smem_f[w0 + (c.c_lo + cc) * 4 + j], v);
      v = warp_sum(v);
      if (lane == 0) smem_f[c.din + r * 4 + j] = v;
    }
    cta_sync();
    const float a = t < R ? smem_f[c.din + t * 4 + 2] : 0.f, b2 = t < R ? smem_f[c.din + t * 4 + 3] : 0.f;
    exchange_pairs<R, CS>(c, c.dinp, a, b2, c.din + 2, 4, 0.f, 0.f);
    stamp(c, 60);
  }
}

constexpr int kMaxTiles = 7 * (kMaxLayers - 1) + 4;      // critic step: 7 (L-1) tiles

// producer warp, first thing in the kernel: its own barrier and the small-parameter copies (their latency runs under the set-up of
// the other threads; the compute threads meet barrier 8 only after the CTA barrier of cl_begin)
template <typename IssueFn>
__device__ __forceinline__ void small_begin(const Cl& c, uint32_t bytes, int items, IssueFn&& issue) {
  const int lane = threadIdx.x - kCT;
  if (lane == 0) {
    mbar_init(cl_bar(c, 8), 1);
    fence_mbar_init();
    mbar_arrive_expect_tx(cl_bar(c, 8), bytes);
  }
  __syncwarp();
  for (int w = lane; w < items; w += 32) issue(w);
}

// common start (all threads of the CTA): the mbarriers.  Ends with a CTA barrier.
__device__ __forceinline__ void cl_begin(Cl& c) {
  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(cl_bar(c, i), 1);     // (barrier 8 is the producer warp's: see small_begin)
    fence_mbar_init();
  }
  __syncthreads();
}
// compute threads: the small parameters have landed; every CTA of the cluster runs and has its mbarriers set up
__device__ __forceinline__ void cl_started(Cl& c) {
  cluster_arrive();                  // waited for in ensure_started()
  mbar_wait(cl_bar(c, 8), 0);
  stamp(c, 1);
  cta_sync();                        // the replay rows gathered by the first R threads
  stamp(c, 2);
}

// ---- critic phase (robot.py:312-366 up to the optimiser steps); see td3_critic_kernel for the arithmetic ---------------------------
template <int R, int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(kClBlock, 1)
td3_critic_cluster_kernel(Arena ar, const float* __restrict__ params, const float* __restrict__ params_t, float* __restrict__ scratch, ReplayView rp,
                          const int32_t* __restrict__ idx, const float* __restrict__ noise, int B, Td3Hyper hp, float* __restrict__ loss,
                          float* __restrict__ q_out, float* __restrict__ y_out, int32_t* __restrict__ steps, double* __restrict__ beta_pows, int ns,
                          long long* prof) {
  Cl c;
  const int L = ar.critic.layers;
  cl_carve(c, R, CS, ar.critic.hid, L, ns, 5, L);
  if (blockIdx.x == 0) c.prof = prof;
  stamp(c, 0);
  const int r0 = (int)cluster_id_x() * R;
  const int t = threadIdx.x;

  const int j_row = (t < R && r0 + t < B) ? idx[r0 + t] : 0;      // replay row of this thread's batch row (its loads follow below)
  // weight tiles in the order of use: passes 0-2 forward, passes 3-4 forward then backward
  __shared__ const float* tiles[kMaxTiles];
  if (t < kMaxTiles) {
    const int n = L - 1;
    const float* p = nullptr;
    if (n > 0 && t < 7 * n) {
      int pass, l;
      bool bwd = false;
      if (t < 3 * n) { pass = t / n; l = 1 + t % n; }
      else {
        const int j = t - 3 * n;
        pass = 3 + j / (2 * n);
        const int jj = j % (2 * n);
        bwd = jj >= n;
        l = bwd ? (L - 1 - (jj - n)) : 1 + jj;
      }
      const int net = pass == 0 ? 3 : (pass == 1 ? 4 : (pass == 2 ? 5 : pass - 2));
      p = (bwd ? params_t : params) + ar.off(net) + net_w_off(pass == 0 ? ar.actor : ar.critic, l);
    }
    tiles[t] = p;
  }
  if (t >= kCT)                          // small parameters of the five passes: work item = (pass, copy)
    small_begin(c, small_bytes(c, ar.actor) + 4u * small_bytes(c, ar.critic), 5 * (L + 1), [&](int w) {
      const int pass = w / (L + 1), net = pass < 3 ? pass + 3 : pass - 2;
      small_issue(c, pass, params + ar.off(net), pass == 0 ? ar.actor : ar.critic, w - pass * (L + 1));
    });
  cl_begin(c);
  stamp(c, 3);
  if (t >= kCT) {                        // producer warp: weight tiles, in the order of use
    cluster_arrive();                                      // its share of the start barrier first: nobody waits for its copies to be issued
    cl_producer(c, tiles, 0, min(c.ns, 7 * (L - 1)));      // the first tiles need no free slot; then join the start barrier
    if (blockIdx.x == 0 && t == kCT) advance_adam_clock(steps, beta_pows, 1);   // (read by the optimiser kernel that follows)
    cluster_wait();
    cl_producer(c, tiles, c.ns, 7 * (L - 1));
    cluster_sync();
    return;
  }
  stamp(c, 4);
  float* S = smem_f + c.S;       // [R][8]: 0 s.x 1 s.y 2 a.x 3 a.y 4 reward 5 notdone 6 y 7 valid
  float* in0 = smem_f + c.in0;
  float* out = smem_f + c.out;
  float* dout = smem_f + c.dout;
  float2 zn = make_float2(0.f, 0.f);     // this row's smoothing noise (Philox + log + sincos: off the chain between the passes)
  if (t < R) {
    zn = target_noise(noise, hp, min(r0 + t, B - 1));
    const int row = r0 + t;
    const bool valid = row < B;
    const int j = j_row;
    const float2 s = rp.s[j], a = rp.a[j], s2 = rp.s2[j];
    S[t * 8 + 0] = s.x; S[t * 8 + 1] = s.y; S[t * 8 + 2] = a.x; S[t * 8 + 3] = a.y;
    S[t * 8 + 4] = rp.r[j]; S[t * 8 + 5] = rp.notdone[j]; S[t * 8 + 7] = valid ? 1.f : 0.f;
    in0[t * 4 + 0] = s2.x; in0[t * 4 + 1] = s2.y; in0[t * 4 + 2] = 0.f; in0[t * 4 + 3] = 0.f;
  }
  stamp(c, 5);
  cl_started(c);

  int ti = 0;
#pragma unroll 1
  for (int pass = 0; pass < 5; ++pass) {
    const NetShape shape = pass == 0 ? ar.actor : ar.critic;
    const bool train = pass >= 3;
    RowScratch rs{scratch + (train ? (pass - 3) : 0) * RowScratch::floats(B, ar.critic.hid, L), B, ar.critic.hid, L};
    cl_forward<R, CS>(c, pass, shape, train, 0, train ? &rs : nullptr, r0, ti);
    if (t < R) {
      if (pass == 0) {                                   // smoothing noise and clips (robot.py:338-339)
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
        if (y_out && c.rank == 0 && r0 + t < B) y_out[r0 + t] = y;
        in0[t * 4 + 0] = S[t * 8 + 0]; in0[t * 4 + 1] = S[t * 8 + 1];
        in0[t * 4 + 2] = S[t * 8 + 2]; in0[t * 4 + 3] = S[t * 8 + 3];
      } else {                                           // MSE loss and its gradient (robot.py:348-353)
        const int cr = pass - 3;
        const float valid = S[t * 8 + 7];
        const float q = out[t * 2];
        const float diff = (q - S[t * 8 + 6]) * valid;
        dout[t * 2] = 2.0f * diff / (float)B;
        dout[t * 2 + 1] = 0.f;
        if (q_out && c.rank == 0 && valid != 0.f) q_out[cr * B + r0 + t] = q;
        float l = diff * diff / (float)B;                // this row's share of the mean
#pragma unroll
        for (int o = R / 2; o > 0; o >>= 1) l += __shfl_xor_sync((R >= 32) ? 0xffffffffu : ((1u << R) - 1u), l, o);
        if (t == 0 && c.rank == 0) atomicAdd(loss + cr, l);
      }
    }
    cta_sync();
    if (train) cl_backward<R, CS>(c, pass, shape, 0, &rs, r0, false, ti);
  }
  stamp(c, 98);
  cluster_sync();        // no CTA leaves while stores of its peers may still be on their way to it
  stamp(c, 99);
  if (c.prof && t == 0) c.prof[0] = c.pn;
}

// ---- actor phase (robot.py:369-398 up to the optimiser step) ----------------------------------------------------------------------
template <int R, int CS>
__global__ void __cluster_dims__(CS, 1, 1) __launch_bounds__(kClBlock, 1)
td3_actor_cluster_kernel(Arena ar, const float* __restrict__ params, const float* __restrict__ params_t, float* __restrict__ scratch, ReplayView rp,
                         const int32_t* __restrict__ idx, int B, float* __restrict__ loss, int32_t* __restrict__ steps, double* __restrict__ beta_pows,
                         int ns, long long* prof) {
  Cl c;
  const int L = ar.critic.layers;
  cl_carve(c, R, CS, ar.critic.hid, L, ns, 2, 2 * L);
  if (blockIdx.x == 0) c.prof = prof;
  stamp(c, 0);
  const int r0 = (int)cluster_id_x() * R;
  const int t = threadIdx.x;
  __shared__ const float* tiles[kMaxTiles];
  if (t < kMaxTiles) {
    const int n = L - 1;
    const float* p = nullptr;
    if (n > 0 && t < 4 * n) {
      const int seg = t / n, j = t % n;          // 0 actor forward, 1 critic forward, 2 critic backward, 3 actor backward
      const int net = (seg == 0 || seg == 3) ? 0 : 1;
      const int l = seg < 2 ? 1 + j : L - 1 - j;
      p = (seg < 2 ? params : params_t) + ar.off(net) + net_w_off(net == 0 ? ar.actor : ar.critic, l);
    }
    tiles[t] = p;
  }
  if (t >= kCT)
    small_begin(c, small_bytes(c, ar.actor) + small_bytes(c, ar.critic), 2 * (L + 1), [&](int w) {
      const int pass = w / (L + 1);
      small_issue(c, pass, params + ar.off(pass), pass == 0 ? ar.actor : ar.critic, w - pass * (L + 1));
    });
  cl_begin(c);
  if (t >= kCT) {
    cluster_arrive();
    cl_producer(c, tiles, 0, min(c.ns, 4 * (L - 1)));
    if (blockIdx.x == 0 && t == kCT) advance_adam_clock(steps, beta_pows, 0);
    cluster_wait();
    cl_producer(c, tiles, c.ns, 4 * (L - 1));
    cluster_sync();
    return;
  }
  float* S = smem_f + c.S;
  float* in0 = smem_f + c.in0;
  RowScratch rs{scratch, B, ar.actor.hid, ar.actor.layers};
  if (t < R) {
    const int row = r0 + t;
    const bool valid = row < B;
    const float2 s = rp.s[valid ? idx[row] : 0];
    in0[t * 4 + 0] = s.x; in0[t * 4 + 1] = s.y; in0[t * 4 + 2] = 0.f; in0[t * 4 + 3] = 0.f;
    S[t * 8 + 7] = valid ? 1.f : 0.f;
  }
  cl_started(c);

  int ti = 0;
  // forward: a = pi(s) (fed the raw replay state, robot.py:386), then Q1(s, a).  The two passes are iterations of ONE loop (and so are
  // the two backward passes): every inlined copy of the layer code costs instruction-cache misses that a kernel of ~30 us does not amortise
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    cl_forward<R, CS>(c, pass, pass == 0 ? ar.actor : ar.critic, true, pass == 0 ? 0 : L, pass == 0 ? &rs : nullptr, r0, ti);
    if (t < R) {
      if (pass == 0) {
        in0[t * 4 + 2] = smem_f[c.out + t * 2];
        in0[t * 4 + 3] = smem_f[c.out + t * 2 + 1];
      } else {
        const float valid = S[t * 8 + 7];
        smem_f[c.dout + t * 2] = -valid / (float)B;
        smem_f[c.dout + t * 2 + 1] = 0.f;
        float l = -smem_f[c.out + t * 2] * valid / (float)B;
#pragma unroll
        for (int o = R / 2; o > 0; o >>= 1) l += __shfl_xor_sync((R >= 32) ? 0xffffffffu : ((1u << R) - 1u), l, o);
        if (t == 0 && c.rank == 0) atomicAdd(loss, l);
      }
    }
    cta_sync();
  }
  // backward through critic 1 (only dQ/d(action) is needed), then through the actor
#pragma unroll 1
  for (int pass = 0; pass < 2; ++pass) {
    cl_backward<R, CS>(c, 1 - pass, pass == 0 ? ar.critic : ar.actor, pass == 0 ? L : 0, pass == 0 ? nullptr : &rs, r0, pass == 0, ti);
    if (pass == 0) {
      if (t < R) {
        smem_f[c.dout + t * 2] = smem_f[c.din + t * 4 + 2];
        smem_f[c.dout + t * 2 + 1] = smem_f[c.din + t * 4 + 3];
        // cl_backward stores in0 of the network it differentiates: the actor's input was (s, 0, 0)
        in0[t * 4 + 2] = 0.f; in0[t * 4 + 3] = 0.f;
      }
      cta_sync();
    }
  }
  stamp(c, 98);
  cluster_sync();
  stamp(c, 99);
  if (c.prof && t == 0) c.prof[0] = c.pn;
}

}  // namespace rtd3

using namespace rtd3;

namespace {
int g_mode = 2;   // rtd3_debug_cluster_mode: 0 = never, 2 = wherever the plan fits and the batch is one wave of clusters
// clusters of 4 with 8 rows: 32 clusters for the benchmark batch of 256 (the device holds 33 of them at once, but only 15 clusters
// of 8); larger batches run in several waves (16 rows per cluster do not fit the shared memory next to two 64 KB weight tiles)
constexpr int kClR = 8, kClCS = 4;
long long* g_prof[2] = {nullptr, nullptr};   // development: stamp buffers of the critic / actor kernels (rtd3_debug_cluster_prof)
}  // namespace

// The cluster kernels win while the batch is ONE wave of clusters (B = 256: 32 of the 33 clusters a B200 holds; 47.9 against 77.5 us
// per epoch); from the second wave on the row-tile kernels are faster again (B = 512: 88.4 against 83.9, B = 1024: 171.8 against
// 120.7 us per epoch), so larger batches keep them.
bool rtd3::cluster_path_ok(const rtd3_td3* h, int batch) {
  if (g_mode == 0) return false;
  const int H = h->ar.critic.hid, L = h->ar.critic.layers;
  if (H % 4 != 0 || H < 4) return false;
  if (make_plan(kClR, kClCS, H, L, 5, L).bytes > kClSmemLimit || make_plan(kClR, kClCS, H, L, 2, 2 * L).bytes > kClSmemLimit) return false;
  return ceil_div(batch, kClR) <= h->cluster_cap;
}

int32_t rtd3::critic_cluster_launch(rtd3_td3* h, const float* params, const float* params_t, float* scratch, const ReplayView& rp, const int32_t* idx,
                                    const float* noise, int32_t batch, const Td3Hyper& hp, float* loss2, float* q_out, float* y_out, int32_t* steps,
                                    double* beta_pows, cudaStream_t st) {
  const int H = h->ar.critic.hid, L = h->ar.critic.layers;
  const ClPlan p = make_plan(kClR, kClCS, H, L, 5, L);
  const int grid = (int)ceil_div(batch, kClR) * kClCS;
  auto* fn = td3_critic_cluster_kernel<kClR, kClCS>;
  RTD3_CUDA(ensure_dyn_smem((const void*)fn, p.bytes));
  fn<<<grid, kClBlock, p.bytes, st>>>(h->ar, params, params_t, scratch, rp, idx, noise, batch, hp, loss2, q_out, y_out, steps, beta_pows, p.ns,
                                      g_prof[0]);
  RTD3_LAUNCHED();
  return 0;
}

int32_t rtd3::actor_cluster_launch(rtd3_td3* h, const float* params, const float* params_t, float* scratch, const ReplayView& rp, const int32_t* idx,
                                   int32_t batch, float* loss1, int32_t* steps, double* beta_pows, cudaStream_t st) {
  const int H = h->ar.critic.hid, L = h->ar.critic.layers;
  const ClPlan p = make_plan(kClR, kClCS, H, L, 2, 2 * L);
  const int grid = (int)ceil_div(batch, kClR) * kClCS;
  auto* fn = td3_actor_cluster_kernel<kClR, kClCS>;
  RTD3_CUDA(ensure_dyn_smem((const void*)fn, p.bytes));
  fn<<<grid, kClBlock, p.bytes, st>>>(h->ar, params, params_t, scratch, rp, idx, batch, loss1, steps, beta_pows, p.ns, g_prof[1]);
  RTD3_LAUNCHED();
  return 0;
}

extern "C" {

int32_t rtd3_td3_cluster_supported(const rtd3_td3* h, int32_t batch) { return (h && batch > 0 && rtd3::cluster_path_ok(h, batch)) ? 1 : 0; }

int32_t rtd3_td3_cluster_occupancy(const rtd3_td3* h, int32_t batch) {
  if (!h || batch <= 0) return -1;
  const int H = h->ar.critic.hid, L = h->ar.critic.layers;
  const ClPlan p = make_plan(kClR, kClCS, H, L, 5, L);
  if (H % 4 != 0 || H < 4 || p.bytes > kClSmemLimit || make_plan(kClR, kClCS, H, L, 2, 2 * L).bytes > kClSmemLimit) return 0;   // no plan: no clusters
  auto* fn = td3_critic_cluster_kernel<kClR, kClCS>;
  if (ensure_dyn_smem((const void*)fn, p.bytes) != cudaSuccess) { (void)cudaGetLastError(); return -2; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ceil_div(batch, kClR) * kClCS), 1, 1);
  cfg.blockDim = dim3(kClBlock, 1, 1);
  cfg.dynamicSmemBytes = p.bytes;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeClusterDimension;
  attr.val.clusterDim.x = (unsigned)kClCS; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  int n = 0;
  const cudaError_t e = cudaOccupancyMaxActiveClusters(&n, fn, &cfg);
  if (e != cudaSuccess) { (void)cudaGetLastError(); rtd3::set_error("cudaOccupancyMaxActiveClusters: %s", cudaGetErrorString(e)); return -3; }
  return n;
}

int32_t rtd3_debug_cluster_mode(int32_t mode) {
  const int prev = g_mode;
  if (mode == 0 || mode == 2) g_mode = mode;
  return prev;
}

int32_t rtd3_debug_cluster_prof(long long* critic_buf, long long* actor_buf) {
  g_prof[0] = critic_buf;
  g_prof[1] = actor_buf;
  return 0;
}

}  // extern "C"
