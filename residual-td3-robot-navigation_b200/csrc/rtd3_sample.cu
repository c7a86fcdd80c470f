// ReplayBuffer.sample's index draw (robot.py:111): np.random.choice(len, B, replace=False) on a numpy-legacy
// MT19937 stream = the first B entries of a legacy Fisher-Yates shuffle of arange(len)
// (RandomState.shuffle: for i = len-1 .. 1: j = random_interval(i); swap(x[i], x[j])).  Bit-exact with numpy;
// `count` consecutive samples are drawn per call (a TD3 update needs 150 of them: robot.py:272-285).
//
// The shuffle looks serial, but only two small parts of it are:
//   1. which raw 32-bit draws are accepted by the masked rejection loop of random_interval - a chain through the
//      stream because the bound i drops by one per accepted draw.  One warp resolves 32 draws at a time: every lane
//      assumes a set of accepted lower lanes, derives its own bound, and the ballot is iterated to its fixed point
//      (lane L's decision depends only on lanes < L, so the fixed point is the sequential answer).
//   2. nothing else: the B outputs do not need the permutation.  Output p is found by walking the swap list
//      BACKWARDS from position p (pos==i -> j_i, pos==j_i -> i), independently per output and per sample.
// Kernel A (sample_swaps_pipelined_kernel, one CTA) writes the swap lists J[s][i]; kernel B (sample_trace_kernel, one CTA per sample)
// back-traces the B outputs.
#include "rtd3_common.cuh"
#include "rtd3_mt.cuh"

namespace rtd3 {

__device__ __forceinline__ uint32_t mt_twist(uint32_t cur, uint32_t nxt, uint32_t far) {
  const uint32_t y = (cur & 0x80000000u) | (nxt & 0x7fffffffu);
  return far ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

// ---- Kernel A: swap lists.  J[s*n + i] = j_i for i = 1..n-1 (entry 0 unused) --------------------------------------------------------
// A round takes up to 32 NW consecutive raw draws, consumer thread t owning draw t.  With i swaps still to draw, thread t's bound
// (i minus the number of accepted draws before it) lies in [i - t, i].  If the mask is the same at both ends the draw is classified
// without knowing the exact bound: v <= i - t  -> accepted whatever happened before ("sure"), v > i -> rejected, in between ->
// undecided (a band of at most t values out of >= 2^k, ~1 % of the draws); threads whose range crosses a power of two are undecided
// too.  The sure draws are ranked by ballot counts, the undecided ones resolved in stream order with their exact bounds, and the round
// ends early at the draw that completes a sample.
// A first, block-per-round form of this kernel (256 threads that also twisted the generator whenever a 624-word block ran out, and
// compacted the undecided draws for ONE resolver warp between block barriers) took 13.3 ms per 150 draws of 10 000 rows: ~1.3 us per
// round, 10 000 rounds.  This kernel is the same classification restructured around what made a round cost that much (8.75 ms):
//  * the generator runs in its OWN warps (threads 32 NW .. 32 NW + 255): they twist and temper block after block into a ring of six
//    624-word blocks (full / empty mbarriers), so a round never stops at the end of a block and never waits for a twist;
//  * ONE block barrier per round: before it, every warp publishes its count of sure draws and its undecided draws (value + sure
//    draws before it inside the warp); after it, EVERY warp resolves the undecided draws of the round with the ballot fixed point -
//    redundantly - instead of compaction, a resolver warp and three more barriers (a per-thread serial walk over them was tried
//    first: 2 000 of a round's 2 900 cycles);
//  * smaller rounds only at the lowest mask levels, where the undecided band is wide.
// Also tried, all bit-exact and all slower or equal:
//  (a) ONE consumer warp with eight consecutive draws per lane, every prefix from per-slot ballots, rounds cut at the mask level, no
//      block barrier at all - 27 ms: ~600 dependent instructions per lane and round on a single warp run at 4-6 cycles each, where
//      eight warps with one draw per lane and one barrier need 1 650 cycles;
//  (b) undecided draws that decide themselves from their exact interval [i - S - M, i - S] plus a second barrier for the counts, the
//      walk only for a truly undecided draw - 8.9 ms against 8.75: the walk was not what a round waits for;
//  (c) 16 consumer warps (512-draw rounds) - 12.2 ms against 8.75;
//  (d) in the block-per-round form, 1024-draw rounds over a ring of four generator states, so that no round stops at the end of a
//      624-word block: 14.1 ms against 13.3, and 16.0 with the round sized to keep ~32 draws undecided - the number of undecided
//      draws grows with the square of the round, and they were resolved by ONE warp; the serial resolver, not the round count, was
//      the floor.  And undecided draws decided block-parallel from their bound intervals [i - S - m, i - S] (the serial resolver then
//      ran only when a value fell inside its own window, ~never) with rounds of 2^(lvl-2) draws: 18.2 ms - a 1024-thread round costs
//      ~3 us against ~1.5 us for a 256-thread round and the low mask levels force small rounds either way.
// The block-per-round kernel and the 16-warp instantiation are in the tree at 8344fb3, the variants of (d) at 57e703c.
// The state written back is the un-tempered ring block the stream ended in.
constexpr int kRing = 6;
constexpr int kRingWords = kRing * RTD3_MT_N;

__device__ __forceinline__ uint32_t mt_untemper(uint32_t y) {
  y ^= y >> 18;
  y ^= (y << 15) & 0xefc60000u;                       // one round: the mask has no bit below 17
  uint32_t t = y;
  t = y ^ ((t << 7) & 0x9d2c5680u);
  t = y ^ ((t << 7) & 0x9d2c5680u);
  t = y ^ ((t << 7) & 0x9d2c5680u);
  t = y ^ ((t << 7) & 0x9d2c5680u);
  y = t;
  t = y ^ (y >> 11);
  t = y ^ (t >> 11);
  return t;
}

__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void bar_named(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

struct MaybeRec { int S; uint32_t rw; };

// NW consumer warps (a round takes up to 32 NW draws) + 8 generator warps
template <int NW>
__global__ void __launch_bounds__(NW * 32 + 256)
sample_swaps_pipelined_kernel(rtd3_mt_bank b, int64_t stream_id, int32_t n, int32_t count, int32_t* __restrict__ J) {
  constexpr int NC = NW * 32;
  __shared__ uint32_t mt[RTD3_MT_N], ring[kRingWords];
  __shared__ int w_cnt[2][NW];                        // per warp: sure draws | undecided draws << 16
  __shared__ MaybeRec mb[2][NW][32];
  __shared__ __align__(8) uint64_t full[kRing], empty[kRing];
  __shared__ volatile int s_done, s_last;
  __shared__ int s_gen_stop;                          // s_done as the generator's thread 0 read it before the generator barrier
  const int tid = threadIdx.x;
  for (int k = tid; k < RTD3_MT_N; k += NC + 256) mt[k] = b.mt[(int64_t)k * b.n + stream_id];
  const int pos0 = b.pos[stream_id];
  if (tid == 0) {
    for (int k = 0; k < kRing; ++k) { mbar_init(&full[k], 1); mbar_init(&empty[k], 1); }
    s_done = 0;
    s_last = -1;
  }
  __syncthreads();

  if (tid >= NC) {
    // ---- generator warps: block 0 is the state as it stands, block k its k-th twist
    const int t = tid - NC;
    constexpr int N = RTD3_MT_N, M = 397;
    for (int blk = 0;; ++blk) {
      const int slot = blk % kRing;
      if (t == 0) {
        if (blk >= kRing)                                // one thread polls (the others wait at the barrier, off the issue slots)
          while (!mbar_try_wait(&empty[slot], (uint32_t)((blk / kRing - 1) & 1)) && !s_done) __nanosleep(64);
        // the consumers may set s_done at any time: one read decides for all 256 threads, or some warps could leave the loop
        // while the others wait for them at the next generator barrier.  Thread 0 writes s_gen_stop again only after the barrier
        // that ends this block, which every thread reaches after its read.
        s_gen_stop = s_done;
      }
      bar_named(2, 256);
      if (s_gen_stop) break;
      if (blk > 0) {
        const int lo[3] = {0, N - M, 2 * (N - M)}, hi[3] = {N - M, 2 * (N - M), N};
#pragma unroll
        for (int ph = 0; ph < 3; ++ph) {             // every range reads only words finished by earlier ranges (or still old)
          const int kk = lo[ph] + t;
          uint32_t v = 0u;
          if (kk < hi[ph]) v = mt_twist(mt[kk], mt[kk + 1 < N ? kk + 1 : 0], mt[kk + M < N ? kk + M : kk + M - N]);
          bar_named(2, 256);
          if (kk < hi[ph]) mt[kk] = v;
          bar_named(2, 256);
        }
      }
      for (int k = t; k < N; k += 256) ring[slot * N + k] = mt_temper(mt[k]);
      bar_named(2, 256);
      if (t == 0) mbar_arrive(&full[slot]);
    }
    return;
  }

  // ---- consumer warps
  const int t = tid, lane = t & 31, warp = t >> 5;
  const uint32_t lt = (1u << lane) - 1u;
  uint32_t gpos = (uint32_t)pos0;                    // index into the stream of blocks 0, 1, ... (pos0 may be 624: block 1, word 0)
  int rpos = pos0;                                   // gpos modulo the ring size (pos0 <= 624 < ring size)
  int avail = 0;                                     // blocks known to be in the ring
  uint32_t avail_words = 0u;                         // = avail * 624
  int released = 0;                                  // blocks handed back to the generator
  uint32_t released_words = 0u;
  int par = 0;
  for (int s = 0; s < count; ++s) {
    int32_t* Js = J + (int64_t)s * n;
    int i = n - 1;                                   // swaps still to draw: indices i, i-1, ..., 1 (same value in every thread)
    while (i >= 1) {
      const int lvl = 31 - __clz(i);                 // mask(i) = 2^(lvl+1) - 1
      const int gap = i - (1 << lvl);                // bounds down to i - gap keep mask(i)
      // about sqrt(32 * 2^(lvl+1)) draws keep the expected number of undecided draws near 16
      const int want = lvl >= 10 ? NC : (lvl >= 8 ? 256 : (lvl >= 6 ? 128 : 64));
      // close to the next power of two the round runs over it: about two raw draws per remaining index of this level cross the
      // boundary (acceptance there is ~50 %), the draws behind it are undecided (their mask depends on how many were accepted) and are
      // resolved exactly like the others - instead of five or six ever shorter rounds that stop at the boundary
      const int g = min(2 * (gap + 1) + 32, want);
      // ring upkeep: blocks before the one holding draw gpos - 1 are finished with; blocks up to the one of draw gpos + g - 1 are needed
      if (t == 0)
        while (released_words + (uint32_t)RTD3_MT_N + 1u <= gpos) {
          mbar_arrive(&empty[released % kRing]);
          ++released; released_words += (uint32_t)RTD3_MT_N;
        }
      while (avail_words < gpos + (uint32_t)g) {
        mbar_wait(&full[avail % kRing], (uint32_t)((avail / kRing) & 1));
        ++avail; avail_words += (uint32_t)RTD3_MT_N;
      }
      const bool active = t < g;
      int ri = rpos + t;
      if (ri >= kRingWords) ri -= kRingWords;
      const uint32_t rw = active ? ring[ri] : 0u;
      const int lo = i - t;                          // bound if every earlier draw of the round was accepted
      const bool uniform = lo >= 1 && __clz(lo) == __clz(i);
      const uint32_t v_hi = rw & (0xffffffffu >> __clz(i));
      const bool sure = active && uniform && (int)v_hi <= lo;
      const bool maybe = active && !sure && lo < i && ((uniform && (int)v_hi <= i) || !uniform);
      const uint32_t bs = __ballot_sync(0xffffffffu, sure), bm = __ballot_sync(0xffffffffu, maybe);
      const int S_in = __popc(bs & lt), m_in = __popc(bm & lt);
      if (lane == 0) w_cnt[par][warp] = __popc(bs) | (__popc(bm) << 16);
      if (maybe) mb[par][warp][m_in] = MaybeRec{S_in, rw};
      bar_named(1, NC);
      // every WARP resolves the undecided draws of the whole round, 32 at a time in stream order (lane q: the q-th of them): bound_q =
      // i - (sure draws before q) - (accepted undecided draws before q); the last term by iterating the ballot to its fixed point
      // (lane L depends only on lanes < L).  Redundant in all eight warps - what it saves is compaction, a resolver warp, three barriers.
      int sbef[NW], mbef[NW], sure_run = 0, maybe_run = 0;
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const int cnt = w_cnt[par][w];
        sbef[w] = sure_run; mbef[w] = maybe_run;
        sure_run += cnt & 0xffff; maybe_run += cnt >> 16;
      }
      int S_base = 0, nb = m_in;                     // sure draws before my warp; undecided draws before me
#pragma unroll
      for (int w = 0; w < NW; ++w)
        if (w == warp) { S_base = sbef[w]; nb += mbef[w]; }
      int extra = 0, my_before = 0;
      bool my_acc = false;
      for (int q0 = 0; q0 < maybe_run; q0 += 32) {
        const int q = q0 + lane;
        const bool on = q < maybe_run;
        int wq = 0, sb = sbef[0], mq = mbef[0];
#pragma unroll
        for (int w = 1; w < NW; ++w)
          if (q >= mbef[w]) { wq = w; sb = sbef[w]; mq = mbef[w]; }
        MaybeRec r = MaybeRec{0, 0u};
        if (on) r = mb[par][wq][q - mq];
        const int Sq = sb + r.S;
        uint32_t acc = 0u, prev;
        do {
          prev = acc;
          const int bound = i - Sq - extra - __popc(prev & lt);
          const bool a = on && bound >= 1 && (int)(r.rw & (0xffffffffu >> __clz(max(bound, 1)))) <= bound;
          acc = __ballot_sync(0xffffffffu, a);
        } while (acc != prev);
        const int cb = min(max(nb - q0, 0), 32);     // undecided draws of this chunk that come before me
        my_before += __popc(acc & (cb >= 32 ? 0xffffffffu : ((1u << cb) - 1u)));
        if (maybe && nb >= q0 && nb < q0 + 32) my_acc = (acc >> (nb - q0)) & 1u;
        extra += __popc(acc);
      }
      const int rank = S_base + S_in + my_before;
      const bool accepted = sure || (maybe && my_acc);
      const int my_i = i - rank;
      if (accepted && my_i >= 1) {
        Js[my_i] = (int32_t)(maybe ? (rw & (0xffffffffu >> __clz(max(my_i, 1)))) : v_hi);
        if (my_i == 1) s_last = t;                   // the draw that completes this sample
      }
      const int total_acc = sure_run + extra;        // the same number in every thread
      par ^= 1;
      if (total_acc >= i) {
        bar_named(1, NC);
        gpos += (uint32_t)(s_last + 1);
        rpos += s_last + 1;
        i = 0;
        bar_named(1, NC);                           // everybody has read s_last before the next sample's last round writes it
      } else {
        gpos += (uint32_t)g;
        rpos += g;
        i -= total_acc;
      }
      if (rpos >= kRingWords) rpos -= kRingWords;
    }
  }
  // ---- stop the generator, write the stream back: the un-tempered block the stream stands in, numpy's position convention
  int blk = (int)(gpos / (uint32_t)RTD3_MT_N);
  int pos = (int)(gpos % (uint32_t)RTD3_MT_N);
  if (pos == 0 && gpos > 0u) { blk -= 1; pos = RTD3_MT_N; }
  // block blk is still in the ring (nothing at or after the block of draw gpos - 1 was released); make sure it has been produced
  while (avail <= blk) { mbar_wait(&full[avail % kRing], (uint32_t)((avail / kRing) & 1)); ++avail; }
  bar_named(1, NC);
  if (t == 0) s_done = 1;                              // the generator polls this word while it waits for a free slot
  for (int k = t; k < RTD3_MT_N; k += NC) b.mt[(int64_t)k * b.n + stream_id] = mt_untemper(ring[(blk % kRing) * RTD3_MT_N + k]);
  if (t == 0) b.pos[stream_id] = pos;
}

// Kernel B: out[s][p] = x[p] after the shuffle, by unwinding the swaps from position p.
__global__ void __launch_bounds__(256)
sample_trace_kernel(const int32_t* __restrict__ J, int32_t n, int32_t batch, int32_t* __restrict__ out) {
  extern __shared__ __align__(16) int32_t js[];     // swap list of this sample (n entries, padded to a multiple of 4)
  const int s = blockIdx.x;
  const int32_t* Js = J + (int64_t)s * n;
  const int n4 = (n + 3) & ~3;
  for (int k = threadIdx.x; k < n4; k += blockDim.x) js[k] = (k >= 1 && k < n) ? Js[k] : k;   // entries 0 and >= n are self-swaps
  __syncthreads();
  for (int p = threadIdx.x; p < batch; p += blockDim.x) {
    int pos = p;
    for (int i = 0; i < n4; i += 4) {
      const int4 j = *reinterpret_cast<const int4*>(js + i);
      pos = (pos == i + 0) ? j.x : ((pos == j.x) ? i + 0 : pos);
      pos = (pos == i + 1) ? j.y : ((pos == j.y) ? i + 1 : pos);
      pos = (pos == i + 2) ? j.z : ((pos == j.z) ? i + 2 : pos);
      pos = (pos == i + 3) ? j.w : ((pos == j.w) ? i + 3 : pos);
    }
    out[(int64_t)s * batch + p] = pos;
  }
}

__global__ void sample_philox_kernel(uint64_t seed, uint64_t offset, uint32_t n, int64_t total, int32_t* __restrict__ out) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (4 * t >= total) return;
  const uint64_t c = offset + (uint64_t)t;
  const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), 0u, 0u), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint32_t v[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int k = 0; k < 4; ++k)
    if (4 * t + k < total) out[4 * t + k] = (int32_t)__umulhi(v[k], n);   // multiply-shift map to [0, n)
}

}  // namespace rtd3

using namespace rtd3;

extern "C" int32_t rtd3_sample_indices_philox(uint64_t seed, uint64_t offset, int64_t n, int32_t batch, int32_t count, int32_t* out,
                                              void* stream) {
  RTD3_CHECK_ARG(out && n >= 1 && n < (1ll << 31) && batch >= 1 && count >= 0, "bad argument");
  const int64_t total = (int64_t)batch * count;
  if (total == 0) return 0;
  sample_philox_kernel<<<(int)ceil_div(ceil_div(total, 4), 256), 256, 0, (cudaStream_t)stream>>>(seed, offset, (uint32_t)n, total, out);
  RTD3_LAUNCHED();
  return 0;
}


extern "C" int32_t rtd3_sample_indices_mt19937(const rtd3_mt_bank* bank, int64_t stream_id, int32_t n, int32_t batch, int32_t count,
                                               int32_t* out, int32_t* scratch, void* stream) {
  RTD3_CHECK_ARG(bank && bank->mt && bank->pos && out, "null argument");
  RTD3_CHECK_ARG(stream_id >= 0 && stream_id < bank->n, "stream id out of range");
  RTD3_CHECK_ARG(n >= 1 && batch >= 1 && batch <= n && count >= 0, "need 1 <= batch <= n");
  RTD3_CHECK_ARG(n <= 56000, "replay sizes above 56000 rows are not supported by the exact sampler");
  RTD3_CHECK_ARG((int64_t)n * count < (1ll << 30), "count * n must stay below 2^30 raw draws per call");
  if (count == 0) return 0;
  RTD3_CHECK_ARG(scratch, "scratch (count * n int32) is required");
  RTD3_CUDA(ensure_dyn_smem((const void*)sample_trace_kernel, 56000 * 4));
  cudaStream_t st = (cudaStream_t)stream;
  sample_swaps_pipelined_kernel<8><<<1, 8 * 32 + 256, 0, st>>>(*bank, stream_id, n, count, scratch);
  RTD3_LAUNCHED();
  const size_t smem = (size_t)((n + 3) & ~3) * 4;
  sample_trace_kernel<<<count, 256, smem, st>>>(scratch, n, batch, out);
  RTD3_LAUNCHED();
  return 0;
}
