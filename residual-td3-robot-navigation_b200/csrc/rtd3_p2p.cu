// Gradient all-reduce of the data-parallel learner over NVLink peer memory (SURVEY.md 8e: the one collective of the path).
// Every rank owns a receive area its peers have mapped (CUDA IPC): recv[2][W][count] floats + a flag array.  One launch per
// optimiser step, PUSH model - remote stores are fire-and-forget, remote loads are round trips:
//   (1) every block copies its slice of the local gradient buffer into slot [step parity][rank] of EVERY rank's receive area
//       (its own included) and clears the local slice for the next step;
//   (2) the last block to finish (system-scope fences, a block counter) stores the step number into the peers' flag arrays;
//   (3) every block waits until all W flags show this step, then adds the W slots of its own receive area in rank order - the
//       same order on every rank, so the replicas stay bit-identical - into the private buffer the optimiser kernel consumes.
// The two parities make a second barrier unnecessary: a rank overwrites slot [p] two steps later, after it has seen the flags of the
// step in between, which every peer raises only after it has finished reading slot [p].
// The step number lives in device memory and is advanced by the kernel, so a replayed CUDA graph counts on by itself; a rank whose
// peers do not arrive within kSpinLimitNs traps instead of hanging.  (A pull version - flags, then loads from the peers' gradient
// buffers, then a second barrier before they may be overwritten - took as long as the NCCL call it replaced: three serialised
// NVLink round trips.)
#include <algorithm>

#include "rtd3_common.cuh"
#include "rtd3_p2p.cuh"
#include "rtd3_td3.cuh"

namespace rtd3 {

// phases (1) and (2) of the header comment + the wait of phase (3); returns this step's number
template <int kWorld>
__device__ __forceinline__ unsigned long long p2p_push_and_wait(const P2pPeers& peers, int rank, unsigned long long* seq_counter,
                                                                float* __restrict__ local_grads, int64_t count4, int64_t stride4,
                                                                unsigned int* block_counter) {
  __shared__ bool s_last;
  __shared__ unsigned long long s_seq;
  const int tid = threadIdx.x;
  if (tid == 0) s_seq = *reinterpret_cast<volatile unsigned long long*>(seq_counter) + 1ull;
  __syncthreads();
  const unsigned long long seq = s_seq;
  // [parity][rank] in every receive area; slots are `stride4` apart whatever this call's count (calls of different sizes may
  // alternate - critic and actor gradients - and a slot of one parity must never reach into the other parity's half)
  const int64_t slot = ((int64_t)(seq & 1ull) * kWorld + rank) * stride4;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  // (1) push (the kernels that produced local_grads precede this one in stream order)
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + tid; i < count4; i += stride) {
    const float4 v = reinterpret_cast<const float4*>(local_grads)[i];
#pragma unroll
    for (int q = 0; q < kWorld; ++q) reinterpret_cast<float4*>(peers.recv[q])[slot + i] = v;
    reinterpret_cast<float4*>(local_grads)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // (2) the last block of this rank raises the flags
  __syncthreads();
  if (tid == 0) {
    __threadfence_system();
    s_last = atomicAdd(block_counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {
    if (tid < kWorld) {
      __threadfence_system();
      st_release_sys(peers.flags[tid] + rank, seq);
    }
    if (tid == 0) {
      *block_counter = 0u;                             // every block of this launch has passed the counter ...
      *seq_counter = seq;                              // ... and has read the step number
    }
  }
  // (3) all W gradients of this step have landed here
  if (tid < kWorld) wait_flag(peers.flags[rank] + tid, seq);
  __syncthreads();
  return seq;
}

template <int kWorld>
__device__ __forceinline__ float4 p2p_sum_slots(const float4* mine, int64_t stride4, int64_t i) {
  float4 v[kWorld];
#pragma unroll
  for (int r = 0; r < kWorld; ++r) v[r] = ld_fresh(mine + (int64_t)r * stride4 + i);
  float4 acc = v[0];
#pragma unroll
  for (int r = 1; r < kWorld; ++r) { acc.x += v[r].x; acc.y += v[r].y; acc.z += v[r].z; acc.w += v[r].w; }   // rank order on every rank
  return acc;
}

template <int kWorld>
__global__ void __launch_bounds__(256) p2p_allreduce_kernel(P2pPeers peers, int rank, unsigned long long* seq_counter, float* __restrict__ out,
                                                            float* __restrict__ local_grads, int64_t count4, int64_t stride4,
                                                            unsigned int* block_counter) {
  const unsigned long long seq = p2p_push_and_wait<kWorld>(peers, rank, seq_counter, local_grads, count4, stride4, block_counter);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const float4* mine = reinterpret_cast<const float4*>(peers.recv[rank]) + (int64_t)(seq & 1ull) * kWorld * stride4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count4; i += stride)
    reinterpret_cast<float4*>(out)[i] = p2p_sum_slots<kWorld>(mine, stride4, i);
}

// The same all-reduce with the optimiser applied to the sums, and with the hand-over made BLOCK-LOCAL: block b of every rank owns the
// same arena elements in the push and in the reduction, so it raises its own flag (flag area [16 + rank * 256 + block]) right after
// its own pushes and waits only for block b of its peers - no block counter and no last-block hop on the way to the flags, and a
// slow block delays only its own elements.  Phase (3) walks the online arena like td3_adam_polyak_kernel - Adam on the elements of
// the reduced slice (gradient = sum of the W slots x grad_scale), the Polyak blend where asked for - so the summed gradients never
// go back to memory and the separate optimiser launch (one more pass over the arena) disappears.
template <int kWorld>
__global__ void __launch_bounds__(256) p2p_allreduce_adam_kernel(P2pPeers peers, int rank, unsigned long long* seq_counter,
                                                                 float* __restrict__ local_grads, int64_t count4, int64_t stride4,
                                                                 unsigned int* block_counter, P2pAdamArgs o) {
  __shared__ float s_step[2], s_bc2[2];
  __shared__ unsigned long long s_seq;
  const int tid = threadIdx.x;
  if (tid < 2) {                                                      // 0: actor optimiser, 1: both critic optimisers
    const AdamStep k = adam_step(tid == 0 ? o.adam.lr[0] : o.adam.lr[1], o.adam.beta_pows[2 * tid], o.adam.beta_pows[2 * tid + 1]);
    s_step[tid] = k.step;
    s_bc2[tid] = k.sqrt_bc2;
  }
  if (tid == 0) s_seq = *reinterpret_cast<volatile unsigned long long*>(seq_counter) + 1ull;
  __syncthreads();
  const unsigned long long seq = s_seq;
  const int n4 = (int)(o.adam.ar.online_total() >> 2), off4 = (int)(o.off >> 2), end4 = off4 + (int)count4;
  const int gstride = gridDim.x * blockDim.x;
  const int64_t slot = ((int64_t)(seq & 1ull) * kWorld + rank) * stride4;
  // (1) push this block's elements of the slice into slot [step parity][rank] of every rank, clear them locally
  for (int i4 = blockIdx.x * blockDim.x + tid; i4 < n4; i4 += gstride) {
    if (i4 < off4 || i4 >= end4) continue;
    const float4 v = reinterpret_cast<const float4*>(local_grads)[i4];
#pragma unroll
    for (int q = 0; q < kWorld; ++q) reinterpret_cast<float4*>(peers.recv[q])[slot + (i4 - off4)] = v;
    reinterpret_cast<float4*>(local_grads)[i4] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  // (2) this block's flag at every rank (the fence of each storing thread covers the block's pushes: they precede the barrier)
  __syncthreads();
  if (tid < kWorld) {
    __threadfence_system();
    st_release_sys(peers.flags[tid] + kP2pBlockFlagBase + rank * kP2pBlockFlags + blockIdx.x, seq);
  }
  if (tid == 32) {                                                    // bookkeeping off the critical path: the step number
    if (atomicAdd(block_counter, 1u) == gridDim.x - 1) {              // every block of this launch has read it
      *block_counter = 0u;
      *seq_counter = seq;
    }
  }
  // (3) block b of every rank has pushed: reduce in rank order, apply the optimiser
  if (tid < kWorld) wait_flag(peers.flags[rank] + kP2pBlockFlagBase + tid * kP2pBlockFlags + blockIdx.x, seq);
  __syncthreads();
  const float4* mine = reinterpret_cast<const float4*>(peers.recv[rank]) + (int64_t)(seq & 1ull) * kWorld * stride4;
  const int off1 = (int)o.adam.ar.off(1), off2 = (int)o.adam.ar.off(2);
  for (int i4 = blockIdx.x * blockDim.x + tid; i4 < n4; i4 += gstride) {
    const int i = i4 * 4;
    const int net = i < off1 ? 0 : (i < off2 ? 1 : 2);               // slots are multiples of 4 floats: a group never straddles two
    const bool do_adam = (o.nets >> net) & 1, do_polyak = (o.polyak >> net) & 1;
    if (!do_adam && !do_polyak) continue;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (do_adam) g = p2p_sum_slots<kWorld>(mine, stride4, (int64_t)(i4 - off4));
    const float gg[4] = {g.x * o.grad_scale, g.y * o.grad_scale, g.z * o.grad_scale, g.w * o.grad_scale};
    const int k = net == 0 ? 0 : 1;
    adam_polyak_apply4(o.adam, i, net, gg, AdamStep{s_step[k], s_bc2[k]}, do_adam, do_polyak);
  }
}

}  // namespace rtd3

using namespace rtd3;

extern "C" int32_t rtd3_p2p_allreduce(float* const* peer_recv, uint64_t* const* peer_flags, int32_t rank, int32_t world, uint64_t* seq_counter,
                                      float* out, float* local_grads, int64_t count, int64_t slot_floats, uint32_t* block_counter, void* stream) {
  RTD3_CHECK_ARG(peer_recv && peer_flags && out && local_grads && block_counter && seq_counter, "null argument");
  RTD3_CHECK_ARG(world >= 2 && world <= kP2pMaxWorld && rank >= 0 && rank < world, "bad rank / world");
  RTD3_CHECK_ARG(count > 0 && count % 4 == 0, "count must be a positive multiple of 4");
  RTD3_CHECK_ARG(slot_floats >= count && slot_floats % 4 == 0, "slot_floats must be a multiple of 4 and at least count");
  RTD3_CHECK_ARG((uintptr_t)out % 16 == 0 && (uintptr_t)local_grads % 16 == 0, "out / local_grads must be 16 B aligned");
  P2pPeers p{};
  for (int r = 0; r < world; ++r) {
    RTD3_CHECK_ARG(peer_recv[r] && peer_flags[r], "null peer pointer");
    RTD3_CHECK_ARG((uintptr_t)peer_recv[r] % 16 == 0 && (uintptr_t)peer_flags[r] % 8 == 0, "misaligned peer pointer");
    p.recv[r] = peer_recv[r];
    p.flags[r] = (unsigned long long*)peer_flags[r];
  }
  // All blocks wait for the peers' flags, and a peer raises its flag from the LAST of its blocks: the grid must be co-resident
  // whatever else runs on the device.  At most one CTA per SM, launched COOPERATIVELY - the runtime places a cooperative grid
  // as a whole or not at all, so a kernel of another stream that holds some SMs delays the launch instead of starving blocks that
  // others are spinning for (VERDICT r1: a concurrent kernel could have turned the spin into the 20 s trap).
  const int64_t count4 = count / 4;
  int num_sms = 0;
  RTD3_CUDA(current_num_sms(&num_sms));
  const int grid = (int)std::min<int64_t>((int64_t)num_sms, ceil_div(count4, 256));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* sc = (unsigned long long*)seq_counter;
  int64_t stride4 = slot_floats / 4;
  void* kargs[] = {&p, &rank, &sc, &out, &local_grads, (void*)&count4, &stride4, &block_counter};
  const void* fn = nullptr;
  switch (world) {
#define RTD3_P2P_CASE(W) case W: fn = (const void*)p2p_allreduce_kernel<W>; break;
    RTD3_P2P_CASE(2) RTD3_P2P_CASE(3) RTD3_P2P_CASE(4) RTD3_P2P_CASE(5) RTD3_P2P_CASE(6) RTD3_P2P_CASE(7) RTD3_P2P_CASE(8)
#undef RTD3_P2P_CASE
  }
  RTD3_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(256), kargs, 0, st));
  RTD3_LAUNCHED();
  return 0;
}


int32_t rtd3::p2p_allreduce_adam_launch(const rtd3_p2p_state* ps, float* local_grads, int64_t count, const P2pAdamArgs& opt, cudaStream_t st) {
  RTD3_CHECK_ARG(ps && ps->peer_recv && ps->peer_flags && local_grads && ps->block_counter && ps->seq_counter, "null argument");
  const int world = ps->world, rank = ps->rank;
  RTD3_CHECK_ARG(world >= 2 && world <= kP2pMaxWorld && rank >= 0 && rank < world, "bad rank / world");
  RTD3_CHECK_ARG(count > 0 && count % 4 == 0 && opt.off % 4 == 0, "count / offset must be multiples of 4");
  RTD3_CHECK_ARG(ps->slot_floats >= count && ps->slot_floats % 4 == 0, "slot_floats must be a multiple of 4 and at least count");
  P2pPeers p{};
  for (int r = 0; r < world; ++r) {
    RTD3_CHECK_ARG(ps->peer_recv[r] && ps->peer_flags[r], "null peer pointer");
    p.recv[r] = ps->peer_recv[r];
    p.flags[r] = (unsigned long long*)ps->peer_flags[r];
  }
  // cooperative launch with at most one CTA per SM: see rtd3_p2p_allreduce
  int64_t count4 = count / 4, stride4 = ps->slot_floats / 4;
  int num_sms = 0;
  RTD3_CUDA(current_num_sms(&num_sms));
  const int grid = (int)std::min<int64_t>(std::min<int64_t>((int64_t)num_sms, kP2pBlockFlags), ceil_div(opt.adam.ar.online_total() / 4, 256));
  unsigned long long* sc = (unsigned long long*)ps->seq_counter;
  int rk = rank;
  unsigned int* bc = ps->block_counter;
  P2pAdamArgs o = opt;
  // every element of a reduced slice must have an optimiser bit: the pushes and the reduction use the same element -> block map
  void* kargs[] = {&p, &rk, &sc, &local_grads, &count4, &stride4, &bc, &o};
  const void* fn = nullptr;
  switch (world) {
#define RTD3_P2P_CASE(W) case W: fn = (const void*)p2p_allreduce_adam_kernel<W>; break;
    RTD3_P2P_CASE(2) RTD3_P2P_CASE(3) RTD3_P2P_CASE(4) RTD3_P2P_CASE(5) RTD3_P2P_CASE(6) RTD3_P2P_CASE(7) RTD3_P2P_CASE(8)
#undef RTD3_P2P_CASE
  }
  RTD3_CUDA(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(256), kargs, 0, st));
  RTD3_LAUNCHED();
  return 0;
}
