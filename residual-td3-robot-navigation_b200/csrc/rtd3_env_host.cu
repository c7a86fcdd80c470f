// rtd3_env_rollout_host: the T-step rollout for HOST buffers (pinned), the call behind Environment.rollout_host and the `e2e` figure
// of bench.py.  The T steps are cut into time slices; the copy engines move the actions of slice c+1 to HBM and the trajectory of
// slice c-1 back while the rollout kernel runs slice c.  The whole pipeline - 2 x chunks memcpy nodes on two branches and chunks
// kernel nodes - is captured ONCE per (buffers, shape) into a CUDA graph kept in the env handle, so a call is one cudaGraphLaunch:
// no per-slice launch / event / stream-wait calls on the host, and the two copy directions run concurrently on their own engines.
// (The loop this serves: robot-learning.py:97-100 with the actions supplied, as rtd3_env_rollout.)
#include <mutex>
#include <vector>

#include "rtd3_common.cuh"
#include "rtd3_env_step.cuh"

namespace rtd3 {

struct HostGraph {
  const void *x, *y, *act, *traj;
  int64_t n, T;
  int32_t chunks, mode;
  // The map configuration the captured rollout kernels hold as arguments (and whether they are the single-map or the bank
  // kernels).  Reallocating the bank or the index drops the cached graphs; a change of K or m without one makes them miss.
  MapBank map;
  cudaGraphExec_t exec;
};

static std::mutex g_pipe_mu;         // one host-buffer call at a time per process: creation, capture and the graph cache are not re-entrant

struct HostPipe {
  cudaStream_t cap = nullptr, s_in = nullptr, s_out = nullptr;
  float *d_act = nullptr, *d_traj = nullptr;
  size_t floats = 0;                 // capacity of each staging buffer
  std::vector<cudaEvent_t> events;   // capture-time dependency markers, reused by every capture
  std::vector<HostGraph> graphs;     // oldest first
};

constexpr size_t kMaxHostGraphs = 16;

static void drop_graphs(HostPipe* p) {
  if (p->graphs.empty()) return;
  cudaDeviceSynchronize();           // a cached graph may still be running on the caller's stream
  for (auto& g : p->graphs) cudaGraphExecDestroy(g.exec);
  p->graphs.clear();
}

void host_pipe_drop_graphs(rtd3_env* h) {
  if (h->host_pipe) drop_graphs((HostPipe*)h->host_pipe);
}

void host_pipe_destroy(rtd3_env* h) {
  HostPipe* p = (HostPipe*)h->host_pipe;
  if (!p) return;
  DeviceGuard guard;
  guard.enter(h->device);
  drop_graphs(p);
  for (cudaEvent_t e : p->events) cudaEventDestroy(e);
  if (p->d_act) cudaFree(p->d_act);
  if (p->d_traj) cudaFree(p->d_traj);
  if (p->cap) cudaStreamDestroy(p->cap);
  if (p->s_in) cudaStreamDestroy(p->s_in);
  if (p->s_out) cudaStreamDestroy(p->s_out);
  delete p;
  h->host_pipe = nullptr;
}

static int32_t pipe_prepare(rtd3_env* h, HostPipe** out, size_t floats, int n_events) {
  HostPipe* p = (HostPipe*)h->host_pipe;
  if (!p) {
    p = new HostPipe();
    h->host_pipe = p;
    RTD3_CUDA(cudaStreamCreateWithFlags(&p->cap, cudaStreamNonBlocking));
    RTD3_CUDA(cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking));
    RTD3_CUDA(cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking));
  }
  if (floats > p->floats) {
    drop_graphs(p);                  // they hold the old staging addresses
    if (p->d_act) cudaFree(p->d_act);
    if (p->d_traj) cudaFree(p->d_traj);
    p->d_act = p->d_traj = nullptr;
    p->floats = 0;
    RTD3_CUDA(cudaMalloc(&p->d_act, floats * sizeof(float)));
    RTD3_CUDA(cudaMalloc(&p->d_traj, floats * sizeof(float)));
    p->floats = floats;
  }
  while ((int)p->events.size() < n_events) {
    cudaEvent_t e;
    RTD3_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    p->events.push_back(e);
  }
  *out = p;
  return 0;
}

// The pipeline issued into the capturing stream p->cap and its two forks.
static int32_t issue_pipeline(rtd3_env* h, HostPipe* p, float* x, float* y, const float* act, float* traj, int64_t n, int64_t T,
                              int32_t chunks, bool stage_in, bool stage_out) {
  const int64_t plane = 2 * n;
  cudaEvent_t* ev = p->events.data();
  int e_next = 0;
  cudaEvent_t fork = ev[e_next++];
  RTD3_CUDA(cudaEventRecord(fork, p->cap));
  if (stage_in) RTD3_CUDA(cudaStreamWaitEvent(p->s_in, fork, 0));
  if (stage_out) RTD3_CUDA(cudaStreamWaitEvent(p->s_out, fork, 0));
  std::vector<int64_t> lo(chunks + 1);
  for (int c = 0; c <= chunks; ++c) lo[c] = (int64_t)((double)c * (double)T / (double)chunks + 0.5);
  std::vector<cudaEvent_t> in_done(chunks);
  if (stage_in)
    for (int c = 0; c < chunks; ++c) {
      const int64_t t0 = lo[c], len = lo[c + 1] - lo[c];
      if (len == 0) continue;
      RTD3_CUDA(cudaMemcpyAsync(p->d_act + t0 * plane, act + t0 * plane, (size_t)(len * plane) * sizeof(float), cudaMemcpyHostToDevice, p->s_in));
      in_done[c] = ev[e_next++];
      RTD3_CUDA(cudaEventRecord(in_done[c], p->s_in));
    }
  for (int c = 0; c < chunks; ++c) {
    const int64_t t0 = lo[c], len = lo[c + 1] - lo[c];
    if (len == 0) continue;
    if (stage_in) RTD3_CUDA(cudaStreamWaitEvent(p->cap, in_done[c], 0));
    const float* src = (stage_in ? p->d_act : act) + t0 * plane;
    float* dst = (stage_out ? p->d_traj : traj) + t0 * plane;
    if (int32_t e = env_rollout(h, x, y, src, dst, n, len, !stage_out, p->cap)) return e;
    if (stage_out) {
      cudaEvent_t k = ev[e_next++];
      RTD3_CUDA(cudaEventRecord(k, p->cap));
      RTD3_CUDA(cudaStreamWaitEvent(p->s_out, k, 0));
      RTD3_CUDA(cudaMemcpyAsync(traj + t0 * plane, p->d_traj + t0 * plane, (size_t)(len * plane) * sizeof(float), cudaMemcpyDeviceToHost, p->s_out));
    }
  }
  if (stage_out) {                   // join (the s_in branch is joined through the last slice's in_done event)
    cudaEvent_t j = ev[e_next++];
    RTD3_CUDA(cudaEventRecord(j, p->s_out));
    RTD3_CUDA(cudaStreamWaitEvent(p->cap, j, 0));
  }
  return 0;
}

static bool is_pinned(const void* ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

}  // namespace rtd3

using namespace rtd3;

extern "C" int32_t rtd3_env_rollout_host(rtd3_env* h, float* x, float* y, const float* actions_host, float* traj_host, int64_t n,
                                         int64_t T, int32_t chunks, int32_t mode, void* stream) {
  RTD3_CHECK_ARG(h && h->num_maps > 0, "environment has no dynamics map (call rtd3_env_set_map)");
  RTD3_CHECK_ARG(n >= 0 && T >= 0, "negative n or T");
  RTD3_CHECK_ARG(mode >= 0 && mode <= 3, "mode is a bit set: 1 = stage the actions, 2 = stage the trajectory");
  if (n == 0 || T == 0) return 0;
  RTD3_CHECK_ARG(x && y && actions_host && traj_host, "null state / action / trajectory pointer");
  RTD3_CHECK_ARG(is_pinned(actions_host) && is_pinned(traj_host), "actions_host and traj_host must be page-locked host memory");
  if (mode == 0)                     // zero copy: the kernel's TMA tiles cross PCIe themselves
    return env_rollout(h, x, y, actions_host, traj_host, n, T, true, (cudaStream_t)stream);
  chunks = (int32_t)std::max<int64_t>(1, std::min<int64_t>(chunks, std::min<int64_t>(T, 256)));
  const bool stage_in = mode & 1, stage_out = mode & 2;
  DeviceGuard guard;
  RTD3_CUDA(guard.enter(h->device));
  std::lock_guard<std::mutex> lock(g_pipe_mu);
  HostPipe* p = nullptr;
  int32_t rc = pipe_prepare(h, &p, (size_t)(2 * n * T), 2 * chunks + 2);
  cudaGraphExec_t exec = nullptr;
  const MapBank mk = map_bank(h);
  if (rc == 0) {
    for (auto& g : p->graphs)
      if (g.x == x && g.y == y && g.act == actions_host && g.traj == traj_host && g.n == n && g.T == T && g.chunks == chunks && g.mode == mode &&
          g.map == mk)
        exec = g.exec;
    if (!exec) {
      if (p->graphs.size() >= kMaxHostGraphs) {
        cudaDeviceSynchronize();
        cudaGraphExecDestroy(p->graphs.front().exec);
        p->graphs.erase(p->graphs.begin());
      }
      cudaGraph_t graph = nullptr;
      cudaError_t ce = cudaStreamBeginCapture(p->cap, cudaStreamCaptureModeThreadLocal);
      if (ce != cudaSuccess) {
        set_error("rtd3_env_rollout_host: cudaStreamBeginCapture -> %s", cudaGetErrorString(ce));
        rc = (int32_t)ce;
      } else {
        rc = issue_pipeline(h, p, x, y, actions_host, traj_host, n, T, chunks, stage_in, stage_out);
        ce = cudaStreamEndCapture(p->cap, &graph);       // always ends the capture, also after a failed issue
        if (rc == 0 && ce != cudaSuccess) {
          set_error("rtd3_env_rollout_host: cudaStreamEndCapture -> %s", cudaGetErrorString(ce));
          rc = (int32_t)ce;
        }
        if (rc == 0) {
          ce = cudaGraphInstantiate(&exec, graph, 0);
          if (ce != cudaSuccess) {
            set_error("rtd3_env_rollout_host: cudaGraphInstantiate -> %s", cudaGetErrorString(ce));
            rc = (int32_t)ce;
            exec = nullptr;
          }
        }
        if (graph) cudaGraphDestroy(graph);
        if (rc != 0) cudaGetLastError();
      }
      if (rc == 0) p->graphs.push_back(HostGraph{x, y, actions_host, traj_host, n, T, chunks, mode, mk, exec});
    }
    if (rc == 0) {
      cudaError_t ce = cudaGraphLaunch(exec, (cudaStream_t)stream);
      if (ce != cudaSuccess) {
        set_error("rtd3_env_rollout_host: cudaGraphLaunch -> %s", cudaGetErrorString(ce));
        rc = (int32_t)ce;
      } else {
        count_launch(chunks);        // the kernel nodes of the replayed graph (the capture counted them once)
      }
    }
  }
  return rc;
}
