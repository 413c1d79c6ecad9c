// engine.hpp — the host-side engine object behind the C ABI (include/selfplay_b200.h): one `Mcts` + its `Vec<Tree>` on
// one GPU (ref: src/mcts.rs:41-44, src/learner_concurrent.rs:174).  Shared by engine.cu (engine + entry points that
// launch kernels, device code in kernels.cuh) and gather.cu (NCCL trajectory gather, learner hand-off).
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "async.cuh"
#include "evaluator.cuh"
#include "trajectory.cuh"
#include "tree.cuh"

namespace spb {

constexpr int CTL_WORDS = 9 * 32;   // control words of the asynchronous pipeline, one 128-byte line each

// ---- self-play ply (ref: learner_concurrent.rs:179-238): device buffers of the trajectories ----------------------
// parked[g] = 1 | terminal status << 1 | terminal side to move << 3
using SelfPlay = Trajectories<spb_position>;

}  // namespace spb

#define SPB_CUDA(expr)                                                                         \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                           \
      return SPB_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

// the same for code outside the engine's methods
#define SPB_CUDA_E(e, expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      (e)->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                      \
      return SPB_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

extern thread_local std::string g_create_error;   // text of the last failure that had no engine to attach to (spb_last_error(NULL))

struct spb_engine {
  using Trees = spb::Trees; using SelfPlay = spb::SelfPlay; using Evaluator = spb::Evaluator; using AsyncCtl = spb::AsyncCtl;
  spb_config cfg{};
  std::string err;
  Trees T{};
  SelfPlay P{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<void*> allocs;
  Evaluator evaluator;
  // staging
  void* h_stage = nullptr; size_t h_stage_bytes = 0;   // pinned
  void* d_stage = nullptr; size_t d_stage_bytes = 0;
  uint8_t* d_rc_actions = nullptr; uint32_t* d_rc_counts = nullptr; uint32_t* d_rc_ids = nullptr; uint32_t* d_rc_n = nullptr;
  unsigned long long* d_misc = nullptr;   // [4] scratch u64
  uint64_t launches = 0;
  float last_search_ms = 0.f, last_eval_ms = 0.f;
  uint32_t last_eval_launches = 0;
  int last_eval_parity = -1;   // parity of the work list the last evaluator launch of spb_search consumed
  // CUDA graph of one split-pipeline step pair (parity 0 and 1)
  cudaGraphExec_t step_graph = nullptr;
  // asynchronous pipeline: rings + control words (async.cuh)
  AsyncCtl ctl{};
  uint32_t* d_ctl_words = nullptr;   // [CTL_WORDS] one 128-byte line per counter
  unsigned long long* d_ring_slots = nullptr;   // [2][ring_size]
  uint32_t ring_size = 0;
  uint64_t last_async_stats[16] = {};
  // multi-GPU trajectory gather (gather.cu): NCCL communicator of this engine's rank, records staged on the learner rank
  void* nccl_comm = nullptr;
  int comm_rank = -1, comm_world = 0;
  bool gather_pending = false;
  std::vector<spb_position> gather_pos;
  std::vector<unsigned long long> gather_ids;
  int A = 0, max_depth = 0, eval_stride = 0, max_ply = 0;
  // EXTENSION: Dirichlet noise at the root (spb_set_root_noise).  The buffers are allocated by the first call that turns
  // the noise on; T.root_noise points at them while it is on.
  float* d_noise_eta = nullptr;
  uint32_t* d_noise_n = nullptr;
  float noise_alpha = 0.0f;
  unsigned long long noise_seed = 0;

  void set_error(const std::string& s) { err = s; }

  template <class T_> int32_t dalloc(T_** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, count * sizeof(T_));
    if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); return SPB_ERR_NOMEM; }
    allocs.push_back(q);
    *p = static_cast<T_*>(q);
    return SPB_OK;
  }
  int32_t ensure_capacity(uint32_t num_searches);
  int32_t ensure_stage(size_t bytes) {
    if (bytes > h_stage_bytes) {
      if (h_stage) cudaFreeHost(h_stage);
      h_stage = nullptr; h_stage_bytes = 0;
      size_t nb = std::max(bytes, (size_t)1 << 20);
      SPB_CUDA(cudaMallocHost(&h_stage, nb));
      h_stage_bytes = nb;
    }
    if (bytes > d_stage_bytes) {
      if (d_stage) cudaFree(d_stage);
      d_stage = nullptr; d_stage_bytes = 0;
      size_t nb = std::max(bytes, (size_t)1 << 20);
      SPB_CUDA(cudaMalloc(&d_stage, nb));
      d_stage_bytes = nb;
    }
    return SPB_OK;
  }
  int32_t check_device_errors();
  int32_t init();
  void destroy();
  template <class G> int32_t search_t(uint32_t num_searches);
  template <class G> int32_t launch_eval_step(uint32_t parity);
  template <class G> int32_t search_async(uint32_t num_searches);
  int32_t launch_root_noise();
};

#define SPB_CHECK_LAUNCH() SPB_CUDA(cudaGetLastError())
