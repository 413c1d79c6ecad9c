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

#include "async.cuh"
#include "evaluator.cuh"
#include "host_engine.hpp"
#include "tree.cuh"

namespace spb {

constexpr int CTL_WORDS = 9 * 32;   // control words of the asynchronous pipeline, one 128-byte line each

// ---- self-play ply (ref: learner_concurrent.rs:179-238): device buffers of the trajectories ----------------------
// parked[g] = 1 | terminal status << 1 | terminal side to move << 3
using SelfPlay = Trajectories<spb_position>;

}  // namespace spb

// Members shared with the chess engine are in HostEngine (host_engine.hpp).
struct spb_engine : spb::HostEngine<spb::Trees, spb_position, uint8_t> {
  using Evaluator = spb::Evaluator; using AsyncCtl = spb::AsyncCtl;
  spb_engine() : HostEngine("spb_", SPB_MAX_ACTIONS) {}
  Evaluator evaluator;
  float last_eval_ms = 0.f;
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
  // evaluation cache of the asynchronous pipeline (ctl.cache, tree.cuh: EvalCache): grow-only, never cleared between
  // searches; every asynchronous search takes the next epoch
  uint32_t cache_epoch = 0;
  uint32_t cache_tried = 0;    // largest table (slots per tree) an allocation was attempted for
  int A = 0, max_depth = 0, eval_stride = 0, max_ply = 0;

  int32_t ensure_capacity(uint32_t num_searches);
  int32_t ensure_eval_cache(uint32_t num_searches);
  void drop_step_graph() {
    if (step_graph) { cudaGraphExecDestroy(step_graph); step_graph = nullptr; }
  }
  int32_t init();
  void release();
  template <class G> int32_t search_t(uint32_t num_searches);
  template <class G> int32_t launch_eval_step(uint32_t parity);
  template <class G> int32_t search_async(uint32_t num_searches);
  int32_t launch_root_noise();
};
