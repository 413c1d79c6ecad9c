// chess_engine.hpp — the host-side chess engine behind the spb_chess_* entry points (include/selfplay_b200.h): one
// `Mcts<chess Net>` + its `Vec<Tree<chess::State>>` on one GPU (ref: src/mcts.rs:41-44 over src/game/chess.rs and
// src/model/chess.rs).  Shared by chess.cu (rules entry points), chess_engine.cu (trees, search) and chess_net.cu
// (the 10 x 256 network).
#pragma once
#include <algorithm>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

#include <cuda_runtime.h>

#include "chess_tree.cuh"
#include "trajectory.cuh"

namespace spb {
namespace chess {
struct Net;   // chess_net.cu
}
}  // namespace spb

struct spb_chess_engine {
  spb_config cfg{};
  std::string err;
  spb::chess::CTrees T{};
  cudaStream_t stream = nullptr, stream2 = nullptr;   // stream2: the second half of the trees in the network pipeline
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_fork = nullptr, ev_join = nullptr;
  std::vector<void*> allocs;
  spb::chess::Net* net = nullptr;
  uint64_t launches = 0;
  float last_search_ms = 0.f;
  // device scratch for results of whole-batch queries
  uint16_t* d_rc_moves = nullptr; uint32_t* d_rc_counts = nullptr; uint32_t* d_rc_ids = nullptr; uint32_t* d_rc_n = nullptr;
  unsigned long long* d_misc = nullptr;
  // device staging of spb_chess_reset_games (allocated once: cudaMalloc / cudaFree per call would synchronise the device)
  uint32_t* d_reset_slots = nullptr; spb::chess::Pos* d_reset_roots = nullptr; unsigned long long* d_reset_hist = nullptr;
  uint32_t* d_adv_ids = nullptr; int32_t* d_adv_err = nullptr;   // spb_chess_advance (with d_reset_slots / d_reset_roots)
  // self-play trajectories (spb_chess_selfplay_step); all null until the first step allocates them.
  // parked[g] = 1 | won << 1 | terminal side to move << 2 | adjudicated << 3
  spb::Trajectories<spb_chess_position> P{};
  // multi-GPU trajectory gather (gather.cu): NCCL communicator of this engine's rank, records staged on the learner rank
  void* nccl_comm = nullptr;
  int comm_rank = -1, comm_world = 0;
  bool gather_pending = false;
  std::vector<spb_chess_position> gather_pos;
  std::vector<unsigned long long> gather_ids;
  // EXTENSION: Dirichlet noise at the root (spb_chess_set_root_noise).  [G][SPB_CHESS_MAX_MOVES] of eta, allocated by the first
  // call that turns the noise on; T.root_noise points at it while it is on.
  float* d_noise_eta = nullptr;
  uint32_t* d_noise_n = nullptr;
  float noise_alpha = 0.0f;
  unsigned long long noise_seed = 0;

  void set_error(const std::string& s) { err = s; }
  template <class T_> int32_t dalloc(T_** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T_));
    if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); return SPB_ERR_NOMEM; }
    allocs.push_back(q);
    *p = static_cast<T_*>(q);
    return SPB_OK;
  }
  int32_t check_device_errors();
  int32_t ensure_selfplay();
};

extern thread_local std::string g_create_error;   // engine.cu

#define CH_CUDA(e, expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      (e)->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                      \
      return SPB_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)
#define CH_GUARD(e)                                                   \
  if (!(e)) return SPB_ERR_ARG;                                       \
  if (cudaSetDevice((e)->cfg.device) != cudaSuccess) { (e)->set_error("cudaSetDevice failed"); return SPB_ERR_CUDA; }
#define CH_ARG(e, cond, msg) \
  if (!(cond)) { (e)->set_error(msg); return SPB_ERR_ARG; }

namespace spb {
namespace chess {
// device scratch for one call of a test / tooling entry point: a few plain allocations, freed on return
struct Scratch {
  std::vector<void*> ptrs;
  ~Scratch() { for (void* p : ptrs) cudaFree(p); }
  template <class T> T* alloc(size_t count) {
    void* p = nullptr;
    if (cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) return nullptr;
    ptrs.push_back(p);
    return static_cast<T*>(p);
  }
};
}  // namespace chess
}  // namespace spb
