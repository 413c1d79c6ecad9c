// chess_engine.hpp — the host-side chess engine behind the spb_chess_* entry points (include/selfplay_b200.h): one
// `Mcts<chess Net>` + its `Vec<Tree<chess::State>>` on one GPU (ref: src/mcts.rs:41-44 over src/game/chess.rs and
// src/model/chess.rs).  Shared by chess.cu (rules entry points), chess_engine.cu (trees, search) and chess_net.cu
// (the 10 x 256 network); what it shares with the Connect4 / tic-tac-toe engine is in host_engine.hpp.
#pragma once
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "chess_tree.cuh"
#include "host_engine.hpp"

namespace spb {
namespace chess {
struct Net;   // chess_net.cu
}
}  // namespace spb

// The self-play trajectories P are allocated by the first spb_chess_selfplay_step (an engine that never plays does not
// pay for them); P.parked[g] = 1 | won << 1 | terminal side to move << 2 | adjudicated << 3.
struct spb_chess_engine : spb::HostEngine<spb::chess::CTrees, spb_chess_position, uint16_t> {
  spb_chess_engine() : HostEngine("spb_chess_") {}
  cudaStream_t stream2 = nullptr;   // the second half of the trees in the network pipeline
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  spb::chess::Net* net = nullptr;

  int32_t init();
  void release();
};
