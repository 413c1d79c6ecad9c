// trajectory.cuh — the trajectory buffers of the self-play ply (ref: learner_concurrent.rs:179-238), shared by the
// Connect4 / tic-tac-toe engine (kernels.cuh, record spb_position) and the chess engine (chess_engine.cu, record
// spb_chess_position): per-slot in-progress histories on the device, one output buffer of finished games, and the order
// in which the drain (HostEngine::drain_trajectories, host_engine.hpp) and the gather hand them over: (game id, ply).
#pragma once
#include <algorithm>
#include <numeric>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/selfplay_b200.h"

namespace spb {

template <class Rec>
struct Trajectories {
  Rec* hist;                 // [G][max_ply]
  uint32_t* hist_len;        // [G]
  uint8_t* parked;           // [G]  0, or 1 | how the game ended << 1 (engine-specific): the game has ended but its trajectory
                             //      did not fit the output buffer; the slot is idle until the next self-play step emits it
  unsigned long long* game_id;     // [G]
  Rec* out;                  // [out_cap]
  unsigned long long* out_game;    // [out_cap]
  unsigned long long* out_cursor;  // [1]
  uint32_t* finished;        // [1]
  uint32_t out_cap;
  uint32_t max_ply;
  unsigned long long id_stride;
};

// Reserves `plies` records of the trajectory output buffer (lane 0; all lanes get the answer).  The cursor only moves
// when the whole trajectory fits, so every record below the cursor is fully written: a drain never sees a hole.
template <class Rec>
__device__ __forceinline__ bool reserve_output(const Trajectories<Rec>& P, uint32_t plies, int lane, unsigned long long* base_out) {
  unsigned long long base = ~0ull;
  if (lane == 0) {
    unsigned long long cur = *reinterpret_cast<volatile unsigned long long*>(P.out_cursor);
    for (;;) {
      if (cur + plies > P.out_cap) { base = ~0ull; break; }
      const unsigned long long seen = atomicCAS(P.out_cursor, cur, cur + plies);
      if (seen == cur) { base = cur; break; }
      cur = seen;
    }
  }
  base = __shfl_sync(0xffffffffu, base, 0);
  *base_out = base;
  return base != ~0ull;
}

// Bookkeeping of a slot whose trajectory has just been emitted (lane 0): the next game starts with an empty history and
// the slot's next game id.
template <class Rec>
__device__ __forceinline__ void finish_trajectory(const Trajectories<Rec>& P, uint32_t g) {
  atomicAdd(P.finished, 1u);
  P.hist_len[g] = 0;
  P.parked[g] = 0;
  P.game_id[g] += P.id_stride;
}

// Deterministic order of drained records: game id, then ply (games finish in a nondeterministic order on the device).
template <class Rec>
std::vector<size_t> record_order(const std::vector<Rec>& pos, const std::vector<unsigned long long>& ids) {
  std::vector<size_t> order(pos.size());
  std::iota(order.begin(), order.end(), (size_t)0);
  std::sort(order.begin(), order.end(), [&](size_t a, size_t b) {
    if (ids[a] != ids[b]) return ids[a] < ids[b];
    return pos[a].ply < pos[b].ply;
  });
  return order;
}

}  // namespace spb
