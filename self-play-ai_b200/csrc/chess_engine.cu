// chess_engine.cu — chess trees and search behind the C ABI (include/selfplay_b200.h, spb_chess_*): BASELINE config 5.
// Device primitives: chess_tree.cuh (select / expand / backup / warp move generation), chess.cuh (rules).
//   Mcts::search (ref: src/mcts.rs:196-332)      -> k_chess_search_fused (DetEval / uniform: all simulations of a tree in
//                                                   one warp) and, for the network, the lock-step pair k_chess_select ->
//                                                   [chess_net.cu] -> k_chess_finish: exactly the reference's loop, one
//                                                   evaluator batch per simulation step over all trees
//   Tree::use_subtree (:161-192)                 -> reroot: k_chess_advance (breadth-first compaction into the other arena)
//   Tree::with_root_state (:86-89)               -> restart_tree: k_chess_reset
//   SelfPlayWorker::self_play
//     (learner_concurrent.rs:169-242)            -> k_chess_selfplay_step (pick, record, end / re-root) + the drain
#include "chess_engine.hpp"
#include "chess_net.cuh"
#include "root_noise.cuh"

namespace spb {
namespace chess {

constexpr int WARPS = 4;
constexpr int THREADS = WARPS * 32;
constexpr uint32_t SPLIT_MIN_TREES = 128;   // the network pipeline runs as two half-loops on two streams from 2 x this many trees on

using ChessSelfPlay = Trajectories<spb_chess_position>;
static_assert(sizeof(spb_chess_position) == 1624 && sizeof(spb_chess_position) % 8 == 0, "spb_chess_position layout");

// Tree::with_root_state (mcts.rs:86-89) for slot g by threads t = 0..nt-1: the root, the game history that travels with it
// (hist NULL: a game that starts at its root) and one unvisited root node.
__device__ __forceinline__ void restart_tree(const CTrees& T, uint32_t g, Pos root, const unsigned long long* hist, uint32_t t, uint32_t nt) {
  if (!hist) root.hist_len = 0;
  if (root.hist_len > SPB_CHESS_MAX_HISTORY) root.hist_len = SPB_CHESS_MAX_HISTORY;
  if (hist)
    for (uint32_t k = t; k < root.hist_len; k += nt) T.root_hist[(size_t)g * SPB_CHESS_MAX_HISTORY + k] = hist[k];
  if (t == 0) {
    T.root[g] = root;
    T.buf[g] = 0;
    T.live[g] = 1;
    T.n_nodes[g] = 1;
    T.leaf_depth[g] = 0;
    T.rec[0][(size_t)g * T.cap] = make_uint4(0u, 0u, 0u, 0u);
    T.meta[0][(size_t)g * T.cap] = make_uint2(NO_PARENT, make_meta(MOVE_NONE, 0, ST_UNVISITED));
    T.hash[0][(size_t)g * T.cap] = 0ull;
  }
}

// P.hist_len is null until the first self-play step; after it, a reset slot starts a new trajectory.
__global__ void k_chess_reset(CTrees T, ChessSelfPlay P, const uint32_t* slots, const Pos* roots, const unsigned long long* hist, uint32_t n) {
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  const uint32_t g = slots ? slots[i] : i;
  restart_tree(T, g, roots ? roots[i] : start_position(), hist ? hist + (size_t)i * SPB_CHESS_MAX_HISTORY : nullptr, threadIdx.x, blockDim.x);
  if (threadIdx.x == 0 && P.hist_len) {
    P.hist_len[g] = 0;
    P.parked[g] = 0;
  }
}

__device__ __forceinline__ void flush_counters(const CTrees& T, const unsigned long long* ctr, int lane) {
  if (lane == 0)
    for (int i = 0; i < CTR_COUNT; ++i)
      if (ctr[i]) atomicAdd(&T.counters[i], ctr[i]);
}

// What a simulation finds at its leaf (get_value_and_terminated, chess.rs:168-174, evaluated once per node): the legal
// moves in ws.moves, their hash, the repetition count; returns the node's status (ST_EXPANDED = not terminal).
__device__ __forceinline__ uint32_t visit_leaf(const CTrees& T, uint32_t g, const Pos& pos, int depth, int lane, WarpScratch& ws, int& n,
                                               unsigned long long& h, uint32_t& reps) {
  n = warp_legal_moves(pos, lane, ws, T.error);
  h = warp_list_hash(ws, n, lane);
  reps = warp_repetitions(h, T.root_hist + (size_t)g * SPB_CHESS_MAX_HISTORY, T.root[g].hist_len, ws, depth, lane);
  if (n == 0) return in_check(pos, pos.side) ? ST_WON : ST_TIED;     // chess.rs:156-157
  if (reps >= 3 || pos.fifty >= 100) return ST_TIED;                  // :159-160
  return ST_EXPANDED;
}

// Fused search (DetEval / uniform): all simulations of one tree inside one warp.
template <int EVAL>
__global__ void __launch_bounds__(THREADS) k_chess_search_fused(CTrees T, uint32_t num_searches) {
  __shared__ WarpScratch s_ws[WARPS];
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint32_t g = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (g >= T.G || !T.live[g]) return;
  const uint32_t b = T.buf[g];
  uint4* rec = T.rec[b] + (size_t)g * T.cap;
  uint2* meta = T.meta[b] + (size_t)g * T.cap;
  unsigned long long* hash = T.hash[b] + (size_t)g * T.cap;
  const Pos root = T.root[g];
  uint32_t n_nodes = T.n_nodes[g];
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  for (uint32_t s = 0; s < num_searches; ++s) {                        // mcts.rs:214
    Pos pos = root;
    uint32_t node, lmeta;
    int depth;
    if (!descend(rec, meta, hash, T.c, root_noise_of(T, g), lane, ws, pos, node, depth, lmeta, T.error)) break;
    ctr[CTR_SIMS] += 1;
    ctr[CTR_PATHSUM] += (unsigned)depth;
    uint32_t st = meta_status(lmeta);
    int n = 0;
    unsigned long long h = 0;
    uint32_t reps = 0;
    if (st == ST_UNVISITED) {
      st = visit_leaf(T, g, pos, depth, lane, ws, n, h, reps);
      if (st != ST_EXPANDED && lane == 0) {                            // terminal: remember it (mcts.rs:245 on every later visit)
        meta[node].y = make_meta(meta_move(lmeta), 0, st);
        hash[node] = h;
      }
    }
    float v;
    if (st != ST_EXPANDED) {
      v = st == ST_WON ? 1.0f : 0.0f;                                  // chess.rs:172
      ctr[CTR_TERMINAL] += 1;
    } else {
      // predict (model/mod.rs:36-98) by a built-in evaluator + mask_invalid_actions (chess.rs:251-271)
      const uint64_t dh = det_hash(pos);
      float sum = 0.0f;
      if (EVAL == SPB_EVAL_DET) {
        for (int i = lane; i < n; i += 32) sum += det_raw_prob(dh, policy_index(pos.side, ws.moves[i]));   // dyadic: exact in any order
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        v = det_value(dh);
      } else {
        sum = (float)n;
        v = 0.0f;
      }
      ctr[CTR_EVALS] += 1;
      const int side = pos.side;
      const bool ok = expand(rec, meta, hash, T.cap, n_nodes, node, ws, n, h, lane, [&](int i) {
        const float raw = EVAL == SPB_EVAL_DET ? det_raw_prob(dh, policy_index(side, ws.moves[i])) : 1.0f;
        return __fdiv_rn(raw, sum);
      });
      if (!ok) {
        if (lane == 0) atomicOr(T.error, (uint32_t)ERRBIT_POOL);
        break;
      }
      ctr[CTR_CHILDREN] += (unsigned)n;
    }
    __syncwarp();
    backup(rec, ws, depth, v, lane);
    __syncwarp();
  }
  if (lane == 0) T.n_nodes[g] = n_nodes;
  flush_counters(T, ctr, lane);
}

// EXTENSION (DESIGN.md §4.6): eta of every live root, one warp per slot, launched at the head of spb_chess_search (and by
// spb_chess_root_noise).  n = the root's legal-move count; the game id is P.game_id[g], or game_id_base + g (the value that
// array will hold) while the self-play buffers do not exist yet; the ply is the root's plies.
__global__ void __launch_bounds__(THREADS) k_chess_root_noise(CTrees T, const unsigned long long* game_id, unsigned long long game_id_base, float alpha,
                                                              unsigned long long seed) {
  __shared__ WarpScratch s_ws[WARPS];
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint32_t g = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (g >= T.G) return;
  if (!T.live[g]) {
    if (lane == 0) T.noise_n[g] = 0;
    return;
  }
  const Pos root = T.root[g];
  const uint32_t n = (uint32_t)warp_legal_moves(root, lane, ws, T.error);
  const unsigned long long id = game_id ? game_id[g] : game_id_base + g;
  warp_dirichlet<(MAX_MOVES + 31) / 32>(noise_key(seed, id, root.plies, n), n, alpha, lane, T.root_noise + (size_t)g * SPB_CHESS_MAX_MOVES,
                                        SPB_CHESS_MAX_MOVES);
  if (lane == 0) T.noise_n[g] = n;
}

// ---- lock-step pipeline for the network --------------------------------------------------------------------------
// k_chess_select: the select of one simulation per tree; terminal leaves are backed up at once, the others are stored
// with their legal moves as the tree's pending leaf and appended to the evaluator's work list (mcts.rs:236-252).
__global__ void __launch_bounds__(THREADS) k_chess_select(CTrees T, TreeRange R) {
  __shared__ WarpScratch s_ws[WARPS];
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint32_t g = R.g0 + blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (g >= R.g1 || !T.live[g]) return;
  const uint32_t b = T.buf[g];
  uint4* rec = T.rec[b] + (size_t)g * T.cap;
  uint2* meta = T.meta[b] + (size_t)g * T.cap;
  unsigned long long* hash = T.hash[b] + (size_t)g * T.cap;
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  Pos pos = T.root[g];
  uint32_t node, lmeta;
  int depth;
  if (!descend(rec, meta, hash, T.c, root_noise_of(T, g), lane, ws, pos, node, depth, lmeta, T.error)) return;
  ctr[CTR_SIMS] += 1;
  ctr[CTR_PATHSUM] += (unsigned)depth;
  uint32_t st = meta_status(lmeta);
  int n = 0;
  unsigned long long h = 0;
  uint32_t reps = 0;
  if (st == ST_UNVISITED) {
    st = visit_leaf(T, g, pos, depth, lane, ws, n, h, reps);
    if (st != ST_EXPANDED && lane == 0) {
      meta[node].y = make_meta(meta_move(lmeta), 0, st);
      hash[node] = h;
    }
  }
  if (st != ST_EXPANDED) {
    ctr[CTR_TERMINAL] += 1;
    __syncwarp();
    backup(rec, ws, depth, st == ST_WON ? 1.0f : 0.0f, lane);
  } else {
    ctr[CTR_EVALS] += 1;
    for (int i = lane; i < n; i += 32) T.leaf_moves[(size_t)g * MAX_MOVES + i] = ws.moves[i];
    for (int d = lane; d <= depth; d += 32) T.path[(size_t)g * MAX_DEPTH + d] = ws.path[d];
    if (lane == 0) {
      T.leaf_pos[g] = pos;
      T.leaf_node[g] = node;
      T.leaf_depth[g] = (uint32_t)depth | LEAF_PENDING;
      T.leaf_nmoves[g] = (uint32_t)n;
      T.leaf_reps[g] = reps;
      T.leaf_hash[g] = h;
      R.list[atomicAdd(R.count, 1u)] = g;
    }
  }
  flush_counters(T, ctr, lane);
}

// k_chess_finish: expand + backup of the evaluated leaf (mcts.rs:268-284).  Model::predict's tail (model/mod.rs:64-95):
// softmax over all 4,672 logits, then mask_invalid_actions = keep the legal cells and divide by their sum
// (chess.rs:251-271).  The normaliser of the softmax cancels in that division, so only the legal logits are read:
// prior_i = exp(l_i - m) / sum_legal exp(l_j - m), m = max over the legal logits.
// RAW = true (parity harness, SPB_FLAG_FORCE_SPLIT): eval_logits holds the raw probabilities of a built-in evaluator for the
// legal cells (k_chess_builtin_eval) and the prior is raw / sum, exactly as in the fused kernel.
template <bool RAW>
__global__ void __launch_bounds__(THREADS) k_chess_finish(CTrees T, TreeRange R) {
  __shared__ WarpScratch s_ws[WARPS];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  WarpScratch& ws = s_ws[w];
  // the exponentials of the legal logits live in the scratch's path-hash array, which this kernel does not use: 10 KB of
  // shared memory per block, so that a block fits next to a resident k_conv CTA (chess_net.cu)
  static_assert(sizeof(ws.phash) >= MAX_MOVES * sizeof(float), "phash too small for the priors");
  float* s_ev = reinterpret_cast<float*>(ws.phash);
  const uint32_t g = R.g0 + blockIdx.x * WARPS + w;
  if (g >= R.g1 || !T.live[g]) return;
  const uint32_t ld = T.leaf_depth[g];
  if (!(ld & LEAF_PENDING)) return;
  const int depth = (int)(ld & 0xFFu);
  const uint32_t b = T.buf[g];
  uint4* rec = T.rec[b] + (size_t)g * T.cap;
  uint2* meta = T.meta[b] + (size_t)g * T.cap;
  unsigned long long* hash = T.hash[b] + (size_t)g * T.cap;
  const uint32_t node = T.leaf_node[g];
  const int n = (int)T.leaf_nmoves[g];
  const int side = T.leaf_pos[g].side;
  const float* logits = T.eval_logits + (size_t)g * LOGIT_STRIDE;
  for (int i = lane; i < n; i += 32) ws.moves[i] = T.leaf_moves[(size_t)g * MAX_MOVES + i];
  for (int d = lane; d <= depth; d += 32) ws.path[d] = T.path[(size_t)g * MAX_DEPTH + d];
  __syncwarp();
  float mx = -INFINITY;
  for (int i = lane; i < n; i += 32) {
    const float l = logits[policy_index(side, ws.moves[i])];
    s_ev[i] = l;
    mx = fmaxf(mx, l);
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.0f;
  for (int i = lane; i < n; i += 32) {
    const float e = RAW ? s_ev[i] : __expf(s_ev[i] - mx);
    s_ev[i] = e;
    sum += e;                                                        // RAW: dyadic values, exact in any order
  }
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncwarp();
  uint32_t n_nodes = T.n_nodes[g];
  const float* ev = s_ev;
  const bool ok = expand(rec, meta, hash, T.cap, n_nodes, node, ws, n, T.leaf_hash[g], lane, [&](int i) { return __fdiv_rn(ev[i], sum); });
  if (!ok) {
    if (lane == 0) { atomicOr(T.error, (uint32_t)ERRBIT_POOL); T.leaf_depth[g] = 0; }
    return;
  }
  if (lane == 0) {
    T.n_nodes[g] = n_nodes;
    T.leaf_depth[g] = 0;
    atomicAdd(&T.counters[CTR_CHILDREN], (unsigned long long)n);
  }
  __syncwarp();
  backup(rec, ws, depth, T.eval_value[g], lane);
}

// Built-in evaluators for the lock-step pipeline (parity harness): the raw probabilities of the legal cells and the value of
// every pending leaf, where the network would have written its logits.
template <int EVAL>
__global__ void __launch_bounds__(THREADS) k_chess_builtin_eval(CTrees T, TreeRange R) {
  const int lane = threadIdx.x & 31;
  const uint32_t i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= *R.count) return;
  const uint32_t g = R.list[i];
  const Pos pos = T.leaf_pos[g];
  const uint64_t dh = det_hash(pos);
  const int n = (int)T.leaf_nmoves[g];
  float* logits = T.eval_logits + (size_t)g * LOGIT_STRIDE;
  for (int k = lane; k < n; k += 32) {
    const int idx = policy_index(pos.side, T.leaf_moves[(size_t)g * MAX_MOVES + k]);
    logits[idx] = EVAL == SPB_EVAL_DET ? det_raw_prob(dh, idx) : 1.0f;
  }
  if (lane == 0) T.eval_value[g] = EVAL == SPB_EVAL_DET ? det_value(dh) : 0.0f;
}

// ---- results / re-rooting ----------------------------------------------------------------------------------------
__global__ void k_chess_root_children(CTrees T, uint16_t* moves, uint32_t* counts, uint32_t* ids, uint32_t* n_out) {
  const uint32_t g = blockIdx.x;
  if (g >= T.G) return;
  uint32_t nc = 0, fc = 0;
  const uint32_t b = T.buf[g];
  const uint4* rec = T.rec[b] + (size_t)g * T.cap;
  const uint2* meta = T.meta[b] + (size_t)g * T.cap;
  if (T.live[g] && meta_status(meta[0].y) == ST_EXPANDED) { nc = meta_nc(meta[0].y); fc = rec[0].w; }
  for (uint32_t i = threadIdx.x; i < MAX_MOVES; i += blockDim.x) {
    const bool in = i < nc;
    moves[(size_t)g * MAX_MOVES + i] = in ? (uint16_t)meta_move(meta[fc + i].y) : MOVE_NONE;
    counts[(size_t)g * MAX_MOVES + i] = in ? rec[fc + i].x : 0u;
    ids[(size_t)g * MAX_MOVES + i] = in ? fc + i : 0u;
  }
  if (threadIdx.x == 0) n_out[g] = nc;
}

// use_subtree (mcts.rs:161-192) for a child of the root: breadth-first copy of the kept subtree into the other arena,
// ids assigned in queue order with every node's children contiguous and in their old order.  One warp per tree; a
// window of 32 copied nodes per round: a scan of their child counts gives each its new first_child, then the warp
// copies the children of the 32 nodes one node after the other (lanes stride over up to 218 children).  A copied node
// keeps its OLD first_child in rec.w until its own turn in the window.  The root position advances by the child's move
// and the hash of the old root's move list joins the game history (chess.rs:121-122).  The caller has checked that `id`
// is a child of the root and that the history has room; lane 0 writes the new root to *out_state when it is not null.
__device__ __forceinline__ void reroot(const CTrees& T, uint32_t g, uint32_t id, int lane, Pos* out_state) {
  const uint32_t b = T.buf[g], nb = b ^ 1u;
  const uint4* orec = T.rec[b] + (size_t)g * T.cap;
  const uint2* ometa = T.meta[b] + (size_t)g * T.cap;
  const unsigned long long* ohash = T.hash[b] + (size_t)g * T.cap;
  uint4* nrec = T.rec[nb] + (size_t)g * T.cap;
  uint2* nmeta = T.meta[nb] + (size_t)g * T.cap;
  unsigned long long* nhash = T.hash[nb] + (size_t)g * T.cap;
  const Move mv = (Move)meta_move(ometa[id].y);
  if (lane == 0) {
    Pos root = T.root[g];
    T.root_hist[(size_t)g * SPB_CHESS_MAX_HISTORY + root.hist_len] = ohash[0];
    const uint32_t hl = root.hist_len + 1;
    root = apply_move(root, mv);
    root.hist_len = hl;
    T.root[g] = root;
    if (out_state) *out_state = root;
    nrec[0] = orec[id];
    nmeta[0] = make_uint2(NO_PARENT, ometa[id].y);
    nhash[0] = ohash[id];
  }
  __syncwarp();
  uint32_t n_new = 1, j0 = 0;
  while (j0 < n_new) {
    const uint32_t in_window = min(32u, n_new - j0);                   // nodes copied so far that still await their turn
    const uint32_t j = j0 + lane;
    uint32_t nc = 0, old_fc = 0;
    if ((uint32_t)lane < in_window) {
      const uint32_t my = nmeta[j].y;
      if (meta_status(my) == ST_EXPANDED) { nc = meta_nc(my); old_fc = nrec[j].w; }
    }
    int total;
    const uint32_t new_fc = n_new + (uint32_t)warp_excl_scan((int)nc, lane, &total);
    if (n_new + (uint32_t)total > T.cap) {                             // cannot happen: the subtree is part of an arena of <= cap nodes
      if (lane == 0) atomicOr(T.error, (uint32_t)ERRBIT_BOUNDS | (43u << 8));
      break;
    }
    if (nc) nrec[j].w = new_fc;
    for (uint32_t l = 0; l < in_window; ++l) {
      const uint32_t cnc = __shfl_sync(0xffffffffu, nc, l), cold = __shfl_sync(0xffffffffu, old_fc, l), cnew = __shfl_sync(0xffffffffu, new_fc, l);
      for (uint32_t k = lane; k < cnc; k += 32) {
        nrec[cnew + k] = orec[cold + k];
        nmeta[cnew + k] = make_uint2(j0 + l, ometa[cold + k].y);
        nhash[cnew + k] = ohash[cold + k];
      }
    }
    n_new += (uint32_t)total;
    j0 += in_window;
    __syncwarp();
  }
  if (lane == 0) {
    T.n_nodes[g] = n_new;
    T.buf[g] = (uint8_t)nb;
    T.leaf_depth[g] = 0;
  }
}

__global__ void __launch_bounds__(THREADS) k_chess_advance(CTrees T, const uint32_t* slots, const uint32_t* node_ids, uint32_t n, Pos* out_states,
                                                           int32_t* out_err) {
  const int lane = threadIdx.x & 31;
  const uint32_t i = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (i >= n) return;
  const uint32_t g = slots ? slots[i] : i;
  const uint2* ometa = T.meta[T.buf[g]] + (size_t)g * T.cap;
  const uint32_t id = node_ids[i];
  int32_t err = SPB_OK;
  if (!T.live[g] || id == 0 || id >= T.n_nodes[g] || ometa[id].x != 0u) err = SPB_ERR_ARG;        // must be a child of the root
  else if (T.root[g].hist_len >= SPB_CHESS_MAX_HISTORY) err = SPB_ERR_STATE;
  if (err != SPB_OK) {
    if (lane == 0) { out_err[i] = err; if (out_states) out_states[i] = T.root[g]; }
    return;
  }
  if (lane == 0) out_err[i] = SPB_OK;
  reroot(T, g, id, lane, out_states ? out_states + i : nullptr);
}

// ---- self-play ply (ref: learner_concurrent.rs:179-238) ------------------------------------------------------------
// Emits the finished game of slot g (learner_concurrent.rs:200-230) and restarts or retires the slot.  pk: how the game
// ended, as stored in P.parked.  The outcome is the value of the terminal state (chess.rs:172: +1 when its side to move is
// checkmated, 0 for a tie) for positions with that side to move, its negation for the others (:214-226).
__device__ __forceinline__ void emit_game(const CTrees& T, const ChessSelfPlay& P, uint32_t g, uint32_t plies, uint32_t pk, unsigned long long base,
                                          const Pos* restart_roots, const unsigned long long* restart_hist, int lane) {
  const int value = ((pk >> 1) & 1u) ? 1 : 0;
  const uint32_t term_side = (pk >> 2) & 1u;
  const uint8_t flags = ((pk >> 3) & 1u) ? (uint8_t)SPB_CHESS_POS_ADJUDICATED : (uint8_t)0;
  spb_chess_position* hist = P.hist + (size_t)g * P.max_ply;
  SPB_ASSERT(T.error, base + plies <= P.out_cap && plies <= P.max_ply, 44);
  for (uint32_t i = lane; i < plies; i += 32) {
    hist[i].outcome = (int8_t)(hist[i].state.side == term_side ? value : -value);
    hist[i].flags = flags;
  }
  __syncwarp();
  constexpr uint32_t WORDS = sizeof(spb_chess_position) / 8;          // records copied as 8-byte words by the whole warp
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(hist);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(P.out + base);
  for (uint32_t k = lane; k < plies * WORDS; k += 32) dst[k] = src[k];
  const unsigned long long id = P.game_id[g];
  for (uint32_t i = lane; i < plies; i += 32) P.out_game[base + i] = id;
  __syncwarp();
  if (lane == 0) finish_trajectory(P, g);
  if (restart_roots)
    restart_tree(T, g, restart_roots[g], restart_hist ? restart_hist + (size_t)g * SPB_CHESS_MAX_HISTORY : nullptr, (uint32_t)lane, 32u);
  else if (lane == 0)
    T.live[g] = 0;                                                    // trees_vec.remove(i), :230
}

// One warp per slot: pick a root child (greedy last-max or ∝ N^temperature), record the root in the slot's history, then end
// the game (terminal child, or the history cap) or re-root at the child.
__global__ void __launch_bounds__(THREADS) k_chess_selfplay_step(CTrees T, ChessSelfPlay P, int rule, float temperature, unsigned long long seed,
                                                                 const Pos* restart_roots, const unsigned long long* restart_hist) {
  __shared__ WarpScratch s_ws[WARPS];
  const int lane = threadIdx.x & 31;
  WarpScratch& ws = s_ws[threadIdx.x >> 5];
  const uint32_t g = blockIdx.x * WARPS + (threadIdx.x >> 5);
  if (g >= T.G) return;
  const uint32_t parked = P.parked[g];
  if (parked) {
    // A game that ended in an earlier call while the output buffer was full: the slot has been idle since; emit now.
    const uint32_t plies = P.hist_len[g];
    unsigned long long base;
    if (reserve_output(P, plies, lane, &base)) emit_game(T, P, g, plies, parked, base, restart_roots, restart_hist, lane);
    else if (lane == 0) atomicOr(T.error, (uint32_t)ERRBIT_TRAJ_FULL);
    return;
  }
  if (!T.live[g]) return;
  const uint32_t b = T.buf[g];
  const uint4* rec = T.rec[b] + (size_t)g * T.cap;
  const uint2* meta = T.meta[b] + (size_t)g * T.cap;
  const unsigned long long* hash = T.hash[b] + (size_t)g * T.cap;
  const uint32_t y0 = meta[0].y;
  if (meta_status(y0) != ST_EXPANDED) return;                         // nothing searched yet / terminal root
  const uint32_t nc = meta_nc(y0), fc = rec[0].w;
  const Pos root = T.root[g];
  const uint32_t ply = P.hist_len[g];
  int chosen;
  if (rule == SPB_MOVE_TEMPERATURE) {
    // learner_concurrent.rs:189-194: WeightedIndex over count^temperature, as k_selfplay_step draws it: an inclusive scan
    // of the weights in child order (lanes stride over the children, 32 per round, with a carry across rounds), the ball
    // u = U[0,1) * total, the first child whose prefix sum exceeds u.  The counter behind U is (seed, game id, ply).
    constexpr int ROUNDS = MAX_MOVES / 32;
    float incl[ROUNDS];
    uint32_t positive = 0;
    float carry = 0.0f;
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      incl[r] = carry;
      if ((uint32_t)r * 32u < nc) {
        const uint32_t i = (uint32_t)r * 32u + (uint32_t)lane;
        const float w = i < nc ? powf((float)rec[fc + i].x, temperature) : 0.0f;
        float x = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const float t = __shfl_up_sync(0xffffffffu, x, o);
          if (lane >= o) x += t;
        }
        incl[r] = carry + x;
        if (w > 0.0f) positive |= 1u << r;
        carry = __shfl_sync(0xffffffffu, incl[r], 31);
      }
    }
    const unsigned long long h = mix64(seed ^ mix64((P.game_id[g] << 9) + ply));   // ply < 512 = P.max_ply
    const float u = (float)(h >> 40) * (1.0f / 16777216.0f) * carry;
    chosen = (int)nc - 1;
    bool found = false;
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
      const uint32_t i = (uint32_t)r * 32u + (uint32_t)lane;
      const unsigned ball = __ballot_sync(0xffffffffu, i < nc && u < incl[r] && ((positive >> r) & 1u));
      if (ball && !found) { chosen = r * 32 + __ffs((int)ball) - 1; found = true; }
    }
  } else {
    // main.rs:108-112: max_by(total_cmp) over visit counts -> the LAST maximal child
    float best = -INFINITY;
    int best_i = -1;
    for (uint32_t i = lane; i < nc; i += 32) {
      const float s = (float)rec[fc + i].x;
      if (s >= best) { best = s; best_i = (int)i; }
    }
    chosen = warp_argmax_last32(best, best_i);
  }
  // learner_concurrent.rs:197-198: push the root and its visit counts (ply < P.max_ply: a game ends at P.max_ply records)
  SPB_ASSERT(T.error, ply < P.max_ply, 45);
  spb_chess_position* hr = P.hist + (size_t)g * P.max_ply + ply;
  static_assert(sizeof(Pos) == 80, "spb_chess_state is copied as 10 words");
  if (lane < 10) reinterpret_cast<unsigned long long*>(&hr->state)[lane] = reinterpret_cast<const unsigned long long*>(T.root + g)[lane];
  for (uint32_t i = lane; i < MAX_MOVES; i += 32) {
    const bool in = i < nc;
    hr->visit_counts[i] = in ? rec[fc + i].x : 0u;
    hr->moves[i] = in ? (uint16_t)meta_move(meta[fc + i].y) : MOVE_NONE;
  }
  const uint32_t reps = warp_repetitions(hash[0], T.root_hist + (size_t)g * SPB_CHESS_MAX_HISTORY, root.hist_len, ws, 0, lane);
  if (lane == 0) {
    hr->n_moves = (uint16_t)nc;
    hr->ply = (uint16_t)ply;
    hr->repetitions = (uint8_t)min(reps, 255u);
    hr->outcome = 0;
    hr->flags = 0;
    hr->reserved = 0;
  }
  // the chosen child's status: cached by the search, or found now as the search would (history of the root + the root)
  const uint32_t child = fc + (uint32_t)chosen;
  const uint32_t cy = meta[child].y;
  uint32_t cst = meta_status(cy);
  if (cst == ST_UNVISITED) {
    if (lane == 0) ws.phash[0] = hash[0];
    __syncwarp();
    int n;
    unsigned long long lh;
    uint32_t lr;
    cst = visit_leaf(T, g, apply_move(root, (Move)meta_move(cy)), 1, lane, ws, n, lh, lr);
  }
  __syncwarp();                                                       // the record is complete before emit_game reads it
  const uint32_t plies = ply + 1;
  const bool over = cst == ST_TIED || cst == ST_WON;
  // the device keeps SPB_CHESS_MAX_HISTORY plies of history and records per game; the reference has no cap
  const bool capped = !over && (root.hist_len >= SPB_CHESS_MAX_HISTORY || plies >= P.max_ply);
  if (over || capped) {
    const uint32_t pk = 1u | ((cst == ST_WON ? 1u : 0u) << 1) | (((uint32_t)root.side ^ 1u) << 2) | ((capped ? 1u : 0u) << 3);
    unsigned long long base;
    if (reserve_output(P, plies, lane, &base)) {
      emit_game(T, P, g, plies, pk, base, restart_roots, restart_hist, lane);
    } else if (lane == 0) {
      // parked: idle with its history until a later call emits it (the caller drains in between); nothing is lost
      P.hist_len[g] = plies;
      P.parked[g] = (uint8_t)pk;
      T.live[g] = 0;
      atomicOr(T.error, (uint32_t)ERRBIT_TRAJ_FULL);
    }
  } else {
    if (lane == 0) P.hist_len[g] = plies;
    reroot(T, g, child, lane, nullptr);                               // :233-234
  }
}

// arena[node_id].state (mcts.rs:22): the moves from the root to the node, replayed.
__global__ void k_chess_get_state(CTrees T, uint32_t g, uint32_t node_id, Pos* out, int32_t* err) {
  const uint32_t b = T.buf[g];
  const uint2* meta = T.meta[b] + (size_t)g * T.cap;
  if (!T.live[g] || node_id >= T.n_nodes[g]) { *err = SPB_ERR_ARG; return; }
  Move mv[MAX_DEPTH];
  int d = 0;
  for (uint32_t v = node_id; v != 0; v = meta[v].x) {
    if (d >= MAX_DEPTH) { *err = SPB_ERR_STATE; return; }
    mv[d++] = (Move)meta_move(meta[v].y);
  }
  Pos p = T.root[g];
  const uint32_t hl = p.hist_len;
  while (d > 0) p = apply_move(p, mv[--d]);
  p.hist_len = hl;   // the history that travels with the root; the path's own positions are not exported
  *out = p;
  *err = SPB_OK;
}

__global__ void k_chess_node_stats(CTrees T, uint32_t g, uint32_t node_id, uint32_t* out) {
  const uint32_t b = T.buf[g];
  if (!T.live[g] || node_id >= T.n_nodes[g]) { out[7] = 1; return; }
  const uint4 r = T.rec[b][(size_t)g * T.cap + node_id];
  const uint2 m = T.meta[b][(size_t)g * T.cap + node_id];
  out[0] = r.x; out[1] = r.y; out[2] = r.z;
  out[3] = meta_status(m.y) == ST_EXPANDED ? r.w : 0u;
  out[4] = meta_status(m.y) == ST_EXPANDED ? meta_nc(m.y) : 0u;
  out[5] = meta_move(m.y);
  out[6] = meta_status(m.y);
  out[7] = 0;
}

__global__ void k_chess_nodes_live(CTrees T, unsigned long long* out) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < T.G && T.live[g]) { atomicAdd(out, (unsigned long long)T.n_nodes[g]); atomicMax(out + 1, (unsigned long long)T.n_nodes[g]); }
}

}  // namespace chess
}  // namespace spb

using namespace spb;
namespace ch = spb::chess;

// Everything but the self-play trajectories, which the first spb_chess_selfplay_step allocates.
int32_t spb_chess_engine::init() {
  int32_t rc = open_device();
  if (rc) return rc;
  SPB_CUDA(this, cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
  SPB_CUDA(this, cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
  SPB_CUDA(this, cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
  T.G = cfg.num_games; T.cap = cfg.max_nodes_per_tree; T.c = cfg.c;
  const size_t G = T.G, pool = G * (size_t)T.cap;
  for (int b = 0; b < 2 && !rc; ++b) {
    if (!rc) rc = dalloc(&T.rec[b], pool);
    if (!rc) rc = dalloc(&T.meta[b], pool);
    if (!rc) rc = dalloc(&T.hash[b], pool);
  }
  if (!rc) rc = dalloc(&T.root, G);
  if (!rc) rc = dalloc(&T.root_hist, G * SPB_CHESS_MAX_HISTORY);
  if (!rc) rc = dalloc(&T.n_nodes, G);
  if (!rc) rc = dalloc(&T.buf, G);
  if (!rc) rc = dalloc(&T.live, G);
  if (!rc) rc = dalloc(&T.counters, (size_t)CTR_COUNT);
  if (!rc) rc = dalloc(&T.error, 1);
  if (!rc) rc = dalloc(&T.leaf_node, G);
  if (!rc) rc = dalloc(&T.leaf_depth, G);
  if (!rc) rc = dalloc(&T.path, G * ch::MAX_DEPTH);
  if (!rc) rc = dalloc(&T.leaf_pos, G);
  if (!rc) rc = dalloc(&T.leaf_moves, G * ch::MAX_MOVES);
  if (!rc) rc = dalloc(&T.leaf_nmoves, G);
  if (!rc) rc = dalloc(&T.leaf_reps, G);
  if (!rc) rc = dalloc(&T.leaf_hash, G);
  if (!rc) rc = dalloc(&T.eval_list, G);
  if (!rc) rc = dalloc(&T.eval_count, 2);
  if (!rc) rc = dalloc(&T.eval_value, G);
  if (!rc && (cfg.evaluator == SPB_EVAL_NET || (cfg.flags & SPB_FLAG_FORCE_SPLIT))) rc = dalloc(&T.eval_logits, G * (size_t)ch::LOGIT_STRIDE);
  if (!rc) rc = dalloc(&d_rc_moves, G * ch::MAX_MOVES);
  if (!rc) rc = dalloc(&d_rc_counts, G * ch::MAX_MOVES);
  if (!rc) rc = dalloc(&d_rc_ids, G * ch::MAX_MOVES);
  if (!rc) rc = dalloc(&d_rc_n, G);
  if (!rc) rc = dalloc(&d_misc, 4);
  if (rc) return rc;
  SPB_CUDA(this, cudaMemsetAsync(T.live, 0, G, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.buf, 0, G, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.n_nodes, 0, G * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.leaf_depth, 0, G * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.counters, 0, CTR_COUNT * 8, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.error, 0, 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.eval_count, 0, 8, stream));
  SPB_CUDA(this, cudaStreamSynchronize(stream));
  return SPB_OK;
}

// The second stream rejoins the first before every spb_chess_search returns, so the wait in HostEngine::release covers it.
void spb_chess_engine::release() {
  HostEngine::release();
  ch::net_destroy(net);
  if (stream2) cudaStreamDestroy(stream2);
  if (ev_fork) cudaEventDestroy(ev_fork);
  if (ev_join) cudaEventDestroy(ev_join);
}

extern "C" {

// The checks of spb_chess_create beyond HostEngine::config_error (max_nodes_per_tree 0 already replaced by its default).
static const char* config_error(const spb_config& c) {
  if (const char* m = spb_chess_engine::config_error(c)) return m;
  if (c.game != SPB_GAME_CHESS) return "spb_chess_create needs game = SPB_GAME_CHESS";
  if (c.num_games == 0 || c.num_games > (1u << 20)) return "num_games out of range";
  if (c.leaves_per_tree != 1) return "chess search runs one leaf per tree per step";
  if (c.max_nodes_per_tree < 512 || c.max_nodes_per_tree > (1u << 24)) return "max_nodes_per_tree out of range";
  return nullptr;
}

int32_t spb_chess_create(const spb_config* cfg, spb_chess_engine** out) {
  if (!cfg || !out) { g_create_error = "null argument"; return SPB_ERR_ARG; }
  *out = nullptr;
  spb_config c = *cfg;
  if (c.max_nodes_per_tree == 0) c.max_nodes_per_tree = 32768;
  if (const char* m = config_error(c)) { g_create_error = m; return SPB_ERR_ARG; }
  return spb_chess_engine::create(c, out);
}

int32_t spb_chess_destroy(spb_chess_engine* e) {
  if (!e) return SPB_ERR_ARG;
  spb_chess_comm_destroy(e);
  e->release();
  delete e;
  return SPB_OK;
}

const char* spb_chess_last_error(const spb_chess_engine* e) { return spb_chess_engine::last_error(e); }

// The roots of spb_chess_reset_games / spb_chess_selfplay_step (history: [n][SPB_CHESS_MAX_HISTORY], nullable): checked, then
// copied with the slots to the stage.  Each device pointer is set when its host array is given.
static int32_t stage_roots(spb_chess_engine* e, const uint32_t* slots, const spb_chess_state* roots, const uint64_t* history, uint32_t n,
                           uint32_t** d_slots, ch::Pos** d_roots, unsigned long long** d_hist) {
  if (roots) for (uint32_t i = 0; i < n; ++i) {
    SPB_ARG(e, roots[i].side <= 1 && roots[i].ep <= 64, "malformed root state");
    uint64_t kings[2] = {roots[i].piece[5] & roots[i].color[0], roots[i].piece[5] & roots[i].color[1]};
    SPB_ARG(e, kings[0] && !(kings[0] & (kings[0] - 1)) && kings[1] && !(kings[1] & (kings[1] - 1)), "root state needs one king per side");
    SPB_ARG(e, history || roots[i].hist_len == 0, "root with hist_len > 0 needs its history");
    SPB_ARG(e, roots[i].hist_len <= SPB_CHESS_MAX_HISTORY, "hist_len > SPB_CHESS_MAX_HISTORY");
  }
  const size_t hist_bytes = (size_t)n * SPB_CHESS_MAX_HISTORY * 8;
  StageLayout L;
  const size_t o_slots = L.take(slots ? (size_t)n * 4 : 0), o_roots = L.take(roots ? (size_t)n * sizeof(ch::Pos) : 0), o_hist = L.take(history ? hist_bytes : 0);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  if (slots) SPB_CUDA(e, cudaMemcpyAsync(*d_slots = e->d_at<uint32_t>(o_slots), slots, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  if (roots) SPB_CUDA(e, cudaMemcpyAsync(*d_roots = e->d_at<ch::Pos>(o_roots), roots, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(*d_hist = e->d_at<unsigned long long>(o_hist), history, hist_bytes, cudaMemcpyHostToDevice, e->stream));
  return SPB_OK;
}

int32_t spb_chess_reset_games(spb_chess_engine* e, const uint32_t* slots, uint32_t n, const spb_chess_state* roots, const uint64_t* history) {
  SPB_GUARD(e);
  SPB_ARG(e, n <= e->T.G, "more slots than games");
  SPB_ARG(e, !(history && !roots), "history without roots");
  if (n == 0) return SPB_OK;
  if (slots) for (uint32_t i = 0; i < n; ++i) SPB_ARG(e, slots[i] < e->T.G, "slot out of range");
  uint32_t* d_slots = nullptr; ch::Pos* d_roots = nullptr; unsigned long long* d_hist = nullptr;
  if (int32_t rc = stage_roots(e, slots, roots, history, n, &d_slots, &d_roots, &d_hist)) return rc;
  ch::k_chess_reset<<<n, 64, 0, e->stream>>>(e->T, e->P, d_slots, d_roots, d_hist, n);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

// EXTENSION (DESIGN.md §4.6): eta of every live root into T.root_noise (k_chess_root_noise).
static int32_t launch_chess_root_noise(spb_chess_engine* e) {
  ch::k_chess_root_noise<<<(e->T.G + ch::WARPS - 1) / ch::WARPS, ch::THREADS, 0, e->stream>>>(e->T, e->P.game_id, (unsigned long long)e->cfg.game_id_base,
                                                                                             e->noise_alpha, e->noise_seed);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  return SPB_OK;
}

int32_t spb_chess_set_root_noise(spb_chess_engine* e, float alpha, float epsilon, uint64_t seed) {
  SPB_GUARD(e);
  return e->set_root_noise(alpha, epsilon, seed, SPB_CHESS_MAX_MOVES);
}

int32_t spb_chess_root_noise(spb_chess_engine* e, uint32_t slot, float* eta, uint32_t* n) {
  SPB_GUARD(e);
  return e->root_noise(slot, eta, n, SPB_CHESS_MAX_MOVES, [e] { return launch_chess_root_noise(e); });
}

int32_t spb_chess_search(spb_chess_engine* e, uint32_t num_searches) {
  SPB_GUARD(e);
  if (num_searches == 0) return SPB_OK;
  const uint32_t blocks = (e->T.G + ch::WARPS - 1) / ch::WARPS;
  SPB_CUDA(e, cudaEventRecord(e->ev0, e->stream));
  if (e->T.root_noise) { const int32_t rc = launch_chess_root_noise(e); if (rc) return rc; }   // eta of every root, before any descent
  const ch::TreeRange all{0u, e->T.G, e->T.eval_list, e->T.eval_count};
  if (e->cfg.evaluator == SPB_EVAL_NET) {
    SPB_ARG(e, e->net && ch::net_loaded(e->net), "no weights loaded (spb_chess_load_weights)");
    // mcts.rs:214: one evaluator batch per simulation step.  Trees never interact, so the lock-step loop runs separately
    // over the two halves of the trees, on two streams: while the convolutions of one half hold the tensor pipes, the
    // select / expand + backup kernels of the other half run in the SMs' spare issue slots and shared memory (a k_conv CTA
    // leaves room for them).  Results are those of one loop over all trees (tests: node for node against the oracle).
    const uint32_t G = e->T.G, G0 = (G + 1u) / 2u;
    const bool split = G >= 2u * ch::SPLIT_MIN_TREES && !(e->cfg.flags & SPB_FLAG_LOCKSTEP);
    const ch::TreeRange half[2] = {{0u, split ? G0 : G, e->T.eval_list, e->T.eval_count}, {G0, G, e->T.eval_list + G0, e->T.eval_count + 1}};
    const int nh = split ? 2 : 1;
    cudaStream_t st[2] = {e->stream, e->stream2};
    if (split) {
      SPB_CUDA(e, cudaEventRecord(e->ev_fork, e->stream));
      SPB_CUDA(e, cudaStreamWaitEvent(e->stream2, e->ev_fork, 0));
    }
    auto enqueue = [&]() -> int32_t {
      for (uint32_t s = 0; s < num_searches; ++s) {
        for (int h = 0; h < nh; ++h) {
          const ch::TreeRange& R = half[h];
          const uint32_t hb = (R.g1 - R.g0 + ch::WARPS - 1) / ch::WARPS;
          SPB_CUDA(e, cudaMemsetAsync(R.count, 0, 4, st[h]));
          ch::k_chess_select<<<hb, ch::THREADS, 0, st[h]>>>(e->T, R);
          SPB_CUDA(e, cudaGetLastError());
          uint32_t launched = 0;
          const int32_t rc = ch::net_forward_leaves(e, h, R.list, R.count, st[h], &launched);
          if (rc) return rc;
          ch::k_chess_finish<false><<<hb, ch::THREADS, 0, st[h]>>>(e->T, R);
          SPB_CUDA(e, cudaGetLastError());
          e->launches += 2 + launched;
        }
      }
      return SPB_OK;
    };
    const int32_t rc_loop = enqueue();
    if (split) {                                                       // the second stream rejoins the engine's stream, also after an error
      cudaError_t je = cudaEventRecord(e->ev_join, e->stream2);
      if (je == cudaSuccess) je = cudaStreamWaitEvent(e->stream, e->ev_join, 0);
      if (je != cudaSuccess && rc_loop == SPB_OK) { e->set_error(std::string("chess search: ") + cudaGetErrorString(je)); return SPB_ERR_CUDA; }
    }
    if (rc_loop) return rc_loop;
  } else if (e->cfg.flags & SPB_FLAG_FORCE_SPLIT) {
    // parity harness: the built-in evaluators through the kernels of the network pipeline (select -> evaluate -> finish)
    for (uint32_t s = 0; s < num_searches; ++s) {
      SPB_CUDA(e, cudaMemsetAsync(e->T.eval_count, 0, 4, e->stream));
      ch::k_chess_select<<<blocks, ch::THREADS, 0, e->stream>>>(e->T, all);
      if (e->cfg.evaluator == SPB_EVAL_DET) ch::k_chess_builtin_eval<SPB_EVAL_DET><<<blocks, ch::THREADS, 0, e->stream>>>(e->T, all);
      else ch::k_chess_builtin_eval<SPB_EVAL_UNIFORM><<<blocks, ch::THREADS, 0, e->stream>>>(e->T, all);
      ch::k_chess_finish<true><<<blocks, ch::THREADS, 0, e->stream>>>(e->T, all);
      SPB_CUDA(e, cudaGetLastError());
      e->launches += 3;
    }
  } else {
    if (e->cfg.evaluator == SPB_EVAL_DET) ch::k_chess_search_fused<SPB_EVAL_DET><<<blocks, ch::THREADS, 0, e->stream>>>(e->T, num_searches);
    else ch::k_chess_search_fused<SPB_EVAL_UNIFORM><<<blocks, ch::THREADS, 0, e->stream>>>(e->T, num_searches);
    SPB_CUDA(e, cudaGetLastError());
    ++e->launches;
  }
  SPB_CUDA(e, cudaEventRecord(e->ev1, e->stream));
  const int32_t rc = e->check_device_errors();
  if (rc) return rc;
  SPB_CUDA(e, cudaEventElapsedTime(&e->last_search_ms, e->ev0, e->ev1));
  return SPB_OK;
}

int32_t spb_chess_last_search_ms(spb_chess_engine* e, float* ms) {
  SPB_GUARD(e);
  SPB_ARG(e, ms, "null argument");
  *ms = e->last_search_ms;
  return SPB_OK;
}

static int32_t fetch_root_children(spb_chess_engine* e) {
  ch::k_chess_root_children<<<e->T.G, 64, 0, e->stream>>>(e->T, e->d_rc_moves, e->d_rc_counts, e->d_rc_ids, e->d_rc_n);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  return SPB_OK;
}

int32_t spb_chess_root_children_all(spb_chess_engine* e, uint16_t* moves, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children) {
  SPB_GUARD(e);
  int32_t rc = fetch_root_children(e);
  if (rc) return rc;
  const size_t G = e->T.G, M = ch::MAX_MOVES;
  if (moves) SPB_CUDA(e, cudaMemcpyAsync(moves, e->d_rc_moves, G * M * 2, cudaMemcpyDeviceToHost, e->stream));
  if (visit_counts) SPB_CUDA(e, cudaMemcpyAsync(visit_counts, e->d_rc_counts, G * M * 4, cudaMemcpyDeviceToHost, e->stream));
  if (child_ids) SPB_CUDA(e, cudaMemcpyAsync(child_ids, e->d_rc_ids, G * M * 4, cudaMemcpyDeviceToHost, e->stream));
  if (n_children) SPB_CUDA(e, cudaMemcpyAsync(n_children, e->d_rc_n, G * 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_root_children(spb_chess_engine* e, uint32_t slot, uint16_t* moves, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children) {
  SPB_GUARD(e);
  SPB_ARG(e, slot < e->T.G, "slot out of range");
  SPB_ARG(e, n_children, "null argument");
  int32_t rc = fetch_root_children(e);
  if (rc) return rc;
  const size_t M = ch::MAX_MOVES;
  if (moves) SPB_CUDA(e, cudaMemcpyAsync(moves, e->d_rc_moves + slot * M, M * 2, cudaMemcpyDeviceToHost, e->stream));
  if (visit_counts) SPB_CUDA(e, cudaMemcpyAsync(visit_counts, e->d_rc_counts + slot * M, M * 4, cudaMemcpyDeviceToHost, e->stream));
  if (child_ids) SPB_CUDA(e, cudaMemcpyAsync(child_ids, e->d_rc_ids + slot * M, M * 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(n_children, e->d_rc_n + slot, 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

// Policy of Mcts::search's result (mcts.rs:315-328): the root children's visit counts scattered into the 73x8x8 table by
// set_prob (chess.rs:505-514), then normalize (divide by the sum, chess.rs:516-518).
int32_t spb_chess_root_policy(spb_chess_engine* e, uint32_t slot, float* out) {
  SPB_GUARD(e);
  SPB_ARG(e, out, "null argument");
  uint16_t mv[ch::MAX_MOVES];
  uint32_t cnt[ch::MAX_MOVES], n = 0;
  int32_t rc = spb_chess_root_children(e, slot, mv, cnt, nullptr, &n);
  if (rc) return rc;
  ch::Pos root;
  SPB_CUDA(e, cudaMemcpyAsync(&root, e->T.root + slot, sizeof root, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  std::memset(out, 0, sizeof(float) * SPB_CHESS_POLICY_SIZE);
  float sum = 0.0f;
  for (uint32_t i = 0; i < n; ++i) sum += (float)cnt[i];               // integers: exact in any order
  for (uint32_t i = 0; i < n; ++i) out[ch::policy_index(root.side, mv[i])] = (float)cnt[i] / sum;
  return SPB_OK;
}

int32_t spb_chess_advance(spb_chess_engine* e, const uint32_t* slots, const uint32_t* child_ids, uint32_t n, spb_chess_state* out_states) {
  SPB_GUARD(e);
  SPB_ARG(e, child_ids && n <= e->T.G, "bad argument");
  if (n == 0) return SPB_OK;
  if (slots) for (uint32_t i = 0; i < n; ++i) SPB_ARG(e, slots[i] < e->T.G, "slot out of range");
  StageLayout L;
  const size_t o_slots = L.take(slots ? (size_t)n * 4 : 0), o_ids = L.take((size_t)n * 4), o_out = L.take((size_t)n * sizeof(ch::Pos)), o_err = L.take((size_t)n * 4);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  uint32_t* d_slots = slots ? e->d_at<uint32_t>(o_slots) : nullptr;
  uint32_t* d_ids = e->d_at<uint32_t>(o_ids);
  ch::Pos* d_out = e->d_at<ch::Pos>(o_out);
  int32_t* d_err = e->d_at<int32_t>(o_err);
  if (slots) SPB_CUDA(e, cudaMemcpyAsync(d_slots, slots, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(d_ids, child_ids, (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
  ch::k_chess_advance<<<(n + ch::WARPS - 1) / ch::WARPS, ch::THREADS, 0, e->stream>>>(e->T, d_slots, d_ids, n, d_out, d_err);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  std::vector<int32_t> err(n);
  SPB_CUDA(e, cudaMemcpyAsync(err.data(), d_err, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (out_states) SPB_CUDA(e, cudaMemcpyAsync(out_states, d_out, (size_t)n * sizeof(ch::Pos), cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  for (uint32_t i = 0; i < n; ++i)
    if (err[i] != SPB_OK) {
      e->set_error(err[i] == SPB_ERR_STATE ? "game history full (SPB_CHESS_MAX_HISTORY plies)" : "spb_chess_advance: not a child of the root");
      return err[i];
    }
  return SPB_OK;
}

int32_t spb_chess_get_state(spb_chess_engine* e, uint32_t slot, uint32_t node_id, spb_chess_state* out) {
  SPB_GUARD(e);
  SPB_ARG(e, out && slot < e->T.G, "bad argument");
  StageLayout L;
  const size_t o_out = L.take(sizeof(ch::Pos)), o_err = L.take(4);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  ch::Pos* d_out = e->d_at<ch::Pos>(o_out);
  int32_t* d_err = e->d_at<int32_t>(o_err);
  ch::k_chess_get_state<<<1, 1, 0, e->stream>>>(e->T, slot, node_id, d_out, d_err);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  int32_t err = 0;
  SPB_CUDA(e, cudaMemcpyAsync(&err, d_err, 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(out, d_out, sizeof(ch::Pos), cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (err) { e->set_error("spb_chess_get_state: node out of range"); return err; }
  return SPB_OK;
}

int32_t spb_chess_arena_len(spb_chess_engine* e, uint32_t slot, uint32_t* out) {
  SPB_GUARD(e);
  return e->arena_len(slot, out);
}

int32_t spb_chess_node_stats(spb_chess_engine* e, uint32_t slot, uint32_t node_id, uint32_t* visit_count, float* value_sum, float* prior,
                             uint32_t* first_child, uint32_t* n_children, uint16_t* move, uint8_t* status) {
  SPB_GUARD(e);
  SPB_ARG(e, slot < e->T.G, "slot out of range");
  if (int32_t rc = e->ensure_stage(32, 0)) return rc;
  uint32_t* d = e->d_at<uint32_t>(0);
  ch::k_chess_node_stats<<<1, 1, 0, e->stream>>>(e->T, slot, node_id, d);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  uint32_t h[8];
  SPB_CUDA(e, cudaMemcpyAsync(h, d, 32, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  SPB_ARG(e, h[7] == 0, "node out of range");
  if (visit_count) *visit_count = h[0];
  if (value_sum) std::memcpy(value_sum, &h[1], 4);
  if (prior) std::memcpy(prior, &h[2], 4);
  if (first_child) *first_child = h[3];
  if (n_children) *n_children = h[4];
  if (move) *move = (uint16_t)h[5];
  // status in the header's terms: a node that was never reached as a leaf has not been classified yet -> reported Ongoing
  if (status) *status = h[6] == ch::ST_TIED ? SPB_STATUS_TIED : (h[6] == ch::ST_WON ? SPB_STATUS_WON : SPB_STATUS_ONGOING);
  return SPB_OK;
}

int32_t spb_chess_selfplay_step(spb_chess_engine* e, int32_t rule, float temperature, uint64_t seed, const spb_chess_state* restart_roots,
                                const uint64_t* restart_history, uint32_t* n_finished) {
  SPB_GUARD(e);
  SPB_ARG(e, rule == SPB_MOVE_GREEDY_LAST_MAX || rule == SPB_MOVE_TEMPERATURE, "unknown move rule");
  SPB_ARG(e, !(restart_history && !restart_roots), "history without roots");
  const uint32_t G = e->T.G;
  ch::Pos* d_roots = nullptr; unsigned long long* d_hist = nullptr;
  int32_t rc = stage_roots(e, nullptr, restart_roots, restart_history, G, nullptr, &d_roots, &d_hist);
  if (rc) return rc;
  if (!e->P.out) {                                                     // the first step allocates the trajectory buffers
    rc = e->alloc_trajectories(SPB_CHESS_MAX_HISTORY);
    if (rc) return rc;
  }
  SPB_CUDA(e, cudaMemsetAsync(e->P.finished, 0, 4, e->stream));
  ch::k_chess_selfplay_step<<<(G + ch::WARPS - 1) / ch::WARPS, ch::THREADS, 0, e->stream>>>(e->T, e->P, rule, temperature, seed, d_roots, d_hist);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  uint32_t fin = 0;
  SPB_CUDA(e, cudaMemcpyAsync(&fin, e->P.finished, 4, cudaMemcpyDeviceToHost, e->stream));
  rc = e->check_device_errors();                                       // synchronises the stream
  if (n_finished) *n_finished = fin;
  return rc;
}

int32_t spb_chess_drain_trajectories(spb_chess_engine* e, spb_chess_position* buf, size_t capacity, size_t* written, uint64_t* game_ids) {
  SPB_GUARD(e);
  return e->drain_trajectories(buf, capacity, written, game_ids);
}

int32_t spb_chess_drain_trajectories_device(spb_chess_engine* e, spb_chess_position* buf_dev, size_t capacity, size_t* written,
                                            uint64_t* game_ids_dev) {
  SPB_GUARD(e);
  return e->drain_trajectories_device(buf_dev, capacity, written, game_ids_dev);
}

int32_t spb_chess_get_counters(spb_chess_engine* e, spb_counters* out) {
  SPB_GUARD(e);
  return e->get_counters(out, true, [e] { ch::k_chess_nodes_live<<<(e->T.G + 127) / 128, 128, 0, e->stream>>>(e->T, e->d_misc); });
}

int32_t spb_chess_reset_counters(spb_chess_engine* e) {
  SPB_GUARD(e);
  return e->reset_counters();
}

}  // extern "C"
