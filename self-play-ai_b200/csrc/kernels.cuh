// kernels.cuh — the tree / game / self-play kernels of the engine (device code only; included by engine.cu).
//
// Replaces Mcts::search (ref: src/mcts.rs:196-332), Tree::use_subtree (:161-192) and the self-play loop that consumes
// them (ref: src/learner_concurrent.rs:169-242).  One warp owns one tree.  Search pipelines:
//   * fused     (DetEval / uniform evaluators): ONE kernel runs all `num_searches` simulations of every tree; the path
//                 of a simulation lives in registers.
//   * lock-step (SPB_FLAG_LOCKSTEP, K > 1): per simulation step  [evaluator kernel] -> [tree_step kernel], where
//                 tree_step = expand+backup of the evaluated leaf followed by the select of the next simulation.
//   * asynchronous (default for the network): async.cuh — tree warps inside the resident evaluator kernel.
#pragma once
#include "engine.hpp"
#include "root_noise.cuh"

namespace spb {


constexpr int WARPS_PER_BLOCK = 4;
constexpr int THREADS = WARPS_PER_BLOCK * 32;

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------

__global__ void k_reset(Trees T, uint32_t* hist_len, uint8_t* parked, const uint32_t* slots, const PState* roots, uint32_t n) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t g = slots ? slots[i] : i;
  PState root = roots ? roots[i] : ps_make(0, 0, 0, 0, SPB_STATUS_ONGOING);
  T.root_state[g] = root;
  T.buf[g] = 0;
  T.live[g] = 1;
  T.n_nodes[g] = 1;
  parked[g] = 0;
  hist_len[g] = 0;   // a restarted slot starts a new trajectory (Tree::with_root_state has empty histories, mcts.rs:86-89)
  NodeRec r;
  r.N = 0; r.W = 0.0f; r.P = 0.0f;
  r.info = make_info(0, 0, ps_status(root));
  T.rec[0][(size_t)g * T.cap] = r;
  T.par[0][(size_t)g * T.cap] = PAR_NONE | (0xFFu << 24);
  for (uint32_t k = 0; k < T.K; ++k) T.leaf_info[g * T.K + k] = 0;
}

// Fused search: all simulations of one tree inside one warp, evaluator in registers.
template <class G, int EVAL>
__global__ void __launch_bounds__(THREADS) k_search_fused(Trees T, uint32_t num_searches) {
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (g >= T.G || !T.live[g]) return;
  const uint32_t b = T.buf[g];
  NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  uint32_t* par = T.par[b] + (size_t)g * T.cap;
  const PState root = T.root_state[g];
  uint32_t n_nodes = T.n_nodes[g];
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  for (uint32_t s = 0; s < num_searches; ++s) {                       // mcts.rs:214
    WarpPath path;
    uint32_t leaf, linfo;
    int depth;
    PState st;
    descend<G>(rec, root, T.c, root_noise_of(T, g), lane, path, leaf, depth, st, linfo, T.error, n_nodes);
    SPB_ASSERT(T.error, leaf < n_nodes && depth < G::MAX_DEPTH, 6);
    ctr[CTR_SIMS] += 1;
    ctr[CTR_PATHSUM] += (unsigned)depth;
    const uint32_t status = info_status(linfo);
    float v;
    if (status != SPB_STATUS_ONGOING) {                               // mcts.rs:245-247
      v = terminal_value(status);
      ctr[CTR_TERMINAL] += 1;
    } else {                                                          // mcts.rs:268-284
      float probs[G::A];
      if (EVAL == SPB_EVAL_DET) det_eval<G>(st, probs, &v); else uniform_eval<G>(st, probs, &v);
      ctr[CTR_EVALS] += 1;
      uint32_t before = n_nodes;
      if (!expand<G>(rec, par, T.cap, n_nodes, leaf, st, probs, lane)) {
        if (lane == 0) atomicOr(T.error, ERRBIT_POOL);
        break;
      }
      ctr[CTR_CHILDREN] += n_nodes - before;
    }
    backup_regs(rec, path, depth, v, lane);
    __syncwarp();
  }
  if (lane == 0) T.n_nodes[g] = n_nodes;
  flush_counters(T, ctr, lane);
}

// EXTENSION (DESIGN.md §4.6): eta of every live root, one warp per slot, launched at the head of spb_search (and by
// spb_root_noise).  The draw depends on (seed, game id, root ply, number of legal moves) only, so repeated searches of one
// root see the same eta and a new root (advance, self-play step, restart) gets a fresh one.  A terminal root has no children.
template <class G>
__global__ void __launch_bounds__(THREADS) k_root_noise(Trees T, const unsigned long long* game_id, float alpha, unsigned long long seed) {
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (g >= T.G) return;
  if (!T.live[g]) {
    if (lane == 0) T.noise_n[g] = 0;
    return;
  }
  const PState root = T.root_state[g];
  const uint32_t n = ps_status(root) == SPB_STATUS_ONGOING ? (uint32_t)__popc(G::valid_mask(root)) : 0u;
  const unsigned long long key = noise_key(seed, game_id[g], ps_num_actions(root), n);
  warp_dirichlet<1>(key, n, alpha, lane, T.root_noise + (size_t)g * SPB_MAX_ACTIONS, SPB_MAX_ACTIONS);
  if (lane == 0) T.noise_n[g] = n;
}

// Split pipeline.  do_finish: expand + backup the leaf whose evaluation is in eval_out.
// do_select: run the select of the next simulation; terminal leaves are backed up at once,
// the others are appended to the evaluator's work list.
#ifdef SPB_TRACE
__device__ unsigned long long g_pdl_trace[64][8];   // trace build: globaltimer stamps of consecutive kernels, [i][0..2] tree step entry / after wait / exit
__device__ unsigned int g_pdl_idx = 0;
__device__ unsigned long long g_warp_trace[8192][6];   // per tree of the latest tree step: entry, after wait, after finish, after descend, after append, exit
extern "C" int spb_debug_warp_trace(unsigned long long* out, int n) { return (int)cudaMemcpyFromSymbol(out, g_warp_trace, sizeof(unsigned long long) * 6 * (size_t)n); }
#define WTRACE(i) do { if (lane == 0 && g < 8192 && do_select && do_finish) g_warp_trace[g][i] = gtimer(); } while (0)
extern "C" int spb_debug_pdl_trace(unsigned long long* out) {
  unsigned int z = 0;
  int rc = (int)cudaMemcpyFromSymbol(out, g_pdl_trace, sizeof(unsigned long long) * 64 * 8);
  rc |= (int)cudaMemcpyToSymbol(g_pdl_idx, &z, sizeof z);
  return rc;
}
__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#else
#define WTRACE(i) ((void)0)
#endif

template <class G>
__global__ void __launch_bounds__(THREADS) k_tree_step(Trees T, int do_finish, int do_select, uint32_t parity) {
  // Programmatic dependent launch (no-ops for a plain launch): the evaluator that follows may start its set-up while
  // this grid runs, and this grid may have been started before the evaluator in front of it finished.
#ifdef SPB_TRACE
  const unsigned long long tr0 = gtimer();
#endif
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
#ifdef SPB_TRACE
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const unsigned int i = g_pdl_idx++ & 63u;
    g_pdl_trace[i][0] = tr0;
    g_pdl_trace[i][1] = gtimer();
  }
#endif
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (blockIdx.x == 0 && threadIdx.x == 0) T.eval_count[(parity + 1) & 1] = 0;   // for the NEXT step's select
  if (g >= T.G) return;
  // Everything that is addressed by the tree index alone is requested in ONE round trip (the step is bound by the
  // latency of dependent global loads, not by bandwidth): liveness, live arena, the pending leaf, its state, the
  // evaluator's answer, the arena length and the stored path (lane d holds path node d and d + 32).
  const uint32_t slot = g;   // K == 1
  uint32_t* pathm = T.path + (size_t)slot * G::MAX_DEPTH;
  const uint8_t live = T.live[g];
  const uint32_t b = T.buf[g];
  const uint32_t li = T.leaf_info[slot];
  const PState st = T.leaf_state[slot];
  const float* eo = T.eval_out + (size_t)slot * G::EVAL_STRIDE;
  float probs[G::A];
#pragma unroll
  for (int a = 0; a < G::A; ++a) probs[a] = eo[a];
  const float v = eo[G::A];
  uint32_t n_nodes = T.n_nodes[g];
  const uint32_t pn0 = (lane < G::MAX_DEPTH) ? pathm[lane] : 0u;   // tic-tac-toe paths are 12 words: lanes beyond must not read the next slot's
  const uint32_t pn1 = (lane + 32 < G::MAX_DEPTH) ? pathm[lane + 32] : 0u;
  if (!live) return;
#ifdef SPB_TRACE
  if (lane == 0 && g < 8192 && do_select && do_finish) g_warp_trace[g][0] = tr0;
#endif
  WTRACE(1);
  NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  uint32_t* par = T.par[b] + (size_t)g * T.cap;
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  bool ok = true;

  if (do_finish && (li & LEAF_PENDING)) {
    const int depth = (int)(li & 0xFFu);
    const uint32_t leaf = __shfl_sync(0xffffffffu, depth < 32 ? pn0 : pn1, depth & 31);
    SPB_ASSERT(T.error, depth < G::MAX_DEPTH && (lane > depth || pn0 < n_nodes) && (lane + 32 > depth || pn1 < n_nodes), 8);
    // second round trip: the path nodes' statistics (backup, mcts.rs:145-159), requested before the expand's stores
    uint2 nw0 = make_uint2(0, 0), nw1 = make_uint2(0, 0);
    if (lane <= depth) nw0 = *reinterpret_cast<const uint2*>(&rec[pn0]);
    if (lane + 32 <= depth) nw1 = *reinterpret_cast<const uint2*>(&rec[pn1]);
    const uint32_t before = n_nodes;
    if (!expand<G>(rec, par, T.cap, n_nodes, leaf, st, probs, lane)) {
      if (lane == 0) atomicOr(T.error, ERRBIT_POOL);
      ok = false;
    } else {
      ctr[CTR_CHILDREN] += n_nodes - before;
      if (lane == 0) T.n_nodes[g] = n_nodes;
      if (lane <= depth) {                                        // same arithmetic as backup_mem: N += 1, W = W + (+-v)
        nw0.x += 1u;
        nw0.y = __float_as_uint(__fadd_rn(__uint_as_float(nw0.y), ((depth - lane) & 1) ? -v : v));
        *reinterpret_cast<uint2*>(&rec[pn0]) = nw0;
      }
      if (lane + 32 <= depth) {
        nw1.x += 1u;
        nw1.y = __float_as_uint(__fadd_rn(__uint_as_float(nw1.y), ((depth - lane - 32) & 1) ? -v : v));
        *reinterpret_cast<uint2*>(&rec[pn1]) = nw1;
      }
    }
    if (lane == 0) T.leaf_info[slot] = 0;
    __syncwarp();
  }

  WTRACE(2);
  if (do_select && ok) {
    WarpPath path;
    uint32_t leaf, linfo;
    int depth;
    PState st;
    descend<G>(rec, T.root_state[g], T.c, root_noise_of(T, g), lane, path, leaf, depth, st, linfo, T.error, n_nodes);
    SPB_ASSERT(T.error, leaf < n_nodes && depth < G::MAX_DEPTH, 7);
    WTRACE(3);
    ctr[CTR_SIMS] += 1;
    ctr[CTR_PATHSUM] += (unsigned)depth;
    const uint32_t status = info_status(linfo);
    if (status != SPB_STATUS_ONGOING) {
      ctr[CTR_TERMINAL] += 1;
      backup_regs(rec, path, depth, terminal_value(status), lane);
    } else {
      ctr[CTR_EVALS] += 1;
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        int d = lane + 32 * s;
        if (d <= depth) pathm[d] = path.node[s];
      }
      if (lane == 0) {
        T.leaf_state[slot] = st;
        T.leaf_info[slot] = (uint32_t)depth | LEAF_PENDING;
        uint32_t pos = atomicAdd(&T.eval_count[parity & 1], 1u);
        T.eval_list[pos] = slot;
      }
    }
  }
  WTRACE(4);
  flush_counters(T, ctr, lane);
  WTRACE(5);
}

// ---- EXTENSION (not in the reference): K in-flight leaves per tree per step with virtual loss ------------
// BASELINE.json config 4 / SURVEY.md §8(f)-3; the reference runs one leaf per tree per step (mcts.rs:236-252)
// and K = 1 never comes here.  The warp that owns the tree runs its K descents one after the other, so no
// atomics are needed and the result is deterministic.  Definition (identical in oracle/oracle.cc search_vl):
//   select k: PUCT descent on the current statistics.  Terminal leaf: real backup at once.  Otherwise every
//   path node takes a virtual loss (N += 1, W += 1.0) and the leaf is queued — as a duplicate if the same leaf
//   is already queued in this step.  Finish (after the evaluator): entries in selection order; a first
//   occurrence expands; every entry rewrites each path node as W = (W - 1.0) + sign*v.
// leaf_info[slot]: depth[0,8) | LEAF_PENDING | LEAF_DUP | source entry[16,24)
constexpr uint32_t LEAF_DUP = 1u << 9;

__device__ __forceinline__ void backup_virtual(NodeRec* rec, const uint32_t* path, int depth, float v, int lane) {
  for (int d = lane; d <= depth; d += 32) {
    const uint32_t node = path[d];
    const float sv = ((depth - d) & 1) ? -v : v;
    float* w = &rec[node].W;
    *w = __fadd_rn(__fsub_rn(*w, 1.0f), sv);
  }
}

template <class G>
__global__ void __launch_bounds__(THREADS) k_tree_step_multi(Trees T, int do_finish, uint32_t k_select, uint32_t parity) {
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (blockIdx.x == 0 && threadIdx.x == 0) T.eval_count[(parity + 1) & 1] = 0;
  if (g >= T.G || !T.live[g]) return;
  const uint32_t b = T.buf[g];
  NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  uint32_t* par = T.par[b] + (size_t)g * T.cap;
  const uint32_t K = T.K;
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  bool ok = true;

  if (do_finish) {
    uint32_t n_nodes = T.n_nodes[g];
    for (uint32_t k = 0; k < K && ok; ++k) {
      const uint32_t slot = g * K + k;
      const uint32_t li = T.leaf_info[slot];
      if (!(li & (LEAF_PENDING | LEAF_DUP))) continue;
      const int depth = (int)(li & 0xFFu);
      const uint32_t src = (li & LEAF_DUP) ? g * K + ((li >> 16) & 0xFFu) : slot;
      const uint32_t* pathm = T.path + (size_t)src * G::MAX_DEPTH;
      const float* eo = T.eval_out + (size_t)src * G::EVAL_STRIDE;
      if (li & LEAF_PENDING) {
        float probs[G::A];
#pragma unroll
        for (int a = 0; a < G::A; ++a) probs[a] = eo[a];
        const uint32_t before = n_nodes;
        if (!expand<G>(rec, par, T.cap, n_nodes, pathm[depth], T.leaf_state[slot], probs, lane)) {
          if (lane == 0) atomicOr(T.error, ERRBIT_POOL);
          ok = false;
          break;
        }
        ctr[CTR_CHILDREN] += n_nodes - before;
      }
      __syncwarp();
      backup_virtual(rec, pathm, depth, eo[G::A], lane);
      if (lane == 0) T.leaf_info[slot] = 0;
      __syncwarp();
    }
    if (lane == 0) T.n_nodes[g] = n_nodes;
  }

  if (ok) {
    uint32_t my_leaf = 0xFFFFFFFFu;                    // lane j: leaf queued by entry j of this step (first occurrences only)
    const PState root = T.root_state[g];
    for (uint32_t k = 0; k < k_select; ++k) {
      const uint32_t slot = g * K + k;
      WarpPath path;
      uint32_t leaf, linfo;
      int depth;
      PState st;
      descend<G>(rec, root, T.c, root_noise_of(T, g), lane, path, leaf, depth, st, linfo, T.error);
      ctr[CTR_SIMS] += 1;
      ctr[CTR_PATHSUM] += (unsigned)depth;
      const uint32_t status = info_status(linfo);
      if (status != SPB_STATUS_ONGOING) {
        ctr[CTR_TERMINAL] += 1;
        backup_regs(rec, path, depth, terminal_value(status), lane);
      } else {
        const unsigned dupmask = __ballot_sync(0xffffffffu, my_leaf == leaf);
        // virtual loss on the whole path (lane d <-> depth d)
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const int d = lane + 32 * s;
          if (d <= depth) {
            uint2 nw;
            nw.x = path.N[s] + 1u;
            nw.y = __float_as_uint(__fadd_rn(path.W[s], 1.0f));
            *reinterpret_cast<uint2*>(&rec[path.node[s]]) = nw;
          }
        }
        if (dupmask) {
          if (lane == 0) T.leaf_info[slot] = (uint32_t)depth | LEAF_DUP | ((uint32_t)(__ffs((int)dupmask) - 1) << 16);
        } else {
          ctr[CTR_EVALS] += 1;
          uint32_t* pathm = T.path + (size_t)slot * G::MAX_DEPTH;
#pragma unroll
          for (int s = 0; s < 2; ++s) {
            const int d = lane + 32 * s;
            if (d <= depth) pathm[d] = path.node[s];
          }
          if (lane == (int)k) my_leaf = leaf;
          if (lane == 0) {
            T.leaf_state[slot] = st;
            T.leaf_info[slot] = (uint32_t)depth | LEAF_PENDING;
            const uint32_t pos = atomicAdd(&T.eval_count[parity & 1], 1u);
            T.eval_list[pos] = slot;
          }
        }
      }
      __syncwarp();
    }
  }
  flush_counters(T, ctr, lane);
}

// Evaluator stand-ins for the split pipeline (parity harness): DetEval / uniform over the work list.
template <class G, int EVAL>
__global__ void k_eval_builtin(const PState* states, const uint32_t* list, const uint32_t* count, float* out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= *count) return;
  uint32_t slot = list[i];
  float probs[G::A], v;
  if (EVAL == SPB_EVAL_DET) det_eval<G>(states[slot], probs, &v); else uniform_eval<G>(states[slot], probs, &v);
  float* o = out + (size_t)slot * G::EVAL_STRIDE;
#pragma unroll
  for (int a = 0; a < G::A; ++a) o[a] = probs[a];
  o[G::A] = v;
}

// ---- asynchronous pipeline (async.cuh) --------------------------------------------------------------------
// Start of a search: every live tree gets its simulation budget and a ticket of the ready ring.
__global__ void k_async_init(Trees T, AsyncCtl C, uint32_t num_searches) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= T.G || !T.live[g]) return;
  C.sims_left[g] = num_searches;
  atomicAdd(C.n_active, 1u);
  const uint32_t t = atomicAdd(C.ready.tail, 1u);
  C.ready.slots[t & C.ready.mask] = ring_entry(t, g);
}

// The pipeline with the built-in evaluators (parity harness: SPB_FLAG_FORCE_SPLIT): the same rings and tree warps as the
// network pipeline, evaluator CTAs replaced by evaluator warps.  Warps 0,1 evaluate, warps 2,3 own trees.
template <class G, int EVAL>
__global__ void __launch_bounds__(THREADS) k_async_builtin(Trees T, AsyncCtl C) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (warp < 2) builtin_eval_worker<G, EVAL>(T, C, gridDim.x * 2u, lane);
  else tree_worker<G>(T, C, lane);
}

// Replays the moves from the root to `node` (walks the parent links up, then down again).
template <class G>
__device__ PState node_state(const Trees& T, uint32_t g, uint32_t node) {
  const uint32_t b = T.buf[g];
  const NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  const uint32_t* par = T.par[b] + (size_t)g * T.cap;
  uint8_t acts[G::MAX_DEPTH];
  int n = 0;
  uint32_t cur = node;
  while (true) {
    uint32_t p = par[cur];
    if ((p & PAR_NONE) == PAR_NONE || n >= G::MAX_DEPTH) break;
    acts[n++] = (uint8_t)(p >> 24);
    cur = p & PAR_NONE;
  }
  PState st = T.root_state[g];
  for (int i = n - 1; i >= 0; --i) st = G::place(st, acts[i], i == 0 ? info_status(rec[node].info) : (uint32_t)SPB_STATUS_ONGOING);
  return st;
}

// use_subtree, mcts.rs:161-192: breadth-first copy of the subtree under `new_root` into the other
// arena.  New ids are BFS order, children stay contiguous and in action order, statistics are kept.
// A window of 32 already-copied nodes is processed per iteration; a warp scan of the child counts
// assigns the children's new ids exactly as the sequential queue would.
template <class G>
__device__ void reroot(const Trees& T, uint32_t g, uint32_t new_root, int lane) {
  const uint32_t b = T.buf[g];
  const NodeRec* orec = T.rec[b] + (size_t)g * T.cap;
  const uint32_t* opar = T.par[b] + (size_t)g * T.cap;
  NodeRec* nrec = T.rec[b ^ 1] + (size_t)g * T.cap;
  uint32_t* npar = T.par[b ^ 1] + (size_t)g * T.cap;
  PState new_state = node_state<G>(T, g, new_root);
  if (lane == 0) {
    nrec[0] = orec[new_root];                                  // info still holds the OLD first_child
    npar[0] = PAR_NONE | (opar[new_root] & 0xFF000000u);       // parent_id = None, action_taken kept (:166-167)
  }
  __syncwarp();
  uint32_t next = 1;
  for (uint32_t lo = 0; lo < next;) {
    const uint32_t hi = min(next, lo + 32u);                   // nodes [lo, hi) are already in the new arena
    const uint32_t i = lo + lane;
    const bool active = i < hi;
    uint32_t info = active ? nrec[i].info : 0u;
    const uint32_t nc = info_nc(info), ofc = info_fc(info);
    uint32_t incl = nc;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      uint32_t t = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += t;
    }
    const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
    const uint32_t nfc = next + incl - nc;
    SPB_ASSERT(T.error, !active || (nfc + nc <= T.cap && ofc + nc <= T.cap), 9);
    if (active) {
      for (uint32_t j = 0; j < nc; ++j) {
        nrec[nfc + j] = orec[ofc + j];
        npar[nfc + j] = i | (opar[ofc + j] & 0xFF000000u);
      }
      nrec[i].info = make_info(nc ? nfc : 0u, nc, info_status(info));
    }
    next += total;
    lo = hi;
    __syncwarp();
  }
  if (lane == 0) {
    T.n_nodes[g] = next;
    T.buf[g] = (uint8_t)(b ^ 1);
    T.root_state[g] = new_state;
    for (uint32_t k = 0; k < T.K; ++k) T.leaf_info[g * T.K + k] = 0;   // node_id_to_expand = None (learner_concurrent.rs:233)
  }
}

template <class G>
__global__ void __launch_bounds__(THREADS) k_advance(Trees T, const uint32_t* slots, const uint32_t* node_ids, uint32_t n,
                                                     PState* out_states) {
  const int lane = threadIdx.x & 31;
  const uint32_t i = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (i >= n) return;
  const uint32_t g = slots ? slots[i] : i;
  reroot<G>(T, g, node_ids[i], lane);
  __syncwarp();
  if (lane == 0 && out_states) out_states[i] = T.root_state[g];
}

template <class G>
__global__ void k_get_state(Trees T, uint32_t g, uint32_t node, PState* out) { *out = node_state<G>(T, g, node); }

// Root children of every slot, in child order (mcts.rs:310-331).
__global__ void k_root_children(Trees T, uint8_t* actions, uint32_t* counts, uint32_t* ids, uint32_t* ncs) {
  uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= T.G) return;
  const uint32_t b = T.buf[g];
  const NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  const uint32_t* par = T.par[b] + (size_t)g * T.cap;
  uint32_t info = rec[0].info;
  uint32_t nc = T.live[g] ? info_nc(info) : 0u, fc = info_fc(info);
  ncs[g] = nc;
  for (uint32_t j = 0; j < SPB_MAX_ACTIONS; ++j) {
    bool v = j < nc;
    actions[g * SPB_MAX_ACTIONS + j] = v ? (uint8_t)(par[fc + j] >> 24) : (uint8_t)0xFF;
    counts[g * SPB_MAX_ACTIONS + j] = v ? rec[fc + j].N : 0u;
    ids[g * SPB_MAX_ACTIONS + j] = v ? fc + j : 0u;
  }
}

__global__ void k_node_stats(Trees T, uint32_t g, uint32_t node, NodeRec* out) {
  *out = T.rec[T.buf[g]][(size_t)g * T.cap + node];
}

__global__ void k_nodes_live(Trees T, unsigned long long* out) {
  uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < T.G && T.live[g]) atomicAdd(out, (unsigned long long)T.n_nodes[g]);
}

__global__ void k_max_nodes(Trees T, unsigned long long* out) {
  uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g < T.G && T.live[g]) atomicMax(out, (unsigned long long)T.n_nodes[g]);
}

// ---- State trait, batched (ref: game/mod.rs:21-33) ------------------------------------------------
template <class G>
__global__ void k_game_next(const PState* in, const uint8_t* actions, uint32_t n, PState* out, int32_t* err) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  PState o = in[i];
  bool ok = G::next_state(in[i], actions[i], &o);
  out[i] = o;
  err[i] = ok ? SPB_OK : SPB_ERR_ILLEGAL;
}
template <class G>
__global__ void k_game_valid(const PState* in, uint32_t n, uint32_t* masks) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) masks[i] = G::valid_mask(in[i]);
}
template <class G>
__global__ void k_game_encode(const PState* in, uint32_t n, float* out) {
  constexpr int E = 3 * G::ROWS * G::COLS;
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)n * E) return;
  uint32_t i = (uint32_t)(t / E);
  int r = (int)(t % E);
  int plane = r / (G::ROWS * G::COLS), row = (r / G::COLS) % G::ROWS, col = r % G::COLS;
  out[t] = G::encode_cell(in[i], plane, row, col);
}

// Masks + renormalises evaluator output for spb_predict (model/mod.rs:86-93).
template <class G>
__global__ void k_mask_policies(const PState* states, uint32_t n, const float* eval_out, float* policies, float* values) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float probs[G::A], pri[G::A];
#pragma unroll
  for (int a = 0; a < G::A; ++a) probs[a] = eval_out[(size_t)i * G::EVAL_STRIDE + a];
  mask_renorm<G>(G::valid_mask(states[i]), probs, pri);
#pragma unroll
  for (int a = 0; a < G::A; ++a) policies[(size_t)i * G::A + a] = pri[a];
  values[i] = eval_out[(size_t)i * G::EVAL_STRIDE + G::A];
}

// ---- self-play ply (ref: learner_concurrent.rs:179-238) -------------------------------------------

// Emits the finished game of slot g (learner_concurrent.rs:200-230) and restarts or retires the slot.
__device__ __forceinline__ void emit_and_finish(const Trees& T, const SelfPlay& P, uint32_t g, uint32_t plies, uint32_t cstatus,
                                                uint32_t term_player, unsigned long long base, const PState* restart_roots, int lane) {
  const float value = terminal_value(cstatus);                     // from the terminal state's side to move
  SPB_ASSERT(T.error, base + plies <= P.out_cap && plies <= P.max_ply, 10);
  for (uint32_t i = lane; i < plies; i += 32) {
    spb_position p = P.hist[(size_t)g * P.max_ply + i];
    float v = (p.current_player == term_player) ? value : -value;   // :214-226
    p.outcome = (int8_t)v;
    P.out[base + i] = p;
    P.out_game[base + i] = P.game_id[g];
  }
  __syncwarp();
  if (lane == 0) {
    finish_trajectory(P, g);
    if (restart_roots) {                                           // Tree::with_root_state for the next game
      PState nr = restart_roots[g];
      T.root_state[g] = nr;
      T.buf[g] = 0;
      T.n_nodes[g] = 1;
      T.live[g] = 1;
      NodeRec r; r.N = 0; r.W = 0.0f; r.P = 0.0f; r.info = make_info(0, 0, ps_status(nr));
      T.rec[0][(size_t)g * T.cap] = r;
      T.par[0][(size_t)g * T.cap] = PAR_NONE | (0xFFu << 24);
      for (uint32_t k = 0; k < T.K; ++k) T.leaf_info[g * T.K + k] = 0;
    } else {
      T.live[g] = 0;                                               // trees_vec.remove(i), :230
    }
  }
}

template <class G>
__global__ void __launch_bounds__(THREADS) k_selfplay_step(Trees T, SelfPlay P, int rule, float temperature,
                                                           unsigned long long seed, const PState* restart_roots) {
  const int lane = threadIdx.x & 31;
  const uint32_t g = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  if (g >= T.G) return;
  const uint32_t pk = P.parked[g];
  if (pk) {
    // A game that ended in an earlier call while the output buffer was full: the slot has been idle since; emit now.
    const uint32_t plies = P.hist_len[g];
    unsigned long long base;
    if (reserve_output(P, plies, lane, &base)) emit_and_finish(T, P, g, plies, (pk >> 1) & 3u, (pk >> 3) & 1u, base, restart_roots, lane);
    else if (lane == 0) atomicOr(T.error, ERRBIT_TRAJ_FULL);
    return;
  }
  if (!T.live[g]) return;
  const uint32_t b = T.buf[g];
  NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  const uint32_t* par = T.par[b] + (size_t)g * T.cap;
  const uint32_t info = rec[0].info;
  const uint32_t nc = info_nc(info), fc = info_fc(info);
  if (nc == 0) return;                                           // nothing searched / terminal root
  const PState root = T.root_state[g];
  uint32_t cnt = 0, act = 0, cinfo = 0;
  if (lane < (int)nc) { cnt = rec[fc + lane].N; cinfo = rec[fc + lane].info; act = par[fc + lane] >> 24; }
  int chosen;
  if (rule == SPB_MOVE_TEMPERATURE) {
    // learner_concurrent.rs:189-194: WeightedIndex over count^temperature.  Counter-based RNG (the
    // reference uses the unseedable thread_rng, so there is no stream to match).
    float w = lane < (int)nc ? powf((float)cnt, temperature) : 0.0f;
    float incl = w;
#pragma unroll
    for (int off = 1; off < 16; off <<= 1) {
      float t = __shfl_up_sync(0xffffffffu, incl, off);
      if (lane >= off) incl += t;
    }
    float total = __shfl_sync(0xffffffffu, incl, 15);
    unsigned long long h = splitmix64(seed ^ splitmix64(P.game_id[g] * 64ull + P.hist_len[g]));
    float u = (float)(h >> 40) * (1.0f / 16777216.0f) * total;
    unsigned ball = __ballot_sync(0xffffffffu, lane < (int)nc && u < incl && w > 0.0f);
    chosen = ball ? __ffs((int)ball) - 1 : (int)nc - 1;
  } else {
    // main.rs:108-112: max_by(total_cmp) over visit counts -> the LAST maximal child.
    chosen = warp_argmax_last<G::A>(lane < (int)nc ? (float)cnt : -INFINITY, lane < (int)nc ? lane : -1);
    chosen = __shfl_sync(0xffffffffu, chosen, 0);
  }
  // learner_concurrent.rs:197-198: push root state + visit-count policy.
  const uint32_t ply = P.hist_len[g];
  if (ply < P.max_ply) {
    spb_position* h = &P.hist[(size_t)g * P.max_ply + ply];
    if (lane == 0) {
      h->stones[0] = ps_x(root); h->stones[1] = ps_o(root);
      h->current_player = (uint8_t)ps_player(root);
      h->ply = (uint8_t)ply; h->outcome = 0; h->reserved = 0;
      for (int a = 0; a < SPB_MAX_ACTIONS; ++a) h->visit_counts[a] = 0;
    }
    __syncwarp();
    if (lane < (int)nc && act < SPB_MAX_ACTIONS) h->visit_counts[act] = cnt;
    __syncwarp();
  }
  const uint32_t cstatus = info_status(__shfl_sync(0xffffffffu, cinfo, chosen));
  const uint32_t plies = min(ply + 1, P.max_ply);
  if (cstatus != SPB_STATUS_ONGOING) {
    // learner_concurrent.rs:200-230: the game is over.  The trajectory is emitted only when all of it fits the output
    // buffer; otherwise the slot is parked (idle, history kept) and the call reports SPB_ERR_STATE: the caller drains
    // and the next spb_selfplay_step emits the parked games, so no game and no record is ever lost or half-written.
    const uint32_t term_player = ps_player(root) ^ 1u;
    unsigned long long base;
    if (reserve_output(P, plies, lane, &base)) {
      emit_and_finish(T, P, g, plies, cstatus, term_player, base, restart_roots, lane);
    } else if (lane == 0) {
      P.hist_len[g] = plies;
      P.parked[g] = (uint8_t)(1u | (cstatus << 1) | (term_player << 3));
      T.live[g] = 0;
      atomicOr(T.error, ERRBIT_TRAJ_FULL);
    }
  } else {
    if (lane == 0) P.hist_len[g] = plies;
    reroot<G>(T, g, fc + (uint32_t)chosen, lane);                // :233-234
  }
}

}  // namespace spb
