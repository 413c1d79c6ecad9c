// async.cuh — the asynchronous search pipeline (default for the network evaluator).
//
// Mcts::search (ref: src/mcts.rs:214-286) advances every tree by one simulation per iteration and evaluates the
// non-terminal leaves of that iteration as one batch (mcts.rs:268).  The trees never interact: tree i's k-th simulation
// depends only on tree i's own first k-1 simulations and on an evaluator that is a pure function of one position
// (BatchNorm in eval mode, model/mod.rs:62).  So the lock-step across trees is a property of the reference's loop, not
// of its results, and this pipeline drops it: every tree runs its own  select -> evaluate -> expand+backup  cycle as
// fast as the machine allows, and the results are bit-identical to the lock-step pipeline (tests: async == lock-step
// for the network, async == oracle node for node under DetEval / uniform).
//
// Two multi-producer / multi-consumer rings in global memory carry slot ids:
//   ready : trees whose evaluation has arrived (or that have not started)   evaluator -> tree warps
//   leaf  : trees whose selected leaf awaits the evaluator                   tree warps -> evaluator
// A tree is in exactly one place at any time (a ring, a tree warp, an evaluator batch), so a ring of >= G entries never
// overflows.  Tree warps take a ticket and wait for it (more waiters than entries is the idle state); evaluator CTAs
// claim up to a batch of PUBLISHED-or-reserved entries with a CAS so that a batch never waits for leaves that do not
// exist.  Entries are 64-bit (ticket + 1) << 32 | slot, published with st.release / read with ld.acquire at gpu scope;
// everything a tree's next owner reads is read at L2 (ld.cg), since the previous owner was another SM.
#pragma once
#include "tree.cuh"

namespace spb {

struct Ring {
  unsigned long long* slots;   // [mask + 1], zeroed before every search
  uint32_t* head;              // next ticket to consume   (own 128-byte line)
  uint32_t* tail;              // next ticket to produce   (own 128-byte line)
  uint32_t mask;
};

struct AsyncCtl {
  Ring leaf, ready;
  uint32_t* sims_left;         // [G] simulations a tree has still to START in this search
  uint32_t* n_active;          // trees taking part in this search (constant while the search kernels run)
  uint32_t* done_count;        // trees that have completed all their simulations
  uint32_t* abort;             // watchdog: set when the pipeline made no progress for stall_ns (a bug, never expected)
  unsigned long long* stats;   // [ASTAT_COUNT] pipeline statistics of the search (summed over CTAs / warps at kernel exit)
  unsigned long long stall_ns;
  EvalCache cache;             // per-tree evaluation cache (tree.cuh); cache.key == nullptr: none
  uint32_t epoch;              // this search's epoch: cache entries of other epochs are empty slots
};
enum AsyncStat { ASTAT_BATCHES = 0, ASTAT_BOARDS, ASTAT_CLAIM_WAIT_NS, ASTAT_TREE_BUSY_NS, ASTAT_TREE_PHASES, ASTAT_TREE_WARPS,
                 ASTAT_EVAL_CTAS, ASTAT_CLAIM_EMPTY, ASTAT_TICKET_WAIT_NS, ASTAT_AVAIL_SUM, ASTAT_READY_BACKLOG, ASTAT_READY_STARVED, ASTAT_COUNT };

constexpr uint32_t RING_NONE = 0xFFFFFFFFu;

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// Polling uses relaxed loads (served by L2, no side effects on the SM); the acquire is a fence executed once, after the
// awaited value has been seen.  An acquire load in the polling loop costs an L1 invalidation per poll, which slowed the
// evaluator sharing the SM by ~10 % (profiles/r02_async_trace.txt).
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acquire_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long gtime_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ unsigned long long ring_entry(uint32_t ticket, uint32_t value) {
  return ((unsigned long long)(ticket + 1u) << 32) | value;
}

// Spin-loop helper: back-off, end-of-search test and the stall watchdog.  `progress` = leaf.tail + ready.tail moves with
// every hand-off anywhere in the pipeline; if it stands still for stall_ns the search is abandoned (SPB_ERR_STATE).
struct Spin {
  unsigned long long t_last;
  uint32_t seen, n_active, iter;
  unsigned long long backlog = 0, starved = 0;
  __device__ __forceinline__ void init(const AsyncCtl& c, uint32_t n_act) {
    t_last = gtime_ns();
    seen = 0xFFFFFFFFu;
    n_active = n_act;
    iter = 0;
  }
  // true = stop waiting: every tree is done, or the pipeline was aborted
  __device__ __forceinline__ bool over(const AsyncCtl& c) {
    return ld_relaxed_u32(c.done_count) >= n_active || ld_relaxed_u32(c.abort) != 0u;
  }
  // one unsuccessful poll; returns true when the caller must give up
  __device__ __forceinline__ bool idle(const AsyncCtl& c) {
    ++iter;
    // Every poll is a global load through the SM's L1TEX data pipe, which the evaluator's shared-memory traffic saturates:
    // idle warps poll rarely (measured: 87 polls per microsecond per SM with short sleeps cost 7 % of the pipe).
#ifdef SPB_POLL_FAST
    __nanosleep((iter < 8u) ? 32u : 200u);
    if ((iter & 15u) != 0u) return false;
#else
    __nanosleep((iter < 4u) ? 100u : 1000u);
    if ((iter & 7u) != 0u) return false;
#endif
    if (over(c)) return true;
    if ((iter & 255u) == 0u) {
      const uint32_t p = ld_relaxed_u32(c.leaf.tail) + ld_relaxed_u32(c.ready.tail);
      const unsigned long long now = gtime_ns();
      if (p != seen) { seen = p; t_last = now; }
      else if (now - t_last > c.stall_ns) { atomicExch(c.abort, 1u); return true; }
    }
    return false;
  }
  __device__ __forceinline__ void progressed() { iter = 0; }
};

__device__ __forceinline__ void ring_push(const Ring& r, uint32_t value) {   // one lane; its earlier writes are released
  const uint32_t t = atomicAdd(r.tail, 1u);
  st_release_u64(&r.slots[t & r.mask], ring_entry(t, value));
}

// Warp-aggregated push: lanes [0, n) each publish `value` (after their own writes; callers fence other lanes' writes).
__device__ __forceinline__ void ring_push_warp(const Ring& r, uint32_t n, uint32_t value, int lane) {
  uint32_t base = 0;
  if (lane == 0) base = atomicAdd(r.tail, n);
  base = __shfl_sync(0xffffffffu, base, 0);
  if ((uint32_t)lane < n) st_release_u64(&r.slots[(base + (uint32_t)lane) & r.mask], ring_entry(base + (uint32_t)lane, value));
}

// Tree warps: take the next ticket of the ready ring and wait for it.  One lane.  RING_NONE = the search is over.
__device__ __forceinline__ uint32_t ready_pop_wait(const AsyncCtl& c, Spin& sp) {
  const uint32_t t = atomicAdd(c.ready.head, 1u);
  const unsigned long long* p = &c.ready.slots[t & c.ready.mask];
  sp.progressed();
  {
    const int32_t backlog = (int32_t)(ld_relaxed_u32(c.ready.tail) - t);   // > 0: entries were waiting for a tree warp
    if (backlog > 0) { sp.backlog += (unsigned)backlog; } else { sp.starved += 1; }
  }
  for (;;) {
    const unsigned long long v = ld_relaxed_u64(p);
    if ((uint32_t)(v >> 32) == t + 1u) { fence_acquire_gpu(); return (uint32_t)v; }
    if (sp.idle(c)) return RING_NONE;
  }
}

// Evaluator side: a batch is a run of consecutive leaf tickets.  Tickets are taken with a fetch-add (a compare-and-swap
// against the published tail collapses when 148 CTAs claim from one counter: measured 44 us per claim), so a claim may
// run ahead of the producers, like a tree warp's ticket.  A batch never waits for leaves that may not exist: once the
// first ticket has been filled the others get `grace_ns` to arrive, the filled prefix forms the batch and the unfilled
// tickets are carried into this consumer's next batch (nobody else can take them).  The batch size follows the number
// of trees still searching: with many trees every CTA takes full batches (throughput), with few the leaves are spread
// over the CTAs (latency).  Warp-collective; lane i < the returned count receives its slot.  0 = the search is over.
struct LeafClaimer {
  uint32_t tk = 0;      // lane i < n_tk holds ticket tk (tickets ascending with the lane)
  uint32_t n_tk = 0;    // warp-uniform
};
__device__ __forceinline__ uint32_t claim_batch(const AsyncCtl& c, LeafClaimer& lc, uint32_t n_consumers, uint32_t kmax,
                                                uint32_t grace_ns, Spin& sp, int lane, uint32_t* slot_out) {
  const uint32_t alive = sp.n_active - min(sp.n_active, ld_relaxed_u32(c.done_count));
  const uint32_t k = max(1u, min(kmax, (alive + n_consumers - 1u) / n_consumers));
  if (lc.n_tk < k) {
    const uint32_t need = k - lc.n_tk;
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(c.leaf.head, need);
    base = __shfl_sync(0xffffffffu, base, 0);
    if ((uint32_t)lane >= lc.n_tk && (uint32_t)lane < k) lc.tk = base + ((uint32_t)lane - lc.n_tk);
    lc.n_tk = k;
  }
  uint32_t val = RING_NONE;
  if (lane == 0) {                                                  // the oldest ticket: wait for it (or for the end of the search)
    const unsigned long long* p = &c.leaf.slots[lc.tk & c.leaf.mask];
    sp.progressed();
    for (;;) {
      const unsigned long long v = ld_relaxed_u64(p);
      if ((uint32_t)(v >> 32) == lc.tk + 1u) { val = (uint32_t)v; break; }
      if (sp.idle(c)) break;
    }
  }
  if (__shfl_sync(0xffffffffu, val, 0) == RING_NONE) return 0u;
  if (lane > 0 && (uint32_t)lane < lc.n_tk) {
    const unsigned long long* p = &c.leaf.slots[lc.tk & c.leaf.mask];
    const unsigned long long t0 = gtime_ns();
    for (;;) {
      const unsigned long long v = ld_relaxed_u64(p);
      if ((uint32_t)(v >> 32) == lc.tk + 1u) { val = (uint32_t)v; break; }
      if (gtime_ns() - t0 > grace_ns) break;
    }
  }
  fence_acquire_gpu();                                              // the leaves' states are read after this (every lane reads its own)
  const uint32_t filled = __ballot_sync(0xffffffffu, (uint32_t)lane < lc.n_tk && val != RING_NONE);
  const uint32_t nb = (filled == 0xffffffffu) ? 32u : (uint32_t)__ffs((int)~filled) - 1u;   // leading filled tickets (at least the first)
  *slot_out = val;
  const uint32_t carried = __shfl_down_sync(0xffffffffu, lc.tk, nb);   // unfilled tickets move to the front
  lc.n_tk -= nb;
  if ((uint32_t)lane < lc.n_tk) lc.tk = carried;
  return nb;
}

__device__ __forceinline__ void flush_counters(const Trees& T, const unsigned long long* local, int lane) {
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < CTR_COUNT; ++i)
      if (local[i]) atomicAdd(&T.counters[i], local[i]);
  }
}

// ---- evaluation cache (tree.cuh: EvalCache) ------------------------------------------------------------------------
// The evaluator is a pure function of the 16-byte position, so a leaf whose position tree g has already sent to the
// evaluator in this search gets that record back from the cache, with the same bits the evaluator would produce again.
// Only the warp that owns tree g touches its table.  Reads go to L2 (ld.cg): the previous owner of the tree was another
// SM, and a line of this SM's L1 left from an earlier visit could pair a fresh key with a stale record.  Writes reach the
// next owner through the __threadfence + release of the ring push, as the node records do.
constexpr uint32_t CACHE_NONE = 0xFFFFFFFFu;

// One warp-wide probe: lane i examines slot (hash + i) mod slots.  Returns the first slot of the window that holds `st`
// (hit = true) or is empty (hit = false: where its record goes once evaluated); CACHE_NONE = no table or a full window.
// A hit needs all 128 bits of the key to be equal.
__device__ __forceinline__ uint32_t cache_probe(const EvalCache& E, uint32_t epoch, uint32_t g, const PState& st, int lane, bool& hit) {
  hit = false;
  if (E.key == nullptr) return CACHE_NONE;
  const uint32_t s = ((uint32_t)splitmix64(st.x ^ splitmix64(st.o)) + (uint32_t)lane) & (E.slots - 1u);
  const size_t e = (size_t)g * E.slots + s;
  const uint32_t ep = __ldcg(E.epoch + e);
  const ulonglong2 k = __ldcg(E.key + e);
  const bool empty = ep != epoch;
  const uint32_t stop = __ballot_sync(0xffffffffu, empty || (k.x == st.x && k.y == st.o));
  if (stop == 0u) return CACHE_NONE;
  const int first = __ffs((int)stop) - 1;
  hit = !__shfl_sync(0xffffffffu, empty, first);
  return __shfl_sync(0xffffffffu, s, first);
}

// Entry `s` of tree g := (st, record, epoch).  Lane a writes word a of the record (words past the value are padding).
template <class G>
__device__ __forceinline__ void cache_insert(const EvalCache& E, uint32_t epoch, uint32_t g, uint32_t s, const PState& st,
                                             const float* probs, float v, int lane) {
  const size_t e = (size_t)g * E.slots + s;
  float w = 0.0f;
#pragma unroll
  for (int a = 0; a < G::A; ++a) if (lane == a) w = probs[a];
  if (lane == G::A) w = v;
  if (lane < G::EVAL_STRIDE) E.rec[e * G::EVAL_STRIDE + lane] = w;
  if (lane == 0) {
    E.key[e] = make_ulonglong2(st.x, st.o);
    E.epoch[e] = epoch;
  }
}

// expand of an evaluated leaf with its record's probabilities (mcts.rs:278-281), then the backup of its value along the
// path (mcts.rs:282-284).  false = the node pool is full (reported in the error word).
template <class G>
__device__ __forceinline__ bool expand_backup(const Trees& T, uint32_t g, NodeRec* rec, uint32_t* par, uint32_t& n_nodes, uint32_t leaf,
                                              const PState& st, const float* probs, float v, const WarpPath& path, int depth, int lane,
                                              unsigned long long* ctr) {
  const uint32_t before = n_nodes;
  if (!expand<G>(rec, par, T.cap, n_nodes, leaf, st, probs, lane)) {
    if (lane == 0) atomicOr(T.error, ERRBIT_POOL);
    return false;
  }
  ctr[CTR_CHILDREN] += n_nodes - before;
  if (lane == 0) T.n_nodes[g] = n_nodes;
  backup_regs(rec, path, depth, v, lane);                           // backprop, mcts.rs:145-159: N += 1, W += +-v
  return true;
}

// One visit of tree g to a tree warp: expand + backup of the evaluated leaf (mcts.rs:278-284), then selects
// (mcts.rs:236-252) until a leaf needs the evaluator or the tree has started all its simulations.  Terminal leaves are
// backed up at once and the tree carries on: in the reference they take part in the iteration without an evaluation.
// So are leaves whose position the evaluation cache holds: expand + backup with the cached record, then the next select.
template <class G>
__device__ __forceinline__ void tree_phase(const Trees& T, const AsyncCtl& C, uint32_t g, int lane, unsigned long long* ctr) {
  const uint32_t slot = g;                                          // one leaf in flight per tree
  uint32_t* pathm = T.path + (size_t)slot * G::MAX_DEPTH;
  const uint32_t b = T.buf[g];                                      // constant during a search
  const PState root = T.root_state[g];                              // constant during a search
  uint32_t li = __ldcg(&T.leaf_info[slot]);
  uint32_t n_nodes = __ldcg(&T.n_nodes[g]);
  uint32_t remaining = __ldcg(&C.sims_left[g]);
  NodeRec* rec = T.rec[b] + (size_t)g * T.cap;
  uint32_t* par = T.par[b] + (size_t)g * T.cap;
  WarpPath path;
  uint32_t leaf = 0;
  int depth = 0;
  PState st{};
  const float* src = nullptr;                                       // record of the leaf to expand: eval_out or the cache

  if (li & LEAF_PENDING) {                                          // the evaluator's record has arrived
    depth = (int)(li & 0xFFu);
    {
      const ulonglong2 raw = __ldcg(reinterpret_cast<const ulonglong2*>(&T.leaf_state[slot]));
      st.x = raw.x; st.o = raw.y;
    }
    const uint32_t pn0 = (lane < G::MAX_DEPTH) ? __ldcg(pathm + lane) : 0u;
    const uint32_t pn1 = (lane + 32 < G::MAX_DEPTH) ? __ldcg(pathm + lane + 32) : 0u;
    leaf = __shfl_sync(0xffffffffu, depth < 32 ? pn0 : pn1, depth & 31);
    SPB_ASSERT(T.error, depth < G::MAX_DEPTH && (lane > depth || pn0 < n_nodes) && (lane + 32 > depth || pn1 < n_nodes), 2);
    uint2 nw0 = make_uint2(0, 0), nw1 = make_uint2(0, 0);           // the path in registers, as the descent left it
    if (lane <= depth) nw0 = __ldcg(reinterpret_cast<const uint2*>(&rec[pn0]));
    if (lane + 32 <= depth) nw1 = __ldcg(reinterpret_cast<const uint2*>(&rec[pn1]));
    path.node[0] = pn0; path.N[0] = nw0.x; path.W[0] = __uint_as_float(nw0.y);
    path.node[1] = pn1; path.N[1] = nw1.x; path.W[1] = __uint_as_float(nw1.y);
    src = T.eval_out + (size_t)slot * G::EVAL_STRIDE;
  }

  for (;;) {
    if (src != nullptr) {
      float probs[G::A];
#pragma unroll
      for (int a = 0; a < G::A; ++a) probs[a] = __ldcg(src + a);
      const float v = __ldcg(src + G::A);
      if (li & LEAF_PENDING) {                                      // the network's record: into the cache, for the next visits
        const uint32_t ins = li >> LEAF_INSERT_SHIFT;
        if (ins != 0u) cache_insert<G>(C.cache, C.epoch, g, ins - 1u, st, probs, v, lane);
        if (lane == 0) T.leaf_info[slot] = 0;
        li = 0;
      }
      src = nullptr;
      const bool ok = expand_backup<G>(T, g, rec, par, n_nodes, leaf, st, probs, v, path, depth, lane, ctr);
      __syncwarp();
      if (!ok) break;
    }
    if (remaining == 0) break;
    --remaining;
    uint32_t linfo;
    descend<G, true>(rec, root, T.c, root_noise_of(T, g), lane, path, leaf, depth, st, linfo, T.error, n_nodes);
    SPB_ASSERT(T.error, leaf < n_nodes && depth < G::MAX_DEPTH, 3);
    ctr[CTR_SIMS] += 1;
    ctr[CTR_PATHSUM] += (unsigned)depth;
    const uint32_t status = info_status(linfo);
    if (status != SPB_STATUS_ONGOING) {                             // mcts.rs:245-247
      ctr[CTR_TERMINAL] += 1;
      backup_regs(rec, path, depth, terminal_value(status), lane);
      __syncwarp();
      continue;
    }
    ctr[CTR_EVALS] += 1;                                            // mcts.rs:249-250: the leaf goes to the evaluator
    bool hit;
    const uint32_t cs = cache_probe(C.cache, C.epoch, g, st, lane, hit);
    if (hit) {                                                      // ... which gave its record earlier in this search
      src = C.cache.rec + ((size_t)g * C.cache.slots + cs) * G::EVAL_STRIDE;
      continue;
    }
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int d = lane + 32 * s;
      if (d <= depth) pathm[d] = path.node[s];
    }
    if (lane == 0) {
      T.leaf_state[slot] = st;
      T.leaf_info[slot] = (uint32_t)depth | LEAF_PENDING | ((cs + 1u) << LEAF_INSERT_SHIFT);   // CACHE_NONE + 1 = 0: no insert
      C.sims_left[g] = remaining;
    }
    __threadfence();                                                // every lane's stores are at L2 before the hand-off
    __syncwarp();
    if (lane == 0) ring_push(C.leaf, slot);
    return;
  }
  // all simulations of this tree have completed (or its node pool is full): the tree leaves the pipeline
  if (lane == 0) {
    C.sims_left[g] = 0;
    __threadfence();
    atomicAdd(C.done_count, 1u);
  }
}

// A tree warp: serves trees from the ready ring until the search is over.
template <class G>
__device__ __forceinline__ void tree_worker(const Trees& T, const AsyncCtl& C, int lane) {
  unsigned long long ctr[CTR_COUNT] = {0, 0, 0, 0, 0};
  Spin sp;
  sp.init(C, *C.n_active);
  unsigned long long busy = 0, phases = 0;
  for (;;) {
    uint32_t g = RING_NONE;
    if (lane == 0) g = ready_pop_wait(C, sp);
    g = __shfl_sync(0xffffffffu, g, 0);
    if (g == RING_NONE) break;
    SPB_ASSERT(T.error, g < T.G, 4);
    const unsigned long long t0 = gtime_ns();
    tree_phase<G>(T, C, g, lane, ctr);
    busy += gtime_ns() - t0;
    ++phases;
  }
  flush_counters(T, ctr, lane);
  if (lane == 0) {
    atomicAdd(&C.stats[ASTAT_TREE_BUSY_NS], busy);
    atomicAdd(&C.stats[ASTAT_TREE_PHASES], phases);
    atomicAdd(&C.stats[ASTAT_TREE_WARPS], 1ull);
    atomicAdd(&C.stats[ASTAT_READY_BACKLOG], sp.backlog);
    atomicAdd(&C.stats[ASTAT_READY_STARVED], sp.starved);
  }
}

// Evaluator stand-in for the asynchronous pipeline (parity harness): DetEval / uniform on the leaves of the ring, one
// lane per leaf, same claim / publish protocol as the network evaluator.
template <class G, int EVAL>
__device__ __forceinline__ void builtin_eval_worker(const Trees& T, const AsyncCtl& C, uint32_t n_workers, int lane) {
  Spin sp;
  sp.init(C, *C.n_active);
  LeafClaimer lc;
  unsigned long long boards = 0;
  for (;;) {
    uint32_t slot = RING_NONE;
    const uint32_t k = claim_batch(C, lc, n_workers, 32u, 2000u, sp, lane, &slot);
    if (k == 0) {
      if (lane == 0) atomicAdd(&C.stats[ASTAT_BOARDS], boards);   // positions evaluated, as the network's stager counts them
      break;
    }
    boards += k;
    SPB_ASSERT(T.error, (uint32_t)lane >= k || slot < T.G * T.K, 5);
    if ((uint32_t)lane < k) {
      PState st;
      const ulonglong2 raw = __ldcg(reinterpret_cast<const ulonglong2*>(&T.leaf_state[slot]));
      st.x = raw.x; st.o = raw.y;
      float probs[G::A], v;
      if (EVAL == SPB_EVAL_DET) det_eval<G>(st, probs, &v); else uniform_eval<G>(st, probs, &v);
      float* o = T.eval_out + (size_t)slot * G::EVAL_STRIDE;
#pragma unroll
      for (int a = 0; a < G::A; ++a) o[a] = probs[a];
      o[G::A] = v;
    }
    ring_push_warp(C.ready, k, slot, lane);
  }
}

}  // namespace spb
