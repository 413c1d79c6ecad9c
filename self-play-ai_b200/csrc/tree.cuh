// tree.cuh — structure-of-arrays MCTS node pools in HBM and the warp-per-tree primitives.
//
// Replaces src/mcts.rs of the reference: Node (mcts.rs:20-30), Tree (:32-39), get_ucb (:91-100),
// select (:102-114), expand (:116-143), backprop (:145-159), use_subtree (:161-192).
//
// Layout (per engine):
//   rec[b][g*cap + id]   16 B  {visit_count u32, value_sum f32, prior f32, info u32}
//                              info = first_child[0,24) | n_children[24,28) | status[28,30)
//                              A parent's children are contiguous and in get_valid_actions order
//                              (mcts.rs:121-122), so 7 children = 112 contiguous bytes read as
//                              one LDG.128 per lane.
//   par[b][g*cap + id]    4 B  parent_id[0,24) | action_taken[24,32)   (root: parent 0xFFFFFF)
//   b = buf[g] selects one of two arenas; use_subtree compacts from one into the other.
//   root_state[g]        16 B  packed position of arena[0]; node states are NOT stored — a warp
//                              replays the moves while it descends (a few bitboard ops per level).
#pragma once
#include "games.cuh"

namespace spb {

struct __align__(16) NodeRec {
  uint32_t N;
  float W;
  float P;
  uint32_t info;
};
static_assert(sizeof(NodeRec) == 16, "NodeRec must be 16 bytes");

constexpr uint32_t INFO_FC_MASK = 0xFFFFFFu;
constexpr int INFO_NC_SHIFT = 24, INFO_STATUS_SHIFT = 28;
constexpr uint32_t PAR_NONE = 0xFFFFFFu;
constexpr uint32_t MAX_CAP = 1u << 24;

__host__ __device__ __forceinline__ uint32_t info_fc(uint32_t info) { return info & INFO_FC_MASK; }
__host__ __device__ __forceinline__ uint32_t info_nc(uint32_t info) { return (info >> INFO_NC_SHIFT) & 15u; }
__host__ __device__ __forceinline__ uint32_t info_status(uint32_t info) { return (info >> INFO_STATUS_SHIFT) & 3u; }
__host__ __device__ __forceinline__ uint32_t make_info(uint32_t fc, uint32_t nc, uint32_t status) {
  return (fc & INFO_FC_MASK) | (nc << INFO_NC_SHIFT) | (status << INFO_STATUS_SHIFT);
}

enum CounterIdx { CTR_SIMS = 0, CTR_EVALS, CTR_TERMINAL, CTR_PATHSUM, CTR_CHILDREN, CTR_COUNT };
enum ErrorBits : uint32_t { ERRBIT_POOL = 1u, ERRBIT_NAN = 2u, ERRBIT_TRAJ_FULL = 4u, ERRBIT_BOUNDS = 8u };

// Checked build (make VARIANT=-DSPB_BOUNDS_CHECK; tools/build_variant.sh check -DSPB_BOUNDS_CHECK): every index the tree,
// ring and self-play kernels form is compared with the extent of the array it addresses; a failure sets ERRBIT_BOUNDS and
// the site's code in bits 8..15 of the error word, and the next API call returns SPB_ERR_STATE naming it.  This is the
// stand-in for compute-sanitizer memcheck, which is closed on the GPU pool this was developed on (profiles/r02_sanitizer.txt).
#ifdef SPB_BOUNDS_CHECK
#define SPB_ASSERT(err, cond, code) do { if (!(cond)) atomicOr((err), (uint32_t)ERRBIT_BOUNDS | ((uint32_t)(code) << 8)); } while (0)
#else
#define SPB_ASSERT(err, cond, code) ((void)0)
#endif

// leaf_info[slot]: depth[0,8) | pending-eval flag (bit 8) | asynchronous pipeline: evaluation-cache insert position + 1
// [9,32) (0 = no insert)
constexpr uint32_t LEAF_PENDING = 1u << 8;
constexpr int LEAF_INSERT_SHIFT = 9;

// Evaluation cache of the asynchronous pipeline (async.cuh, DESIGN.md §4.2a): per tree an open-addressed table of the
// records the evaluator produced during the current search, keyed by the full 16-byte position.  An entry is live only
// while its epoch equals the search's epoch, so the table is never cleared between searches.  key = nullptr: no table
// (every lookup misses).
constexpr uint32_t EVAL_CACHE_MAX_SLOTS = 4096;   // per tree; the table holds num_searches records at load <= 0.5 up to here
constexpr int EVAL_CACHE_WINDOW = 32;             // consecutive slots one probe examines (one per lane)
struct EvalCache {
  ulonglong2* key;       // [G][slots]  PState {x, o} of the entry
  uint32_t* epoch;       // [G][slots]  search epoch that wrote the entry (0 = never written)
  float* rec;            // [G][slots][EVAL_STRIDE]  the evaluator's record: unmasked softmax + value
  uint32_t slots;        // per tree, a power of two
};

struct Trees {
  NodeRec* rec[2];
  uint32_t* par[2];
  PState* root_state;
  uint32_t* n_nodes;
  uint8_t* buf;
  uint8_t* live;
  uint32_t cap;
  uint32_t G;
  uint32_t K;            // leaves per tree per step
  float c;
  // per leaf slot (g*K + k)
  uint32_t* path;        // [G*K][MAX_DEPTH]
  uint32_t* leaf_info;   // [G*K]
  PState* leaf_state;    // [G*K]  evaluator input
  uint32_t* eval_list;   // [G*K]  compacted leaf slots that need the evaluator
  uint32_t* eval_count;  // [1]
  float* eval_out;       // [G*K][EVAL_STRIDE]  probs (softmax, unmasked) + value
  unsigned long long* counters;  // [CTR_COUNT]
  uint32_t* error;       // [1]
  // EXTENSION: Dirichlet noise at the root (root_noise.cuh, DESIGN.md §4.6).  root_noise is nullptr while the noise is off.
  float* root_noise;     // [G][SPB_MAX_ACTIONS]  eta of the current root, child order (k_root_noise)
  uint32_t* noise_n;     // [G]  number of root children eta was drawn for
  float noise_eps, noise_omeps;   // epsilon and 1 - epsilon (rounded to f32 once, on the host)
};

// The root's noise as a descent sees it: the engine's eta array (nullptr -> the stored priors everywhere), the tree's row
// of it and the two mixing weights.  The row's address is formed only at depth 0.
struct RootNoise {
  const float* eta;      // [G][stride]
  uint32_t row;          // g * stride
  float eps, omeps;
};
__device__ __forceinline__ RootNoise root_noise_of(const Trees& T, uint32_t g) {
  return RootNoise{T.root_noise, g * (uint32_t)SPB_MAX_ACTIONS, T.noise_eps, T.noise_omeps};
}
// P' = (1 - eps) * P + eps * eta, each operation rounded (no FMA contraction); the stored prior is never modified.
__device__ __forceinline__ float noisy_prior(float prior, float eta, float eps, float omeps) {
  return __fadd_rn(__fmul_rn(omeps, prior), __fmul_rn(eps, eta));
}

// get_ucb, mcts.rs:91-100 — every operation individually rounded (no FMA contraction), evaluated in
// the reference's order: q + ((c * prior) * sqrt(N_parent)) / (1 + N_child).
__device__ __forceinline__ float puct_score(float c, uint32_t n_parent, uint32_t n_child, float w_child, float prior) {
  float q = 0.0f;                                              // :95 unvisited child -> q = 0.0
  if (n_child != 0)
    q = __fmul_rn(__fadd_rn(__fdiv_rn(-w_child, (float)n_child), 1.0f), 0.5f);   // :97 (x / 2.0 and x * 0.5 round identically)
  float u = __fmul_rn(c, prior);
  u = __fmul_rn(u, __fsqrt_rn((float)n_parent));
  u = __fdiv_rn(u, __fadd_rn(1.0f, (float)n_child));
  return __fadd_rn(q, u);
}

// select, mcts.rs:102-114: arg-max over the children with Iterator::max_by semantics — among equal
// maxima the LAST child wins.  Lanes >= nc carry (-inf, -1).  Returns the winning child index.
template <int MAX_CHILDREN>
__device__ __forceinline__ int warp_argmax_last(float score, int idx) {
#pragma unroll
  for (int off = (MAX_CHILDREN > 8 ? 8 : 4); off >= 1; off >>= 1) {   // butterfly over the 8 / 16 lanes that can hold a child
    float os = __shfl_xor_sync(0xffffffffu, score, off);
    int oi = __shfl_xor_sync(0xffffffffu, idx, off);
    if (os > score || (os == score && oi > idx)) { score = os; idx = oi; }
  }
  return idx;   // the lanes of the butterfly agree; callers broadcast from lane 0
}

// Path of one simulation, distributed over the warp: lane d holds depth d (set 0) and depth d+32 (set 1).
struct WarpPath {
  uint32_t node[2];
  uint32_t N[2];
  float W[2];
};

// Node-record load.  COHERENT = read at L2 (ld.global.cg): required when another SM may have written the tree since this SM
// last cached it (the asynchronous pipeline hands a tree from SM to SM); the lock-step and fused kernels keep L1.
template <bool COHERENT>
__device__ __forceinline__ NodeRec ld_rec(const NodeRec* p) {
  if (COHERENT) {
    const uint4 v = __ldcg(reinterpret_cast<const uint4*>(p));
    NodeRec r;
    r.N = v.x; r.W = __uint_as_float(v.y); r.P = __uint_as_float(v.z); r.info = v.w;
    return r;
  }
  return *p;
}

// Descend from the root to a leaf (mcts.rs:237-241), replaying the moves on the bitboards.
// All lanes return the same (leaf, depth, st, leaf_info).  With noise.eta set, the root's children (depth 0 only) are
// scored with the noisy prior.
template <class G, bool COHERENT = false>
__device__ __forceinline__ void descend(const NodeRec* rec, const PState& root, float c, const RootNoise& noise, int lane,
                                        WarpPath& path, uint32_t& leaf, int& depth, PState& st, uint32_t& leaf_info,
                                        uint32_t* err, uint32_t n_nodes = 0xFFFFFFFFu) {
  NodeRec r0 = ld_rec<COHERENT>(rec);
  uint32_t node = 0, Np = r0.N, info = r0.info;
  st = root;
  depth = 0;
  if (lane == 0) { path.node[0] = 0; path.N[0] = r0.N; path.W[0] = r0.W; }
  while (info_nc(info) != 0) {
    const int nc = (int)info_nc(info);
    const uint32_t fc = info_fc(info);
    NodeRec ch;
    ch.N = 0; ch.W = 0.0f; ch.P = 0.0f; ch.info = 0;
    float score = -INFINITY;
    int idx = -1;
    SPB_ASSERT(err, fc + (uint32_t)nc <= n_nodes && nc <= G::A && depth + 1 < G::MAX_DEPTH, 1);
    if (lane < nc) {
      ch = ld_rec<COHERENT>(rec + fc + lane);                // 16-B vector load, children contiguous
      float p = ch.P;
      if (noise.eta != nullptr && depth == 0) p = noisy_prior(p, noise.eta[noise.row + lane], noise.eps, noise.omeps);
      score = puct_score(c, Np, ch.N, ch.W, p);
      idx = lane;
      if (score != score) atomicOr(err, ERRBIT_NAN);         // the reference would panic (partial_cmp().unwrap())
    }
    int best = warp_argmax_last<G::A>(score, idx);
    best = __shfl_sync(0xffffffffu, best, 0);
    uint32_t bN = __shfl_sync(0xffffffffu, ch.N, best);
    float bW = __shfl_sync(0xffffffffu, ch.W, best);
    uint32_t binfo = __shfl_sync(0xffffffffu, ch.info, best);
    // The children are in ascending action order (expand): child `best` is the action whose rank among the legal
    // actions is `best`.  Lane a tests action a; two ballots replace the mask loop and the n-th-set-bit search.
    const bool lb = lane < G::A && G::action_legal(st, lane);
    const uint32_t legal = __ballot_sync(0xffffffffu, lb);
    const uint32_t hit = __ballot_sync(0xffffffffu, lb && __popc(legal & ((1u << lane) - 1u)) == best);
    const int action = __ffs((int)hit) - 1;
    st = G::place(st, action, info_status(binfo));
    node = fc + (uint32_t)best;
    ++depth;
    if (depth < 32) {                                        // static register indices: no select chains
      if (lane == depth) { path.node[0] = node; path.N[0] = bN; path.W[0] = bW; }
    } else if (lane == depth - 32) {
      path.node[1] = node; path.N[1] = bN; path.W[1] = bW;
    }
    Np = bN;
    info = binfo;
  }
  leaf = node;
  leaf_info = info;
}

// backprop, mcts.rs:145-159, with the path held in registers: lane d updates the node at depth d.
// The leaf gets +v, its parent -v, ... (sign flips at every level).
__device__ __forceinline__ void backup_regs(NodeRec* rec, const WarpPath& path, int depth, float v, int lane) {
#pragma unroll
  for (int s = 0; s < 2; ++s) {
    int d = lane + 32 * s;
    if (d <= depth) {
      float sv = ((depth - d) & 1) ? -v : v;
      uint2 nw;
      nw.x = path.N[s] + 1u;
      nw.y = __float_as_uint(__fadd_rn(path.W[s], sv));
      *reinterpret_cast<uint2*>(&rec[path.node[s]]) = nw;   // {N, W} are the first 8 bytes of the record
    }
  }
}

// backprop with the path in global scratch (the evaluator kernel ran in between).
__device__ __forceinline__ void backup_mem(NodeRec* rec, const uint32_t* path, int depth, float v, int lane) {
  for (int d = lane; d <= depth; d += 32) {
    uint32_t node = path[d];
    uint2 nw = *reinterpret_cast<const uint2*>(&rec[node]);
    float sv = ((depth - d) & 1) ? -v : v;
    nw.x += 1u;
    nw.y = __float_as_uint(__fadd_rn(__uint_as_float(nw.y), sv));
    *reinterpret_cast<uint2*>(&rec[node]) = nw;
  }
}

// expand, mcts.rs:116-143: append one child per legal action (ascending action order), ids contiguous
// [n_nodes, n_nodes+nc).  probs = evaluator output BEFORE masking; mask_invalid_actions is applied here
// (model/mod.rs:86-93).  Returns false on pool overflow.
template <class G>
__device__ __forceinline__ bool expand(NodeRec* rec, uint32_t* par, uint32_t cap, uint32_t& n_nodes, uint32_t leaf,
                                       const PState& st, const float* probs, int lane) {
  // Lane a tests action a (the leaf is an ongoing position); the ballot is get_valid_actions' mask and the rank of a
  // legal action among the legal ones is its child index, so children come out in ascending action order.
  const bool lb = lane < G::A && G::action_legal(st, lane);
  const uint32_t legal = __ballot_sync(0xffffffffu, lb);
  const int nc = __popc(legal);
  const uint32_t first = n_nodes;
  if (first + (uint32_t)nc > cap) return false;
  if (lb) {
    const int a = lane;
    const uint32_t ci = first + (uint32_t)__popc(legal & ((1u << lane) - 1u));
    PState child;
    G::next_state(st, a, &child);                            // :129 (cannot fail: a is legal)
    const float p = mask_renorm_one<G>(legal, probs, a);     // :128 policy.get_prob(&action) of the masked, renormalised policy
    NodeRec r;
    r.N = 0; r.W = 0.0f; r.P = p;
    r.info = make_info(0, 0, ps_status(child));
    rec[ci] = r;
    par[ci] = leaf | ((uint32_t)a << 24);
  }
  if (lane == 0) rec[leaf].info = make_info(first, (uint32_t)nc, SPB_STATUS_ONGOING);
  n_nodes = first + (uint32_t)nc;
  return true;
}

}  // namespace spb
