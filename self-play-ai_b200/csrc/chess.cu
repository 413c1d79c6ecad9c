// chess.cu — batched chess rules on the device behind the C ABI (include/selfplay_b200.h, spb_chess_*).
// Rules: chess.cuh (bitboards, __host__ __device__); reference: src/game/chess.rs.  BASELINE config 5, first half: the
// State / Policy interface of the chess adapter as device kernels, validated by perft and an array-board oracle.  The
// chess search (trees over these rules, the 10x256 net of src/model/chess.rs) is the next step, see DESIGN.md §7.
#include "chess_engine.hpp"

namespace spb {
namespace chess {

__global__ void k_legal(const Pos* states, const uint64_t* history, uint32_t n, Move* moves, uint32_t* counts, uint16_t* pidx,
                        uint8_t* status_out, uint32_t* reps) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Pos p = states[i];
  Move mv[MAX_MOVES];
  const int m = legal_moves(p, mv);
  const uint64_t h = move_list_hash(mv, m);
  const uint64_t* hist = history ? history + (size_t)i * SPB_CHESS_MAX_HISTORY : nullptr;
  const uint32_t hl = hist ? min(p.hist_len, (uint32_t)SPB_CHESS_MAX_HISTORY) : 0u;
  if (counts) counts[i] = (uint32_t)m;
  if (reps) reps[i] = num_repetitions(h, hist, hl);
  if (status_out) status_out[i] = (uint8_t)status(p, m, h, hist, hl);
  for (int k = 0; k < m; ++k) {
    if (moves) moves[(size_t)i * MAX_MOVES + k] = mv[k];
    if (pidx) pidx[(size_t)i * MAX_MOVES + k] = (uint16_t)policy_index(p.side, mv[k]);
  }
}

__global__ void k_next(const Pos* states, uint64_t* history, const Move* moves, uint32_t n, Pos* out, int32_t* err) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Pos p = states[i];
  Move mv[MAX_MOVES];
  const int m = legal_moves(p, mv);
  const uint64_t h = move_list_hash(mv, m);
  uint64_t* hist = history ? history + (size_t)i * SPB_CHESS_MAX_HISTORY : nullptr;
  const uint32_t hl = hist ? min(p.hist_len, (uint32_t)SPB_CHESS_MAX_HISTORY) : 0u;
  out[i] = p;
  if (status(p, m, h, hist, hl) != SPB_STATUS_ONGOING) { err[i] = SPB_ERR_ILLEGAL; return; }   // chess.rs:113-115
  bool found = false;
  for (int k = 0; k < m; ++k) found |= mv[k] == moves[i];
  if (!found) { err[i] = SPB_ERR_ILLEGAL; return; }                                           // chess.rs:146
  if (!hist || p.hist_len >= SPB_CHESS_MAX_HISTORY) { err[i] = SPB_ERR_STATE; return; }
  hist[p.hist_len] = h;                                                                       // chess.rs:121-122
  Pos q = apply_move(p, moves[i]);
  q.hist_len = p.hist_len + 1;
  out[i] = q;
  err[i] = SPB_OK;
}

__global__ void k_encode(const Pos* states, const uint64_t* history, uint32_t n, float* out) {
  // one block per state: the repetition count needs the legal moves of the position (thread 0), then 19 x 64 values
  __shared__ uint32_t s_reps;
  const uint32_t i = blockIdx.x;
  if (i >= n) return;
  const Pos p = states[i];
  if (threadIdx.x == 0) {
    Move mv[MAX_MOVES];
    const int m = legal_moves(p, mv);
    const uint64_t* hist = history ? history + (size_t)i * SPB_CHESS_MAX_HISTORY : nullptr;
    s_reps = num_repetitions(move_list_hash(mv, m), hist, hist ? min(p.hist_len, (uint32_t)SPB_CHESS_MAX_HISTORY) : 0u);
  }
  __syncthreads();
  for (int t = threadIdx.x; t < SPB_CHESS_PLANES * 64; t += blockDim.x)
    out[(size_t)i * SPB_CHESS_PLANES * 64 + t] = encode_plane(p, s_reps, t / 64, (t / 8) % 8, t % 8);
}

// perft of the frontier positions, depth <= PERFT_DEV_DEPTH below each: iterative (explicit stack of move lists), so
// that the kernel's local memory is sized statically instead of through the device's recursion stack limit.
constexpr int PERFT_DEV_DEPTH = 4;
__global__ void k_perft(const Pos* frontier, uint32_t n, int depth, unsigned long long* total) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  unsigned long long nodes = 0;
  if (depth <= 0) {
    nodes = 1;
  } else {
    Pos pos[PERFT_DEV_DEPTH];
    Move mv[PERFT_DEV_DEPTH][MAX_MOVES];
    int cnt[PERFT_DEV_DEPTH], idx[PERFT_DEV_DEPTH];
    int d = 0;
    pos[0] = frontier[i];
    cnt[0] = legal_moves(pos[0], mv[0]);
    idx[0] = 0;
    for (;;) {
      if (d == depth - 1) {                                           // the moves of this level are the leaves
        nodes += (unsigned long long)cnt[d];
        if (--d < 0) break;
        continue;
      }
      if (idx[d] >= cnt[d]) {
        if (--d < 0) break;
        continue;
      }
      pos[d + 1] = apply_move(pos[d], mv[d][idx[d]++]);
      ++d;
      cnt[d] = legal_moves(pos[d], mv[d]);
      idx[d] = 0;
    }
  }
  atomicAdd(total, nodes);
}

// Breadth-first frontier of perft: pass 1 counts the legal moves of every position and reserves its output range, pass 2
// writes the successor positions there (their order does not matter for a leaf count).
__global__ void k_frontier_count(const Pos* frontier, uint32_t n, uint32_t* offset, unsigned long long* total) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Move mv[MAX_MOVES];
  const int m = legal_moves(frontier[i], mv);
  offset[i] = (uint32_t)atomicAdd(total, (unsigned long long)m);
}
__global__ void k_frontier_expand(const Pos* frontier, uint32_t n, const uint32_t* offset, Pos* next) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Pos p = frontier[i];
  Move mv[MAX_MOVES];
  const int m = legal_moves(p, mv);
  for (int k = 0; k < m; ++k) next[offset[i] + k] = apply_move(p, mv[k]);
}

// ---- training tensors of self-play records on the device (spb_chess_positions_to_training_device) ----------------------
// Pass 1 validates every row as spb_chess_positions_to_training does, plus the index range; the first bad row goes to *bad
// (atomicMin; ~0 = none).  One warp per row, grid-stride: the lanes read the row's moves coalesced.
__global__ void __launch_bounds__(256) k_chess_training_check(const spb_chess_position* __restrict__ pos, unsigned long long n_positions,
                                                              const unsigned long long* __restrict__ indices, unsigned long long n,
                                                              unsigned long long* bad) {
  const int lane = threadIdx.x & 31;
  const unsigned long long warps = (unsigned long long)gridDim.x * (blockDim.x / 32);
  for (unsigned long long i = blockIdx.x * (unsigned long long)(blockDim.x / 32) + threadIdx.x / 32; i < n; i += warps) {
    const unsigned long long src = indices ? indices[i] : i;
    bool ok = src < n_positions;
    if (ok) {
      const spb_chess_position& p = pos[src];
      const uint32_t nm = p.n_moves, side = p.state.side;
      ok = nm >= 1 && nm <= SPB_CHESS_MAX_MOVES && side <= 1;
      if (ok)
        for (uint32_t k = lane; k < nm; k += 32) {
          const int idx = policy_index((int)side, p.moves[k]);
          ok &= idx >= 0 && idx < SPB_CHESS_POLICY_SIZE;
        }
      ok = __all_sync(0xffffffffu, ok);
    }
    if (!ok && lane == 0) atomicMin(bad, i);
  }
}

constexpr int TRAIN_THREADS = 256;                                     // one thread per child of a record
constexpr int REC_WORDS = sizeof(spb_chess_position) / 8;
static_assert(sizeof(spb_chess_position) % 8 == 0, "records are loaded with 8-byte words");
static_assert(SPB_CHESS_MAX_MOVES == TRAIN_THREADS, "the scatter gives child k to thread k");
static_assert(SPB_CHESS_POLICY_SIZE % 4 == 0 && (SPB_CHESS_PLANES * 64) % 4 == 0, "rows are whole float4s");

// Pass 2 (rows validated): one CTA per row at a time.  The record is staged in shared memory, the policy row is built there
// (zero, f32 sum of the counts in child order on one thread, count / sum scattered by policy index with the later child
// winning a duplicated index, as on the host), then the encoding and policy rows are written once each: 16-byte streaming
// stores when the outputs are 16-byte aligned (row strides are multiples of 16 bytes), scalar stores otherwise.  Every
// output float is written exactly once: the kernel is bound by HBM writes (23,556 bytes out per 1,624 read).
__global__ void __launch_bounds__(TRAIN_THREADS) k_chess_training(const spb_chess_position* __restrict__ pos,
                                                                  const unsigned long long* __restrict__ indices, unsigned long long n,
                                                                  float* __restrict__ encodings, float* __restrict__ policies,
                                                                  float* __restrict__ values, bool vec_enc, bool vec_pol) {
  __shared__ unsigned long long s_rec[REC_WORDS];
  __shared__ __align__(16) float s_pol[SPB_CHESS_POLICY_SIZE];
  __shared__ float s_sum;
  const spb_chess_position& r = *reinterpret_cast<const spb_chess_position*>(s_rec);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  constexpr int ENC = SPB_CHESS_PLANES * 64;
  for (unsigned long long i = blockIdx.x; i < n; i += gridDim.x) {
    const unsigned long long src = indices ? indices[i] : i;
    const unsigned long long* g = reinterpret_cast<const unsigned long long*>(pos + src);
    for (int w = t; w < REC_WORDS; w += TRAIN_THREADS) s_rec[w] = __ldg(g + w);
    if (policies) {
      float4* z = reinterpret_cast<float4*>(s_pol);
      for (int w = t; w < SPB_CHESS_POLICY_SIZE / 4; w += TRAIN_THREADS) z[w] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    const int nm = r.n_moves, side = r.state.side;
    if (policies) {
      if (t == 0) {
        float s = 0.0f;
        for (int k = 0; k < nm; ++k) s += (float)r.visit_counts[k];
        s_sum = s;
      }
      __syncthreads();
      const bool mine = t < nm;
      const int idx = mine ? policy_index(side, r.moves[t]) : -1;
      const float v = mine ? (float)r.visit_counts[t] / s_sum : 0.0f;
      // warp w writes in round w, so a later warp overwrites an earlier one; inside a warp the highest lane of a group of
      // equal indices writes
      const unsigned same = __match_any_sync(0xffffffffu, idx);
      const bool last = (31 - __clz(same)) == lane;
      for (int round = 0; round * 32 < nm; ++round) {
        if (warp == round && mine && last) s_pol[idx] = v;
        __syncthreads();
      }
    }
    if (encodings) {
      float* o = encodings + i * (unsigned long long)ENC;
      if (vec_enc) {
        for (int w = t; w < ENC / 4; w += TRAIN_THREADS) {
          const int e0 = w * 4;
          float4 q;
          q.x = encode_plane(r.state, r.repetitions, e0 / 64, (e0 / 8) % 8, e0 % 8);
          q.y = encode_plane(r.state, r.repetitions, (e0 + 1) / 64, ((e0 + 1) / 8) % 8, (e0 + 1) % 8);
          q.z = encode_plane(r.state, r.repetitions, (e0 + 2) / 64, ((e0 + 2) / 8) % 8, (e0 + 2) % 8);
          q.w = encode_plane(r.state, r.repetitions, (e0 + 3) / 64, ((e0 + 3) / 8) % 8, (e0 + 3) % 8);
          __stcs(reinterpret_cast<float4*>(o) + w, q);
        }
      } else {
        for (int w = t; w < ENC; w += TRAIN_THREADS) o[w] = encode_plane(r.state, r.repetitions, w / 64, (w / 8) % 8, w % 8);
      }
    }
    if (policies) {
      float* o = policies + i * (unsigned long long)SPB_CHESS_POLICY_SIZE;
      if (vec_pol) {
        const float4* q = reinterpret_cast<const float4*>(s_pol);
        for (int w = t; w < SPB_CHESS_POLICY_SIZE / 4; w += TRAIN_THREADS) __stcs(reinterpret_cast<float4*>(o) + w, q[w]);
      } else {
        for (int w = t; w < SPB_CHESS_POLICY_SIZE; w += TRAIN_THREADS) o[w] = s_pol[w];
      }
    }
    if (values && t == 0) values[i] = (float)r.outcome;
    __syncthreads();                                                   // s_rec / s_pol are reused by the next row
  }
}

}  // namespace chess
}  // namespace spb

using namespace spb;
namespace ch = spb::chess;

// The device buffers of one spb_chess_perft, freed when it returns: the frontier of every level (up to 2^23 positions of
// 80 bytes, its size known only once the level before it is counted, and read while the next level is written) and the
// output offsets of every level expanded.  They do not go in the engine's grow-only stage, which would keep them.
struct PerftBuffers {
  std::vector<void*> ptrs;
  ~PerftBuffers() { for (void* p : ptrs) cudaFree(p); }
  template <class T> T* alloc(size_t count) {
    void* p = nullptr;
    if (cudaMalloc(&p, count * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    ptrs.push_back(p);
    return static_cast<T*>(p);
  }
};

extern "C" {

int32_t spb_chess_start_position(spb_chess_state* out) {
  if (!out) return SPB_ERR_ARG;
  *out = ch::start_position();
  return SPB_OK;
}
int32_t spb_chess_move_channel(int32_t side, uint16_t move) { return ch::channel(side & 1, move); }
int32_t spb_chess_policy_index(int32_t side, uint16_t move) { return ch::policy_index(side & 1, move); }
uint16_t spb_chess_action(int32_t side, int32_t channel, int32_t row, int32_t col) {
  if (channel < 0 || channel >= 73 || row < 0 || row > 7 || col < 0 || col > 7) return ch::MOVE_NONE;
  return ch::action(side & 1, channel, row, col);
}

// The training tensors of recorded roots (ref: learner_concurrent.rs:126-146 over chess::State; host only).  The policy is
// computed exactly as spb_chess_root_policy computes it: f32 sum of the counts in child order, each count divided by it.
int32_t spb_chess_positions_to_training(const spb_chess_position* positions, size_t n, float* encodings, float* policies, float* values) {
  if (n && !positions) return SPB_ERR_ARG;
  for (size_t i = 0; i < n; ++i) {                                     // validate everything before writing anything
    const spb_chess_position& p = positions[i];
    if (p.n_moves == 0 || p.n_moves > SPB_CHESS_MAX_MOVES || p.state.side > 1) return SPB_ERR_ARG;
    for (uint32_t k = 0; k < p.n_moves; ++k) {
      const int idx = ch::policy_index(p.state.side, p.moves[k]);
      if (idx < 0 || idx >= SPB_CHESS_POLICY_SIZE) return SPB_ERR_ARG;
    }
  }
  for (size_t i = 0; i < n; ++i) {
    const spb_chess_position& p = positions[i];
    if (encodings) {
      float* o = encodings + i * (size_t)SPB_CHESS_PLANES * 64;
      for (int t = 0; t < SPB_CHESS_PLANES * 64; ++t) o[t] = ch::encode_plane(p.state, p.repetitions, t / 64, (t / 8) % 8, t % 8);
    }
    if (policies) {
      float* o = policies + i * (size_t)SPB_CHESS_POLICY_SIZE;
      std::memset(o, 0, sizeof(float) * SPB_CHESS_POLICY_SIZE);
      float sum = 0.0f;
      for (uint32_t k = 0; k < p.n_moves; ++k) sum += (float)p.visit_counts[k];
      for (uint32_t k = 0; k < p.n_moves; ++k) o[ch::policy_index(p.state.side, p.moves[k])] = (float)p.visit_counts[k] / sum;
    }
    if (values) values[i] = (float)p.outcome;
  }
  return SPB_OK;
}

int32_t spb_chess_positions_to_training_device(spb_chess_engine* e, const spb_chess_position* positions, size_t n_positions,
                                               const uint64_t* indices, size_t n, float* encodings, float* policies, float* values) {
  SPB_GUARD(e);
  SPB_ARG(e, indices || n <= n_positions, "n > n_positions without indices");
  if (n == 0) return SPB_OK;
  SPB_ARG(e, positions, "null positions");
  if (int32_t rc = e->check_device_pointers({{positions, "positions", 8}, {indices, "indices", 8}, {encodings, "encodings", 4},
                                              {policies, "policies", 4}, {values, "values", 4}}))
    return rc;
  const unsigned long long none = ~0ull;
  unsigned long long* d_bad = e->d_misc;                               // the engine's scratch word; every call ends synchronised
  const auto* idx = reinterpret_cast<const unsigned long long*>(indices);
  int sms = 0;
  SPB_CUDA(e, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
  SPB_CUDA(e, cudaMemsetAsync(d_bad, 0xFF, 8, e->stream));
  const unsigned long long check_blocks = std::min<unsigned long long>((n + 7) / 8, (unsigned long long)sms * 8);
  ch::k_chess_training_check<<<(unsigned)check_blocks, 256, 0, e->stream>>>(positions, n_positions, idx, n, d_bad);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  unsigned long long bad = none;
  SPB_CUDA(e, cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (bad != none) {
    e->set_error("malformed training row " + std::to_string(bad) +
                 (indices ? " (index out of range, or n_moves outside 1..256, side > 1 or a move outside the policy)"
                          : " (n_moves outside 1..256, side > 1 or a move outside the policy)"));
    return SPB_ERR_ARG;
  }
  const bool vec_enc = (reinterpret_cast<uintptr_t>(encodings) & 15) == 0, vec_pol = (reinterpret_cast<uintptr_t>(policies) & 15) == 0;
  const unsigned long long blocks = std::min<unsigned long long>(n, (unsigned long long)sms * 8);
  ch::k_chess_training<<<(unsigned)blocks, ch::TRAIN_THREADS, 0, e->stream>>>(positions, idx, n, encodings, policies, values, vec_enc, vec_pol);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_legal_moves(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, uint16_t* moves,
                              uint32_t* counts, uint16_t* policy_index, uint8_t* status, uint32_t* repetitions) {
  SPB_GUARD(e);
  if (n == 0) return SPB_OK;
  SPB_ARG(e, states, "null states");
  const size_t hist_bytes = (size_t)n * SPB_CHESS_MAX_HISTORY * 8, row_bytes = (size_t)n * SPB_CHESS_MAX_MOVES * 2;
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(ch::Pos)), o_hist = L.take(history ? hist_bytes : 0);
  const size_t o_moves = L.take(moves ? row_bytes : 0), o_pidx = L.take(policy_index ? row_bytes : 0);
  const size_t o_counts = L.take((size_t)n * 4), o_reps = L.take((size_t)n * 4), o_status = L.take(n);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  auto* d_states = e->d_at<ch::Pos>(o_states);
  auto* d_hist = history ? e->d_at<uint64_t>(o_hist) : nullptr;
  auto* d_moves = moves ? e->d_at<uint16_t>(o_moves) : nullptr;
  auto* d_pidx = policy_index ? e->d_at<uint16_t>(o_pidx) : nullptr;
  auto* d_counts = e->d_at<uint32_t>(o_counts);
  auto* d_reps = e->d_at<uint32_t>(o_reps);
  auto* d_status = e->d_at<uint8_t>(o_status);
  SPB_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(d_hist, history, hist_bytes, cudaMemcpyHostToDevice, e->stream));
  if (moves) SPB_CUDA(e, cudaMemsetAsync(d_moves, 0xFF, row_bytes, e->stream));
  if (policy_index) SPB_CUDA(e, cudaMemsetAsync(d_pidx, 0xFF, row_bytes, e->stream));
  ch::k_legal<<<(n + 63) / 64, 64, 0, e->stream>>>(d_states, d_hist, n, d_moves, d_counts, d_pidx, d_status, d_reps);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  if (moves) SPB_CUDA(e, cudaMemcpyAsync(moves, d_moves, row_bytes, cudaMemcpyDeviceToHost, e->stream));
  if (policy_index) SPB_CUDA(e, cudaMemcpyAsync(policy_index, d_pidx, row_bytes, cudaMemcpyDeviceToHost, e->stream));
  if (counts) SPB_CUDA(e, cudaMemcpyAsync(counts, d_counts, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (repetitions) SPB_CUDA(e, cudaMemcpyAsync(repetitions, d_reps, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (status) SPB_CUDA(e, cudaMemcpyAsync(status, d_status, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_next_states(spb_chess_engine* e, const spb_chess_state* states, uint64_t* history, const uint16_t* moves, uint32_t n,
                              spb_chess_state* out_states, int32_t* err) {
  SPB_GUARD(e);
  if (n == 0) return SPB_OK;
  SPB_ARG(e, states && moves && out_states && err, "null argument");
  const size_t hist_bytes = (size_t)n * SPB_CHESS_MAX_HISTORY * 8;
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(ch::Pos)), o_out = L.take((size_t)n * sizeof(ch::Pos)), o_hist = L.take(history ? hist_bytes : 0);
  const size_t o_moves = L.take((size_t)n * 2), o_err = L.take((size_t)n * 4);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  auto* d_states = e->d_at<ch::Pos>(o_states);
  auto* d_out = e->d_at<ch::Pos>(o_out);
  auto* d_hist = history ? e->d_at<uint64_t>(o_hist) : nullptr;
  auto* d_moves = e->d_at<uint16_t>(o_moves);
  auto* d_err = e->d_at<int32_t>(o_err);
  SPB_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(d_moves, moves, (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(d_hist, history, hist_bytes, cudaMemcpyHostToDevice, e->stream));
  ch::k_next<<<(n + 63) / 64, 64, 0, e->stream>>>(d_states, d_hist, d_moves, n, d_out, d_err);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  SPB_CUDA(e, cudaMemcpyAsync(out_states, d_out, (size_t)n * sizeof(ch::Pos), cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaMemcpyAsync(err, d_err, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(history, d_hist, hist_bytes, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_encode(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, float* out) {
  SPB_GUARD(e);
  if (n == 0) return SPB_OK;
  SPB_ARG(e, states && out, "null argument");
  const size_t hist_bytes = (size_t)n * SPB_CHESS_MAX_HISTORY * 8, out_bytes = (size_t)n * SPB_CHESS_PLANES * 64 * 4;
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(ch::Pos)), o_hist = L.take(history ? hist_bytes : 0), o_out = L.take(out_bytes);
  if (int32_t rc = e->ensure_stage(L.bytes, 0)) return rc;
  auto* d_states = e->d_at<ch::Pos>(o_states);
  auto* d_hist = history ? e->d_at<uint64_t>(o_hist) : nullptr;
  auto* d_out = e->d_at<float>(o_out);
  SPB_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) SPB_CUDA(e, cudaMemcpyAsync(d_hist, history, hist_bytes, cudaMemcpyHostToDevice, e->stream));
  ch::k_encode<<<n, 128, 0, e->stream>>>(d_states, d_hist, n, d_out);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  SPB_CUDA(e, cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_perft(spb_chess_engine* e, const spb_chess_state* state, uint32_t depth, uint64_t* nodes) {
  SPB_GUARD(e);
  SPB_ARG(e, state && nodes, "null argument");
  SPB_ARG(e, depth <= 8, "perft depth > 8");
  // Breadth first on the device while the frontier is too narrow to fill the GPU (or the rest too deep for one thread):
  // k_frontier_count gives every position its output offset, k_frontier_expand writes its children there.  Every
  // frontier position is then searched to the remaining depth by one device thread (k_perft).
  unsigned long long* d_total = e->d_misc;                             // the engine's scratch word; every call ends synchronised
  PerftBuffers buf;
  ch::Pos* d_f = buf.alloc<ch::Pos>(1);
  if (!d_f) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
  SPB_CUDA(e, cudaMemcpyAsync(d_f, state, sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  uint32_t n = 1, remaining = depth;
  while (remaining > 0 && (n < 4096 || remaining > (uint32_t)ch::PERFT_DEV_DEPTH)) {
    uint32_t* d_off = buf.alloc<uint32_t>(n);
    if (!d_off) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
    SPB_CUDA(e, cudaMemsetAsync(d_total, 0, 8, e->stream));
    ch::k_frontier_count<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, d_off, d_total);
    SPB_CUDA(e, cudaGetLastError());
    unsigned long long m = 0;
    SPB_CUDA(e, cudaMemcpyAsync(&m, d_total, 8, cudaMemcpyDeviceToHost, e->stream));
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
    e->launches += 1;
    if (m == 0) { *nodes = 0; return SPB_OK; }
    SPB_ARG(e, m <= (1ull << 23), "perft frontier too large");
    ch::Pos* d_next = buf.alloc<ch::Pos>(m);
    if (!d_next) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
    ch::k_frontier_expand<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, d_off, d_next);
    SPB_CUDA(e, cudaGetLastError());
    e->launches += 1;
    d_f = d_next;
    n = (uint32_t)m;
    --remaining;
  }
  SPB_CUDA(e, cudaMemsetAsync(d_total, 0, 8, e->stream));
  ch::k_perft<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, (int)remaining, d_total);
  SPB_CUDA(e, cudaGetLastError());
  ++e->launches;
  unsigned long long total = 0;
  SPB_CUDA(e, cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  *nodes = total;
  return SPB_OK;
}

}  // extern "C"
