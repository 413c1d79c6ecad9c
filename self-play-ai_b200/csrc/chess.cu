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

}  // namespace chess
}  // namespace spb

using namespace spb;
namespace ch = spb::chess;

using spb::chess::Scratch;

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

int32_t spb_chess_legal_moves(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, uint16_t* moves,
                              uint32_t* counts, uint16_t* policy_index, uint8_t* status, uint32_t* repetitions) {
  CH_GUARD(e);
  if (n == 0) return SPB_OK;
  if (!states) { e->set_error("null states"); return SPB_ERR_ARG; }
  Scratch sc;
  auto* d_states = sc.alloc<ch::Pos>(n);
  auto* d_hist = history ? sc.alloc<uint64_t>((size_t)n * SPB_CHESS_MAX_HISTORY) : nullptr;
  auto* d_moves = moves ? sc.alloc<uint16_t>((size_t)n * SPB_CHESS_MAX_MOVES) : nullptr;
  auto* d_pidx = policy_index ? sc.alloc<uint16_t>((size_t)n * SPB_CHESS_MAX_MOVES) : nullptr;
  auto* d_counts = sc.alloc<uint32_t>(n);
  auto* d_reps = sc.alloc<uint32_t>(n);
  auto* d_status = sc.alloc<uint8_t>(n);
  if (!d_states || (history && !d_hist) || (moves && !d_moves) || (policy_index && !d_pidx) || !d_counts || !d_reps || !d_status) {
    e->set_error("chess: out of device memory");
    return SPB_ERR_NOMEM;
  }
  CH_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) CH_CUDA(e, cudaMemcpyAsync(d_hist, history, (size_t)n * SPB_CHESS_MAX_HISTORY * 8, cudaMemcpyHostToDevice, e->stream));
  if (d_moves) CH_CUDA(e, cudaMemsetAsync(d_moves, 0xFF, (size_t)n * SPB_CHESS_MAX_MOVES * 2, e->stream));
  if (d_pidx) CH_CUDA(e, cudaMemsetAsync(d_pidx, 0xFF, (size_t)n * SPB_CHESS_MAX_MOVES * 2, e->stream));
  ch::k_legal<<<(n + 63) / 64, 64, 0, e->stream>>>(d_states, d_hist, n, d_moves, d_counts, d_pidx, d_status, d_reps);
  CH_CUDA(e, cudaGetLastError());
  ++e->launches;
  if (moves) CH_CUDA(e, cudaMemcpyAsync(moves, d_moves, (size_t)n * SPB_CHESS_MAX_MOVES * 2, cudaMemcpyDeviceToHost, e->stream));
  if (policy_index) CH_CUDA(e, cudaMemcpyAsync(policy_index, d_pidx, (size_t)n * SPB_CHESS_MAX_MOVES * 2, cudaMemcpyDeviceToHost, e->stream));
  if (counts) CH_CUDA(e, cudaMemcpyAsync(counts, d_counts, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (repetitions) CH_CUDA(e, cudaMemcpyAsync(repetitions, d_reps, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (status) CH_CUDA(e, cudaMemcpyAsync(status, d_status, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
  CH_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_next_states(spb_chess_engine* e, const spb_chess_state* states, uint64_t* history, const uint16_t* moves, uint32_t n,
                              spb_chess_state* out_states, int32_t* err) {
  CH_GUARD(e);
  if (n == 0) return SPB_OK;
  if (!states || !moves || !out_states || !err) { e->set_error("null argument"); return SPB_ERR_ARG; }
  Scratch sc;
  auto* d_states = sc.alloc<ch::Pos>(n);
  auto* d_out = sc.alloc<ch::Pos>(n);
  auto* d_hist = history ? sc.alloc<uint64_t>((size_t)n * SPB_CHESS_MAX_HISTORY) : nullptr;
  auto* d_moves = sc.alloc<uint16_t>(n);
  auto* d_err = sc.alloc<int32_t>(n);
  if (!d_states || !d_out || (history && !d_hist) || !d_moves || !d_err) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
  CH_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  CH_CUDA(e, cudaMemcpyAsync(d_moves, moves, (size_t)n * 2, cudaMemcpyHostToDevice, e->stream));
  if (history) CH_CUDA(e, cudaMemcpyAsync(d_hist, history, (size_t)n * SPB_CHESS_MAX_HISTORY * 8, cudaMemcpyHostToDevice, e->stream));
  ch::k_next<<<(n + 63) / 64, 64, 0, e->stream>>>(d_states, d_hist, d_moves, n, d_out, d_err);
  CH_CUDA(e, cudaGetLastError());
  ++e->launches;
  CH_CUDA(e, cudaMemcpyAsync(out_states, d_out, (size_t)n * sizeof(ch::Pos), cudaMemcpyDeviceToHost, e->stream));
  CH_CUDA(e, cudaMemcpyAsync(err, d_err, (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  if (history) CH_CUDA(e, cudaMemcpyAsync(history, d_hist, (size_t)n * SPB_CHESS_MAX_HISTORY * 8, cudaMemcpyDeviceToHost, e->stream));
  CH_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_encode(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, float* out) {
  CH_GUARD(e);
  if (n == 0) return SPB_OK;
  if (!states || !out) { e->set_error("null argument"); return SPB_ERR_ARG; }
  Scratch sc;
  auto* d_states = sc.alloc<ch::Pos>(n);
  auto* d_hist = history ? sc.alloc<uint64_t>((size_t)n * SPB_CHESS_MAX_HISTORY) : nullptr;
  auto* d_out = sc.alloc<float>((size_t)n * SPB_CHESS_PLANES * 64);
  if (!d_states || (history && !d_hist) || !d_out) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
  CH_CUDA(e, cudaMemcpyAsync(d_states, states, (size_t)n * sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  if (history) CH_CUDA(e, cudaMemcpyAsync(d_hist, history, (size_t)n * SPB_CHESS_MAX_HISTORY * 8, cudaMemcpyHostToDevice, e->stream));
  ch::k_encode<<<n, 128, 0, e->stream>>>(d_states, d_hist, n, d_out);
  CH_CUDA(e, cudaGetLastError());
  ++e->launches;
  CH_CUDA(e, cudaMemcpyAsync(out, d_out, (size_t)n * SPB_CHESS_PLANES * 64 * 4, cudaMemcpyDeviceToHost, e->stream));
  CH_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_chess_perft(spb_chess_engine* e, const spb_chess_state* state, uint32_t depth, uint64_t* nodes) {
  CH_GUARD(e);
  if (!state || !nodes) { e->set_error("null argument"); return SPB_ERR_ARG; }
  if (depth > 8) { e->set_error("perft depth > 8"); return SPB_ERR_ARG; }
  // Breadth first on the device while the frontier is too narrow to fill the GPU (or the rest too deep for one thread):
  // k_frontier_count gives every position its output offset, k_frontier_expand writes its children there.  Every
  // frontier position is then searched to the remaining depth by one device thread (k_perft).
  Scratch sc;
  auto* d_total = sc.alloc<unsigned long long>(1);
  ch::Pos* d_f = nullptr;
  if (cudaMalloc(&d_f, sizeof(ch::Pos)) != cudaSuccess || !d_total) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
  struct Free { ch::Pos*& p; ~Free() { cudaFree(p); } } free_f{d_f};
  CH_CUDA(e, cudaMemcpyAsync(d_f, state, sizeof(ch::Pos), cudaMemcpyHostToDevice, e->stream));
  uint32_t n = 1, remaining = depth;
  while (remaining > 0 && (n < 4096 || remaining > (uint32_t)ch::PERFT_DEV_DEPTH)) {
    uint32_t* d_off = nullptr;
    if (cudaMalloc(&d_off, (size_t)n * 4) != cudaSuccess) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
    struct FreeOff { uint32_t* p; ~FreeOff() { cudaFree(p); } } free_off{d_off};
    CH_CUDA(e, cudaMemsetAsync(d_total, 0, 8, e->stream));
    ch::k_frontier_count<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, d_off, d_total);
    CH_CUDA(e, cudaGetLastError());
    unsigned long long m = 0;
    CH_CUDA(e, cudaMemcpyAsync(&m, d_total, 8, cudaMemcpyDeviceToHost, e->stream));
    CH_CUDA(e, cudaStreamSynchronize(e->stream));
    e->launches += 1;
    if (m == 0) { *nodes = 0; return SPB_OK; }
    if (m > (1ull << 23)) { e->set_error("perft frontier too large"); return SPB_ERR_ARG; }
    ch::Pos* d_next = nullptr;
    if (cudaMalloc(&d_next, (size_t)m * sizeof(ch::Pos)) != cudaSuccess) { e->set_error("chess: out of device memory"); return SPB_ERR_NOMEM; }
    ch::k_frontier_expand<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, d_off, d_next);
    const cudaError_t err = cudaGetLastError();
    cudaStreamSynchronize(e->stream);
    cudaFree(d_f);
    d_f = d_next;
    CH_CUDA(e, err);
    e->launches += 1;
    n = (uint32_t)m;
    --remaining;
  }
  CH_CUDA(e, cudaMemsetAsync(d_total, 0, 8, e->stream));
  ch::k_perft<<<(n + 63) / 64, 64, 0, e->stream>>>(d_f, n, (int)remaining, d_total);
  CH_CUDA(e, cudaGetLastError());
  ++e->launches;
  unsigned long long total = 0;
  CH_CUDA(e, cudaMemcpyAsync(&total, d_total, 8, cudaMemcpyDeviceToHost, e->stream));
  CH_CUDA(e, cudaStreamSynchronize(e->stream));
  *nodes = total;
  return SPB_OK;
}

}  // extern "C"
