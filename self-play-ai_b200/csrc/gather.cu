// gather.cu — the one exchange of the multi-GPU path and the learner hand-off (include/selfplay_b200.h).
//
// Games are sharded over GPUs (one engine = one rank); nothing is exchanged while searching.  At the end of a generation
// the finished trajectories go to the learner rank: the role of the replay-buffer push of the reference's workers
// (ref: src/learner_concurrent.rs:281-288).  NCCL has no gatherv: all-gather of the per-rank record counts, then grouped
// ncclSend / ncclRecv of the records into one device buffer on the learner rank; the learner orders them by
// (global game id, ply), so an R-rank generation is byte-identical to the same games played on one rank.  The Connect4 /
// tic-tac-toe engine (spb_position records) and the chess engine (spb_chess_position) run the same code, over the state
// the two share (HostEngine, host_engine.hpp).
// spb_positions_to_training builds the tensors the learners train on (ref: src/learner_concurrent.rs:126-146,
// src/learner.rs:162-182) from the compact records.
//
// NCCL is bound at run time (dlopen of libnccl.so.2): a host that never gathers does not need it, and a host process that
// has already loaded NCCL (PyTorch ships its own) shares that copy.
#include <dlfcn.h>
#include <nccl.h>

#include <mutex>

#include "chess_engine.hpp"
#include "engine.hpp"

using namespace spb;

namespace {

struct NcclApi {
  void* handle = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  std::string error;
};

NcclApi* nccl_api() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, [] {
    const char* names[] = {getenv("SPB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      if (!n || !*n) continue;
      api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (api.handle) break;
    }
    if (!api.handle) { api.error = std::string("cannot load NCCL (libnccl.so.2): ") + (dlerror() ? dlerror() : "not found"); return; }
    auto sym = [&](const char* n) { void* p = dlsym(api.handle, n); if (!p && api.error.empty()) api.error = std::string("NCCL symbol missing: ") + n; return p; };
    api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
    api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
    api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
    api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
    api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
    api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
    api.Send = reinterpret_cast<decltype(api.Send)>(sym("ncclSend"));
    api.Recv = reinterpret_cast<decltype(api.Recv)>(sym("ncclRecv"));
    api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
  });
  return &api;
}

#define SPB_NCCL(e, expr)                                                                                  \
  do {                                                                                                     \
    ncclResult_t _r = (expr);                                                                              \
    if (_r != ncclSuccess) {                                                                               \
      (e)->set_error(std::string(#expr) + ": " + (N->GetErrorString ? N->GetErrorString(_r) : "NCCL error")); \
      return SPB_ERR_CUDA;                                                                                 \
    }                                                                                                      \
  } while (0)

// Orders records by (global game id, ply): games finish in a nondeterministic order on the device and arrive rank by rank.
template <class Rec>
void sort_records(std::vector<Rec>& pos, std::vector<unsigned long long>& ids) {
  const size_t n = pos.size();
  const std::vector<size_t> order = record_order(pos, ids);
  std::vector<Rec> p2(n);
  std::vector<unsigned long long> i2(n);
  for (size_t i = 0; i < n; ++i) { p2[i] = pos[order[i]]; i2[i] = ids[order[i]]; }
  pos.swap(p2);
  ids.swap(i2);
}

// spb_comm_init / spb_chess_comm_init
template <class Trees, class Rec, class Move>
int32_t comm_init(HostEngine<Trees, Rec, Move>* e, const uint8_t* id, int32_t rank, int32_t world_size) {
  if (!id) return SPB_ERR_ARG;
  SPB_GUARD(e);
  SPB_ARG(e, world_size >= 1 && rank >= 0 && rank < world_size, "rank / world_size out of range");
  if (e->nccl_comm) { e->set_error(std::string("communicator already initialised (") + e->api + "comm_destroy first)"); return SPB_ERR_STATE; }
  NcclApi* N = nccl_api();
  if (!N->error.empty()) { e->set_error(N->error); return SPB_ERR_STATE; }
  ncclUniqueId u;
  std::memcpy(&u, id, sizeof u);
  ncclComm_t comm = nullptr;
  SPB_NCCL(e, N->CommInitRank(&comm, world_size, u, rank));
  e->nccl_comm = comm;
  e->comm_rank = rank;
  e->comm_world = world_size;
  return SPB_OK;
}

// spb_comm_destroy / spb_chess_comm_destroy (also called by the engines' destroy)
template <class Trees, class Rec, class Move>
int32_t comm_destroy(HostEngine<Trees, Rec, Move>* e) {
  if (!e) return SPB_ERR_ARG;
  if (e->nccl_comm) {
    cudaSetDevice(e->cfg.device);
    cudaStreamSynchronize(e->stream);
    NcclApi* N = nccl_api();
    if (N->CommDestroy) N->CommDestroy(static_cast<ncclComm_t>(e->nccl_comm));
    e->nccl_comm = nullptr;
    e->comm_rank = -1;
    e->comm_world = 0;
  }
  return SPB_OK;
}

// The checks both gather forms make before the collective.
template <class Trees, class Rec, class Move>
int32_t gather_ready(HostEngine<Trees, Rec, Move>* e, int32_t learner_rank) {
  if (!e->nccl_comm) { e->set_error(std::string("no communicator: call ") + e->api + "comm_init first"); return SPB_ERR_STATE; }
  SPB_ARG(e, learner_rank >= 0 && learner_rank < e->comm_world, "learner rank out of range");
  return SPB_OK;
}

// The collective of spb_gather_trajectories and its device form, over the engine's trajectory buffers P (record type Rec):
// all-gather of the per-rank record counts, then grouped send/recv of every rank's records into one device buffer of the
// learner rank, rank by rank (*d_pos / *d_ids, allocated here and freed by the caller; NULL when *total is 0).  The local
// output buffer is handed over and emptied.  *total = records on the learner rank, 0 on the others.  Everything runs on
// e->stream: the self-play steps that filled P ran there, and the chess search's second stream rejoins it before
// spb_chess_search returns.  Buffers not allocated yet (a chess engine that never played, P.out == NULL) take part with 0
// records and stay unallocated.  Returns with the stream synchronised.
template <class Trees, class Rec, class Move>
int32_t exchange(HostEngine<Trees, Rec, Move>* e, int32_t learner_rank, Rec** d_pos_out, unsigned long long** d_ids_out, size_t* total_out) {
  NcclApi* N = nccl_api();
  ncclComm_t comm = static_cast<ncclComm_t>(e->nccl_comm);
  const int rank = e->comm_rank, world = e->comm_world;
  const bool learner = rank == learner_rank;
  const auto& P = e->P;
  *d_pos_out = nullptr;
  *d_ids_out = nullptr;
  *total_out = 0;
  unsigned long long n_local = 0;
  if (P.out) {
    SPB_CUDA(e, cudaMemcpyAsync(&n_local, P.out_cursor, 8, cudaMemcpyDeviceToHost, e->stream));
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
    n_local = std::min<unsigned long long>(n_local, P.out_cap);
  }
  unsigned long long* d_counts = nullptr;
  SPB_CUDA(e, cudaMalloc((void**)&d_counts, (size_t)world * 8));
  std::vector<unsigned long long> counts((size_t)world, 0);
  cudaError_t ce = cudaMemcpyAsync(d_counts + rank, &n_local, 8, cudaMemcpyHostToDevice, e->stream);
  ncclResult_t nr = ce == cudaSuccess ? N->AllGather(d_counts + rank, d_counts, 1, ncclUint64, comm, e->stream) : ncclSuccess;
  if (ce == cudaSuccess && nr == ncclSuccess) ce = cudaMemcpyAsync(counts.data(), d_counts, (size_t)world * 8, cudaMemcpyDeviceToHost, e->stream);
  if (ce == cudaSuccess && nr == ncclSuccess) ce = cudaStreamSynchronize(e->stream);
  cudaFree(d_counts);
  if (nr != ncclSuccess) { e->set_error(std::string("ncclAllGather: ") + N->GetErrorString(nr)); return SPB_ERR_CUDA; }
  if (ce != cudaSuccess) { e->set_error(std::string("gather counts: ") + cudaGetErrorString(ce)); return SPB_ERR_CUDA; }
  size_t total = 0;
  std::vector<size_t> off((size_t)world, 0);
  for (int r = 0; r < world; ++r) { off[r] = total; total += (size_t)counts[r]; }

  Rec* d_pos = nullptr;
  unsigned long long* d_ids = nullptr;
  if (learner && total) {
    ce = cudaMalloc((void**)&d_pos, total * sizeof(Rec));
    if (ce == cudaSuccess) ce = cudaMalloc((void**)&d_ids, total * 8);
    if (ce != cudaSuccess) { if (d_pos) cudaFree(d_pos); e->set_error("gather: out of device memory"); return SPB_ERR_NOMEM; }
  }
  nr = N->GroupStart();
  if (learner) {
    for (int r = 0; r < world && nr == ncclSuccess; ++r) {
      if (r == rank || counts[r] == 0) continue;
      nr = N->Recv(d_pos + off[r], (size_t)counts[r] * sizeof(Rec), ncclUint8, r, comm, e->stream);
      if (nr == ncclSuccess) nr = N->Recv(d_ids + off[r], (size_t)counts[r] * 8, ncclUint8, r, comm, e->stream);
    }
  } else if (n_local) {
    nr = N->Send(P.out, (size_t)n_local * sizeof(Rec), ncclUint8, learner_rank, comm, e->stream);
    if (nr == ncclSuccess) nr = N->Send(P.out_game, (size_t)n_local * 8, ncclUint8, learner_rank, comm, e->stream);
  }
  ncclResult_t nr2 = N->GroupEnd();
  if (nr == ncclSuccess) nr = nr2;
  ce = cudaSuccess;
  if (learner && n_local) {
    ce = cudaMemcpyAsync(d_pos + off[rank], P.out, (size_t)n_local * sizeof(Rec), cudaMemcpyDeviceToDevice, e->stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(d_ids + off[rank], P.out_game, (size_t)n_local * 8, cudaMemcpyDeviceToDevice, e->stream);
  }
  if (ce == cudaSuccess && P.out) ce = cudaMemsetAsync(P.out_cursor, 0, 8, e->stream);   // the local buffer has been handed over
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
  if (nr != ncclSuccess || ce != cudaSuccess) {
    if (d_pos) cudaFree(d_pos);
    if (d_ids) cudaFree(d_ids);
    e->set_error(nr != ncclSuccess ? std::string("gather send/recv: ") + N->GetErrorString(nr) : std::string("gather: ") + cudaGetErrorString(ce));
    return SPB_ERR_CUDA;
  }
  *d_pos_out = d_pos;
  *d_ids_out = d_ids;
  *total_out = learner ? total : 0;
  return SPB_OK;
}

// spb_gather_trajectories / spb_chess_gather_trajectories: the gathered records are ordered on the host and staged there
// until a call delivers them.
template <class Trees, class Rec, class Move>
int32_t gather_trajectories(HostEngine<Trees, Rec, Move>* e, int32_t learner_rank, Rec* buf, size_t capacity, size_t* written,
                            uint64_t* game_ids) {
  if (!written) return SPB_ERR_ARG;
  SPB_GUARD(e);
  if (int32_t rc = gather_ready(e, learner_rank)) return rc;
  if (e->gather_dpos) {
    e->set_error(std::string("the gathered records are staged in device memory: call ") + e->api + "gather_trajectories_device");
    return SPB_ERR_STATE;
  }
  const bool learner = e->comm_rank == learner_rank;

  if (!e->gather_pending) {
    Rec* d_pos = nullptr;
    unsigned long long* d_ids = nullptr;
    size_t total = 0;
    if (int32_t rc = exchange(e, learner_rank, &d_pos, &d_ids, &total)) return rc;
    e->gather_pos.assign(total, Rec{});
    e->gather_ids.assign(total, 0ull);
    cudaError_t ce = cudaSuccess;
    if (total) {
      ce = cudaMemcpyAsync(e->gather_pos.data(), d_pos, total * sizeof(Rec), cudaMemcpyDeviceToHost, e->stream);
      if (ce == cudaSuccess) ce = cudaMemcpyAsync(e->gather_ids.data(), d_ids, total * 8, cudaMemcpyDeviceToHost, e->stream);
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(e->stream);
    if (d_pos) cudaFree(d_pos);
    if (d_ids) cudaFree(d_ids);
    if (ce != cudaSuccess) { e->set_error(std::string("gather: ") + cudaGetErrorString(ce)); return SPB_ERR_CUDA; }
    if (learner) sort_records(e->gather_pos, e->gather_ids);
    e->gather_pending = true;
  }
  // ---- hand the gathered records to the caller (learner rank; the others hold none) ---------------------------------
  const size_t n = e->gather_pos.size();
  *written = n;
  if (learner && n && (!buf || capacity < n)) return SPB_OK;       // size query: the records stay staged for the next call
  if (n) {
    std::memcpy(buf, e->gather_pos.data(), n * sizeof(Rec));
    if (game_ids) std::memcpy(game_ids, e->gather_ids.data(), n * 8);
  }
  e->gather_pos.clear();
  e->gather_ids.clear();
  e->gather_pending = false;
  return SPB_OK;
}

// spb_gather_trajectories_device / spb_chess_gather_trajectories_device: the gathered records stay in device memory, in
// arrival order, until a call orders them into the caller's device buffers (order_records, records.cu).
template <class Trees, class Rec, class Move>
int32_t gather_trajectories_device(HostEngine<Trees, Rec, Move>* e, int32_t learner_rank, Rec* buf_dev, size_t capacity, size_t* written,
                                   uint64_t* game_ids_dev) {
  if (!written) return SPB_ERR_ARG;
  SPB_GUARD(e);
  if (int32_t rc = gather_ready(e, learner_rank)) return rc;
  if (e->gather_pending) {
    e->set_error(std::string("the gathered records are staged in host memory: call ") + e->api + "gather_trajectories");
    return SPB_ERR_STATE;
  }
  if (!e->gather_dpos) {
    if (int32_t rc = exchange(e, learner_rank, &e->gather_dpos, &e->gather_dids, &e->gather_dn)) return rc;
  }
  const size_t n = e->gather_dn;
  *written = n;
  if (n && (!buf_dev || capacity < n)) return SPB_OK;             // size query: the records stay staged for the next call
  // the caller's pointers are checked by order_into, after the collective: a bad one leaves the records staged and has
  // not kept the other ranks waiting
  if (n)
    if (int32_t rc = e->order_into(e->gather_dpos, e->gather_dids, n, buf_dev, game_ids_dev)) return rc;
  if (e->gather_dpos) cudaFree(e->gather_dpos);
  if (e->gather_dids) cudaFree(e->gather_dids);
  e->gather_dpos = nullptr;
  e->gather_dids = nullptr;
  e->gather_dn = 0;
  return SPB_OK;
}

}  // namespace

extern "C" {

int32_t spb_comm_unique_id(uint8_t* id) {
  if (!id) return SPB_ERR_ARG;
  NcclApi* N = nccl_api();
  if (!N->error.empty()) { g_create_error = N->error; return SPB_ERR_STATE; }
  static_assert(sizeof(ncclUniqueId) == SPB_COMM_ID_BYTES, "ncclUniqueId size");
  ncclUniqueId u;
  if (N->GetUniqueId(&u) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return SPB_ERR_CUDA; }
  std::memcpy(id, &u, sizeof u);
  return SPB_OK;
}

int32_t spb_comm_init(spb_engine* e, const uint8_t* id, int32_t rank, int32_t world_size) { return comm_init(e, id, rank, world_size); }
int32_t spb_comm_destroy(spb_engine* e) { return comm_destroy(e); }
int32_t spb_gather_trajectories(spb_engine* e, int32_t learner_rank, spb_position* buf, size_t capacity, size_t* written,
                                uint64_t* game_ids) {
  return gather_trajectories(e, learner_rank, buf, capacity, written, game_ids);
}
int32_t spb_gather_trajectories_device(spb_engine* e, int32_t learner_rank, spb_position* buf_dev, size_t capacity, size_t* written,
                                       uint64_t* game_ids_dev) {
  return gather_trajectories_device(e, learner_rank, buf_dev, capacity, written, game_ids_dev);
}

int32_t spb_chess_comm_init(spb_chess_engine* e, const uint8_t* id, int32_t rank, int32_t world_size) { return comm_init(e, id, rank, world_size); }
int32_t spb_chess_comm_destroy(spb_chess_engine* e) { return comm_destroy(e); }
int32_t spb_chess_gather_trajectories(spb_chess_engine* e, int32_t learner_rank, spb_chess_position* buf, size_t capacity, size_t* written,
                                      uint64_t* game_ids) {
  return gather_trajectories(e, learner_rank, buf, capacity, written, game_ids);
}
int32_t spb_chess_gather_trajectories_device(spb_chess_engine* e, int32_t learner_rank, spb_chess_position* buf_dev, size_t capacity,
                                             size_t* written, uint64_t* game_ids_dev) {
  return gather_trajectories_device(e, learner_rank, buf_dev, capacity, written, game_ids_dev);
}

// ref: learner_concurrent.rs:126-146 / learner.rs:162-182 — the (N,3,R,C) / (N,A) / (N,1) training tensors.
//   encodings : get_encoding of the recorded root state (connect_four.rs:242-259 / tictactoe.rs:199-216): plane 0 = stones
//               of the side to move, 1 = the opponent's, 2 = empty cells; [plane][row][col], Connect4 row 0 = bottom
//   policies  : the search's first result, root child visit counts scattered by action and divided by their sum
//               (mcts.rs:315-328; f32 sum of integers, f32 divide)
//   values    : +-1 / 0 from the position's side to move (learner_concurrent.rs:214-226)
int32_t spb_positions_to_training(int32_t game, const spb_position* positions, size_t n, float* encodings, float* policies, float* values) {
  if (game != SPB_GAME_CONNECT4 && game != SPB_GAME_TICTACTOE) return SPB_ERR_ARG;
  if (n && !positions) return SPB_ERR_ARG;
  const bool c4 = game == SPB_GAME_CONNECT4;
  const int R = c4 ? 6 : 3, Cc = c4 ? 7 : 3, A = c4 ? 7 : 9, E = 3 * R * Cc;
  for (size_t i = 0; i < n; ++i) {
    const spb_position& p = positions[i];
    if (encodings) {
      const uint64_t mine = p.stones[p.current_player & 1], opp = p.stones[(p.current_player & 1) ^ 1];
      float* o = encodings + i * (size_t)E;
      for (int r = 0; r < R; ++r)
        for (int c = 0; c < Cc; ++c) {
          const int bit = c4 ? c * 7 + r : r * 3 + c;
          const uint32_t m = (uint32_t)(mine >> bit) & 1u, q = (uint32_t)(opp >> bit) & 1u;
          o[(0 * R + r) * Cc + c] = m ? 1.0f : 0.0f;
          o[(1 * R + r) * Cc + c] = q ? 1.0f : 0.0f;
          o[(2 * R + r) * Cc + c] = (m | q) ? 0.0f : 1.0f;
        }
    }
    if (policies) {
      float s = 0.0f;
      for (int a = 0; a < A; ++a) s += (float)p.visit_counts[a];     // integers < 2^24: exact in any summation order
      for (int a = 0; a < A; ++a) policies[i * (size_t)A + a] = (float)p.visit_counts[a] / s;
    }
    if (values) values[i] = (float)p.outcome;
  }
  return SPB_OK;
}

// The same tensors built on the device from records in device memory (launch_training_tensors, records.cu), for the
// engine's game; row i from positions[indices ? indices[i] : i].
int32_t spb_positions_to_training_device(spb_engine* e, const spb_position* positions, size_t n_positions, const uint64_t* indices, size_t n,
                                         float* encodings, float* policies, float* values) {
  SPB_GUARD(e);
  SPB_ARG(e, indices || n <= n_positions, "n > n_positions without indices");
  if (n == 0) return SPB_OK;
  SPB_ARG(e, positions, "null positions");
  if (int32_t rc = e->check_device_pointers({{positions, "positions", 8}, {indices, "indices", 8}, {encodings, "encodings", 4},
                                              {policies, "policies", 4}, {values, "values", 4}}))
    return rc;
  const auto* idx = reinterpret_cast<const unsigned long long*>(indices);
  int sms = 0;
  SPB_CUDA(e, cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->cfg.device));
  if (idx) {
    const unsigned long long none = ~0ull;
    unsigned long long bad = none;
    unsigned long long* d_bad = e->d_misc;                             // the engine's scratch word; every call ends synchronised
    SPB_CUDA(e, cudaMemsetAsync(d_bad, 0xFF, 8, e->stream));
    SPB_CUDA(e, launch_index_check(idx, n, n_positions, d_bad, sms, e->stream));
    ++e->launches;
    SPB_CUDA(e, cudaMemcpyAsync(&bad, d_bad, 8, cudaMemcpyDeviceToHost, e->stream));
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
    if (bad != none) { e->set_error("training row " + std::to_string(bad) + ": index out of range"); return SPB_ERR_ARG; }
  }
  SPB_CUDA(e, launch_training_tensors(e->cfg.game, positions, idx, n, encodings, policies, values, sms, e->stream));
  ++e->launches;
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

}  // extern "C"
