// host_engine.hpp — what the two host engines behind the C ABI (include/selfplay_b200.h) have in common.  spb_engine
// (engine.hpp: Connect4 / tic-tac-toe) and spb_chess_engine (chess_engine.hpp) both derive from HostEngine: configuration,
// last error, stream and timing events, device allocations, result scratch, self-play trajectory buffers, the NCCL gather
// state (gather.cu) and the root-noise state, with their lifecycle and the bodies of the entry points both ABIs share.
#pragma once
#include <algorithm>
#include <cfloat>
#include <cstring>
#include <initializer_list>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "records.cuh"
#include "trajectory.cuh"
#include "tree.cuh"

// Error handling of the host code.  `e` is the engine (`this` inside its methods); each returns the entry point's status.
#define SPB_CUDA(e, expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      (e)->set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                      \
      return SPB_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)
// every entry point that takes an engine: NULL is SPB_ERR_ARG, then the engine's device is made current
#define SPB_GUARD(e)                                                                           \
  if (!(e)) return SPB_ERR_ARG;                                                                \
  if (cudaSetDevice((e)->cfg.device) != cudaSuccess) { (e)->set_error("cudaSetDevice failed"); return SPB_ERR_CUDA; }
#define SPB_ARG(e, cond, msg) \
  if (!(cond)) { (e)->set_error(msg); return SPB_ERR_ARG; }

extern thread_local std::string g_create_error;   // text of the last failure that had no engine to attach to (spb_last_error(NULL))

namespace spb {

// Byte offsets of an entry point's arrays in the engine's stage: take(n) reserves the next n bytes, 16-byte aligned, and
// returns their offset; `bytes` is what the stage must hold.
struct StageLayout {
  size_t bytes = 0;
  size_t take(size_t n) { const size_t off = bytes; bytes = (bytes + n + 15) & ~(size_t)15; return off; }
};

// Trees: the device trees (Trees / chess::CTrees); Rec: the trajectory record; Move: the move of a root child as the
// whole-batch root query reports it (action index / chess move).
template <class Trees, class Rec, class Move>
struct HostEngine {
  explicit HostEngine(const char* api_) : api(api_) {}

  const char* api;   // "spb_" / "spb_chess_": the prefix of this engine's entry points, for messages
  spb_config cfg{};
  std::string err;
  Trees T{};
  // self-play trajectories.  parked[g] = 1 | how the game ended << 1 (engine-specific, see the self-play kernels)
  Trajectories<Rec> P{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  std::vector<void*> allocs;   // device allocations freed by release()
  uint64_t launches = 0;
  float last_search_ms = 0.f;
  // device scratch for results of whole-batch queries
  Move* d_rc_moves = nullptr; uint32_t* d_rc_counts = nullptr; uint32_t* d_rc_ids = nullptr; uint32_t* d_rc_n = nullptr;
  unsigned long long* d_misc = nullptr;   // [4] scratch u64
  // multi-GPU trajectory gather (gather.cu): NCCL communicator of this engine's rank, records staged on the learner rank
  void* nccl_comm = nullptr;
  int comm_rank = -1, comm_world = 0;
  bool gather_pending = false;
  std::vector<Rec> gather_pos;
  std::vector<unsigned long long> gather_ids;
  // a gather staged by the device form (gather_trajectories_device): the learner's records in arrival order, not yet
  // ordered, until a call delivers them; freed by that call or by release()
  Rec* gather_dpos = nullptr;
  unsigned long long* gather_dids = nullptr;
  size_t gather_dn = 0;
  // EXTENSION: Dirichlet noise at the root (set_root_noise).  The buffers are allocated by the first call that turns the
  // noise on (an engine that never enables it keeps its footprint); T.root_noise points at them while it is on.
  float* d_noise_eta = nullptr;
  uint32_t* d_noise_n = nullptr;
  float noise_alpha = 0.0f;
  unsigned long long noise_seed = 0;
  // Staging of the inputs and outputs of an entry point, grow-only: device bytes and pinned host bytes.  Every entry point
  // that uses them synchronises its stream before it returns: the next call reuses them, and a grow frees the old buffer.
  void* d_stage = nullptr; size_t d_stage_bytes = 0;
  void* h_stage = nullptr; size_t h_stage_bytes = 0;

  void set_error(const std::string& s) { err = s; }

  // At least d_bytes of device and h_bytes of pinned host stage (0: a call that copies straight between the caller's
  // memory and the device needs no pinned bytes).
  int32_t ensure_stage(size_t d_bytes, size_t h_bytes) {
    const auto grow = [this](void** p, size_t* have, size_t want, bool pinned) -> int32_t {
      if (want <= *have) return SPB_OK;
      if (*p) pinned ? cudaFreeHost(*p) : cudaFree(*p);
      *p = nullptr; *have = 0;
      const size_t nb = std::max(want, (size_t)1 << 20);
      const cudaError_t ce = pinned ? cudaMallocHost(p, nb) : cudaMalloc(p, nb);
      if (ce != cudaSuccess) {
        cudaGetLastError();                                              // an allocation failure is not sticky: clear it
        set_error(std::string("cannot grow the ") + (pinned ? "pinned" : "device") + " stage to " + std::to_string(nb) + " bytes: " + cudaGetErrorString(ce));
        return SPB_ERR_NOMEM;
      }
      *have = nb;
      return SPB_OK;
    };
    const int32_t rc = grow(&d_stage, &d_stage_bytes, d_bytes, false);
    return rc ? rc : grow(&h_stage, &h_stage_bytes, h_bytes, true);
  }
  template <class T_> T_* d_at(size_t off) const { return reinterpret_cast<T_*>(static_cast<char*>(d_stage) + off); }
  template <class T_> T_* h_at(size_t off) const { return reinterpret_cast<T_*>(static_cast<char*>(h_stage) + off); }

  template <class T_> int32_t dalloc(T_** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T_));
    if (e != cudaSuccess) { set_error(std::string("cudaMalloc: ") + cudaGetErrorString(e)); return SPB_ERR_NOMEM; }
    allocs.push_back(q);
    *p = static_cast<T_*>(q);
    return SPB_OK;
  }

  // The spb_config checks both engines make.  nullptr: none failed.
  static const char* config_error(const spb_config& c) {
    if (c.abi_version != SPB_ABI_VERSION) return "abi_version mismatch";
    if (c.evaluator < SPB_EVAL_NET || c.evaluator > SPB_EVAL_UNIFORM) return "unknown evaluator";
    if (!(c.c == c.c)) return "c is NaN";
    return nullptr;
  }

  // spb_create / spb_chess_create once the config passed its checks: the engine's init() opens the device and allocates;
  // a failure releases what it made and leaves its text for spb_last_error(NULL).
  template <class Eng> static int32_t create(const spb_config& c, Eng** out) {
    Eng* e = new (std::nothrow) Eng();
    if (!e) { g_create_error = "out of host memory"; return SPB_ERR_NOMEM; }
    e->cfg = c;
    const int32_t rc = e->init();
    if (rc) {
      g_create_error = e->err;
      e->release();
      delete e;
      return rc;
    }
    *out = e;
    return SPB_OK;
  }

  // The device of cfg (present, in range, sm_100), the engine's stream and its timing events.
  int32_t open_device() {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { set_error("no CUDA device (this library has no CPU fallback)"); return SPB_ERR_CUDA; }
    if (cfg.device < 0 || cfg.device >= ndev) { set_error("device ordinal out of range"); return SPB_ERR_ARG; }
    SPB_CUDA(this, cudaSetDevice(cfg.device));
    cudaDeviceProp prop;
    SPB_CUDA(this, cudaGetDeviceProperties(&prop, cfg.device));
    if (prop.major != 10) { set_error("device is not sm_100 (B200); this library is built for sm_100a only"); return SPB_ERR_CUDA; }
    SPB_CUDA(this, cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    SPB_CUDA(this, cudaEventCreate(&ev0));
    SPB_CUDA(this, cudaEventCreate(&ev1));
    return SPB_OK;
  }

  // Waits for the stream, then frees what open_device(), dalloc() and ensure_stage() made (also of an engine whose creation
  // failed).
  void release() {
    cudaSetDevice(cfg.device);
    if (stream) cudaStreamSynchronize(stream);
    for (void* p : allocs) cudaFree(p);
    allocs.clear();
    if (d_stage) cudaFree(d_stage);
    if (h_stage) cudaFreeHost(h_stage);
    if (gather_dpos) cudaFree(gather_dpos);
    if (gather_dids) cudaFree(gather_dids);
    if (ev0) cudaEventDestroy(ev0);
    if (ev1) cudaEventDestroy(ev1);
    if (stream) cudaStreamDestroy(stream);
  }

  // The trajectory buffers of the self-play step for games of up to max_ply plies.  A failure frees what this call
  // allocated and leaves the engine as it was.
  int32_t alloc_trajectories(uint32_t max_ply) {
    const size_t G = T.G;
    Trajectories<Rec> Q{};
    Q.max_ply = max_ply;
    Q.out_cap = (uint32_t)std::min<size_t>(G * max_ply * 4, (size_t)1 << 26);
    if (cfg.trajectory_capacity) Q.out_cap = std::max<uint32_t>(cfg.trajectory_capacity, max_ply);   // a whole game always fits
    Q.id_stride = cfg.game_id_stride ? cfg.game_id_stride : (unsigned long long)G;
    const size_t n_allocs = allocs.size();
    int32_t rc = SPB_OK;
    if (!rc) rc = dalloc(&Q.hist, G * max_ply);
    if (!rc) rc = dalloc(&Q.hist_len, G);
    if (!rc) rc = dalloc(&Q.parked, G);
    if (!rc) rc = dalloc(&Q.game_id, G);
    if (!rc) rc = dalloc(&Q.out, (size_t)Q.out_cap);
    if (!rc) rc = dalloc(&Q.out_game, (size_t)Q.out_cap);
    if (!rc) rc = dalloc(&Q.out_cursor, 1);
    if (!rc) rc = dalloc(&Q.finished, 1);
    std::vector<unsigned long long> ids(G);
    for (size_t i = 0; i < G; ++i) ids[i] = (unsigned long long)cfg.game_id_base + i;
    cudaError_t ce = rc ? cudaErrorMemoryAllocation : cudaSuccess;
    if (ce == cudaSuccess) ce = cudaMemsetAsync(Q.hist_len, 0, G * 4, stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(Q.parked, 0, G, stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(Q.out_cursor, 0, 8, stream);
    if (ce == cudaSuccess) ce = cudaMemsetAsync(Q.finished, 0, 4, stream);
    if (ce == cudaSuccess) ce = cudaMemcpyAsync(Q.game_id, ids.data(), G * 8, cudaMemcpyHostToDevice, stream);
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(stream);
    if (ce != cudaSuccess) {
      for (size_t i = n_allocs; i < allocs.size(); ++i) cudaFree(allocs[i]);
      allocs.resize(n_allocs);
      cudaGetLastError();                                                // an allocation failure is not sticky: clear it
      set_error("self-play: cannot set up the trajectory buffers (" + std::to_string(G * max_ply) + " + " + std::to_string(Q.out_cap) +
                " records of " + std::to_string(sizeof(Rec)) + " bytes): " + cudaGetErrorString(ce));
      return rc ? rc : SPB_ERR_CUDA;
    }
    P = Q;
    return SPB_OK;
  }

  // Reads and clears the error word of the kernels (ErrorBits, tree.cuh).  Synchronises the stream.
  int32_t check_device_errors() {
    uint32_t bits = 0;
    SPB_CUDA(this, cudaMemcpyAsync(&bits, T.error, 4, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    if (!bits) return SPB_OK;
    SPB_CUDA(this, cudaMemsetAsync(T.error, 0, 4, stream));
    if (bits & ERRBIT_POOL) { set_error("node pool exhausted: a tree outgrew spb_config.max_nodes_per_tree"); return SPB_ERR_POOL; }
    if (bits & ERRBIT_TRAJ_FULL) { set_error(std::string("trajectory buffer full: call ") + api + "drain_trajectories"); return SPB_ERR_STATE; }
    if (bits & ERRBIT_BOUNDS) { set_error("device check failed at site " + std::to_string((bits >> 8) & 0xFFu) + " (see ERRBIT_BOUNDS in csrc/)"); return SPB_ERR_STATE; }
    set_error("NaN PUCT score (the reference panics here, mcts.rs:109)");   // ERRBIT_NAN: Connect4 / tic-tac-toe
    return SPB_ERR_STATE;
  }

  // A pointer argument of a device entry point: the kernels read or write it with accesses of `align` bytes.
  struct DevicePointer { const void* p; const char* name; size_t align; };

  // Every non-null pointer must be device memory of the engine's GPU, or managed memory, aligned for the kernels' accesses
  // (a misaligned one would fault on the device): SPB_ERR_ARG naming the first that is not.
  int32_t check_device_pointers(std::initializer_list<DevicePointer> ptrs) {
    for (const DevicePointer& d : ptrs) {
      if (!d.p) continue;
      cudaPointerAttributes a{};
      const cudaError_t ce = cudaPointerGetAttributes(&a, d.p);
      if (ce != cudaSuccess) cudaGetLastError();
      const bool ok = ce == cudaSuccess && (a.type == cudaMemoryTypeManaged || (a.type == cudaMemoryTypeDevice && a.device == cfg.device));
      SPB_ARG(this, ok, std::string(d.name) + " is not device memory of the engine's GPU");
      SPB_ARG(this, reinterpret_cast<uintptr_t>(d.p) % d.align == 0, std::string(d.name) + " is not " + std::to_string(d.align) + "-byte aligned");
    }
    return SPB_OK;
  }

  // Orders n records of src / src_ids into the caller's dst / dst_ids (order_records, records.cu) with scratch from the
  // stage, then waits for the stream.  The caller's pointers are checked here, where they are first needed: a failed
  // check leaves the records where they were.
  int32_t order_into(const Rec* src, const unsigned long long* src_ids, size_t n, Rec* dst, uint64_t* dst_ids) {
    SPB_ARG(this, n < ((size_t)1 << 31), "more than 2^31 - 1 records to order");
    if (int32_t rc = check_device_pointers({{dst, "buf_dev", 8}, {dst_ids, "game_ids_dev", 8}})) return rc;
    if (int32_t rc = ensure_stage(order_scratch_bytes<Rec>(n), 0)) return rc;
    SPB_CUDA(this, order_records(src, src_ids, n, dst, reinterpret_cast<unsigned long long*>(dst_ids), d_stage, stream));
    ++launches;
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    return SPB_OK;
  }

  // ---- bodies of the entry points both ABIs have (spb_X / spb_chess_X) ---------------------------------------------
  // `row`: the width of a root's row of moves (SPB_MAX_ACTIONS / SPB_CHESS_MAX_MOVES).

  static const char* last_error(const HostEngine* e) { return e ? e->err.c_str() : g_create_error.c_str(); }

  int32_t set_root_noise(float alpha, float epsilon, uint64_t seed, uint32_t row) {
    SPB_ARG(this, epsilon >= 0.0f && epsilon <= 1.0f, "root noise: epsilon must be in [0, 1]");
    SPB_ARG(this, epsilon == 0.0f || (alpha > 0.0f && alpha <= FLT_MAX), "root noise: alpha must be finite and > 0");
    if (epsilon > 0.0f && !d_noise_eta) {
      int32_t rc = dalloc(&d_noise_eta, (size_t)T.G * row);
      if (!rc) rc = dalloc(&d_noise_n, (size_t)T.G);
      if (rc) return rc;
    }
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    noise_alpha = alpha;
    noise_seed = seed;
    T.noise_n = d_noise_n;
    T.noise_eps = epsilon;
    T.noise_omeps = 1.0f - epsilon;   // rounded to f32 once, here
    T.root_noise = epsilon > 0.0f ? d_noise_eta : nullptr;
    return SPB_OK;
  }

  // launch(): the engine's noise kernel, which draws eta of every live root into T.root_noise
  template <class Launch>
  int32_t root_noise(uint32_t slot, float* eta, uint32_t* n, uint32_t row, Launch launch) {
    SPB_ARG(this, slot < T.G && eta && n, "bad argument");
    if (!T.root_noise) { set_error(std::string("root noise is off (") + api + "set_root_noise)"); return SPB_ERR_STATE; }
    int32_t rc = launch();
    if (rc) return rc;
    uint32_t hn = 0;
    SPB_CUDA(this, cudaMemcpyAsync(eta, T.root_noise + (size_t)slot * row, row * 4, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaMemcpyAsync(&hn, T.noise_n + slot, 4, cudaMemcpyDeviceToHost, stream));
    rc = check_device_errors();   // synchronises the stream
    if (rc) return rc;
    for (uint32_t i = hn; i < row; ++i) eta[i] = 0.0f;
    *n = hn;
    return SPB_OK;
  }

  int32_t arena_len(uint32_t slot, uint32_t* out) {
    SPB_ARG(this, slot < T.G && out, "bad argument");
    SPB_CUDA(this, cudaMemcpyAsync(out, T.n_nodes + slot, 4, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    return SPB_OK;
  }

  // launch_live(): the engine's kernel that sums the live nodes of every tree into d_misc[0] and, with arena_max, writes
  // the largest arena to d_misc[1] (reported in reserved[0]).
  template <class Launch>
  int32_t get_counters(spb_counters* out, bool arena_max, Launch launch_live) {
    SPB_ARG(this, out, "null out");
    std::memset(out, 0, sizeof *out);
    const size_t misc_bytes = arena_max ? 16 : 8;
    unsigned long long c[CTR_COUNT], live[2] = {0, 0};
    SPB_CUDA(this, cudaMemsetAsync(d_misc, 0, misc_bytes, stream));
    launch_live();
    SPB_CUDA(this, cudaGetLastError());
    ++launches;
    SPB_CUDA(this, cudaMemcpyAsync(c, T.counters, sizeof c, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaMemcpyAsync(live, d_misc, misc_bytes, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    out->simulations = c[CTR_SIMS];
    out->evaluations = c[CTR_EVALS];
    out->terminal_leaves = c[CTR_TERMINAL];
    out->path_length_sum = c[CTR_PATHSUM];
    out->children_created = c[CTR_CHILDREN];
    out->nodes_live = live[0];
    out->kernel_launches = launches;
    if (arena_max) out->reserved[0] = live[1];
    return SPB_OK;
  }

  int32_t reset_counters() {
    SPB_CUDA(this, cudaMemsetAsync(T.counters, 0, CTR_COUNT * 8, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    launches = 0;
    return SPB_OK;
  }

  // Copies the finished records out (buf == NULL: size query) and empties the output buffer.  Buffers not allocated yet
  // (P.out == NULL) hold no record.
  int32_t drain_trajectories(Rec* buf, size_t capacity, size_t* written, uint64_t* game_ids) {
    SPB_ARG(this, written, "null written");
    unsigned long long cur = 0;
    if (P.out) {
      SPB_CUDA(this, cudaMemcpyAsync(&cur, P.out_cursor, 8, cudaMemcpyDeviceToHost, stream));
      SPB_CUDA(this, cudaStreamSynchronize(stream));
    }
    const size_t n = (size_t)std::min<unsigned long long>(cur, P.out_cap);
    *written = n;
    if (!buf) return SPB_OK;                        // size query
    SPB_ARG(this, capacity >= n, "trajectory buffer too small");
    if (n == 0) return SPB_OK;
    std::vector<Rec> pos(n);
    std::vector<unsigned long long> ids(n);
    SPB_CUDA(this, cudaMemcpyAsync(pos.data(), P.out, n * sizeof(Rec), cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaMemcpyAsync(ids.data(), P.out_game, n * 8, cudaMemcpyDeviceToHost, stream));
    SPB_CUDA(this, cudaMemsetAsync(P.out_cursor, 0, 8, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    const std::vector<size_t> order = record_order(pos, ids);
    for (size_t i = 0; i < n; ++i) {
      buf[i] = pos[order[i]];
      if (game_ids) game_ids[i] = ids[order[i]];
    }
    return SPB_OK;
  }

  // The device form of drain_trajectories: the same records in the same order, written to the caller's device buffers.
  // capacity < n is SPB_ERR_ARG with nothing drained.
  int32_t drain_trajectories_device(Rec* buf_dev, size_t capacity, size_t* written, uint64_t* game_ids_dev) {
    SPB_ARG(this, written, "null written");
    unsigned long long cur = 0;
    if (P.out) {
      SPB_CUDA(this, cudaMemcpyAsync(&cur, P.out_cursor, 8, cudaMemcpyDeviceToHost, stream));
      SPB_CUDA(this, cudaStreamSynchronize(stream));
    }
    const size_t n = (size_t)std::min<unsigned long long>(cur, P.out_cap);
    *written = n;
    if (!buf_dev) return SPB_OK;                    // size query
    SPB_ARG(this, capacity >= n, "trajectory buffer too small");
    if (n == 0) return SPB_OK;
    if (int32_t rc = order_into(P.out, P.out_game, n, buf_dev, game_ids_dev)) return rc;
    SPB_CUDA(this, cudaMemsetAsync(P.out_cursor, 0, 8, stream));
    SPB_CUDA(this, cudaStreamSynchronize(stream));
    return SPB_OK;
  }
};

}  // namespace spb
