// engine.cu — the Connect4 / tic-tac-toe host engine (spb_engine, engine.hpp) and the C entry points that launch kernels
// (include/selfplay_b200.h).  What it shares with the chess engine is in host_engine.hpp.
// Device code: kernels.cuh (tree / game / self-play kernels), async.cuh (asynchronous pipeline), evaluator_umma.cu.
#include "kernels.cuh"


// ------------------------------------------------------------------------------------------------
// host engine
// ------------------------------------------------------------------------------------------------
using namespace spb;

thread_local std::string g_create_error;

template <class G_> struct GameType { using type = G_; };
// f(GameType<Connect4>) or f(GameType<TicTacToe>) for `game`; in f: using G = typename decltype(g)::type.
template <class F> static auto with_game(int32_t game, F&& f) {
  return game == SPB_GAME_CONNECT4 ? f(GameType<Connect4>{}) : f(GameType<TicTacToe>{});
}

int32_t spb_engine::init() {
  int32_t rc = open_device();
  if (rc) return rc;
  const bool c4 = cfg.game == SPB_GAME_CONNECT4;
  A = c4 ? Connect4::A : TicTacToe::A;
  max_depth = c4 ? Connect4::MAX_DEPTH : TicTacToe::MAX_DEPTH;
  eval_stride = c4 ? Connect4::EVAL_STRIDE : TicTacToe::EVAL_STRIDE;
  max_ply = c4 ? 42 : 9;
  T.G = cfg.num_games; T.K = cfg.leaves_per_tree; T.cap = cfg.max_nodes_per_tree; T.c = cfg.c;
  const size_t G = T.G, slots = G * T.K, pool = G * (size_t)T.cap;
  for (int b = 0; b < 2; ++b) {
    if ((rc = dalloc(&T.rec[b], pool))) return rc;
    if ((rc = dalloc(&T.par[b], pool))) return rc;
  }
  if ((rc = dalloc(&T.root_state, G))) return rc;
  if ((rc = dalloc(&T.n_nodes, G))) return rc;
  if ((rc = dalloc(&T.buf, G))) return rc;
  if ((rc = dalloc(&T.live, G))) return rc;
  if ((rc = dalloc(&T.path, slots * max_depth))) return rc;
  if ((rc = dalloc(&T.leaf_info, slots))) return rc;
  if ((rc = dalloc(&T.leaf_state, slots))) return rc;
  if ((rc = dalloc(&T.eval_list, slots))) return rc;
  if ((rc = dalloc(&T.eval_count, 4))) return rc;   // [0],[1] ping-pong, [2] snapshot for spb_time_evaluator
  if ((rc = dalloc(&T.eval_out, slots * eval_stride))) return rc;
  if ((rc = dalloc(&T.counters, (size_t)CTR_COUNT))) return rc;
  if ((rc = dalloc(&T.error, 1))) return rc;
  if ((rc = dalloc(&d_rc_moves, G * SPB_MAX_ACTIONS))) return rc;
  if ((rc = dalloc(&d_rc_counts, G * SPB_MAX_ACTIONS))) return rc;
  if ((rc = dalloc(&d_rc_ids, G * SPB_MAX_ACTIONS))) return rc;
  if ((rc = dalloc(&d_rc_n, G))) return rc;
  if ((rc = dalloc(&d_misc, 4))) return rc;
  // asynchronous pipeline: two rings of >= 2G entries (a ring never holds more than G) and the control words
  {
    ring_size = 1024;
    while (ring_size < 2 * (size_t)G) ring_size <<= 1;
    if ((rc = dalloc(&d_ring_slots, 2 * (size_t)ring_size))) return rc;
    if ((rc = dalloc(&d_ctl_words, (size_t)CTL_WORDS))) return rc;
    if ((rc = dalloc(&ctl.sims_left, G))) return rc;
    ctl.leaf.slots = d_ring_slots;            ctl.leaf.mask = ring_size - 1;
    ctl.ready.slots = d_ring_slots + ring_size; ctl.ready.mask = ring_size - 1;
    ctl.leaf.head = d_ctl_words + 0 * 32;  ctl.leaf.tail = d_ctl_words + 1 * 32;
    ctl.ready.head = d_ctl_words + 2 * 32; ctl.ready.tail = d_ctl_words + 3 * 32;
    ctl.n_active = d_ctl_words + 4 * 32;   ctl.done_count = d_ctl_words + 5 * 32;
    ctl.abort = d_ctl_words + 6 * 32;
    ctl.stats = reinterpret_cast<unsigned long long*>(d_ctl_words + 7 * 32);   // 2 lines: ASTAT_COUNT u64
    ctl.stall_ns = 2000000000ull;             // 2 s without a single hand-off anywhere: a bug, reported as SPB_ERR_STATE
    SPB_CUDA(this, cudaMemsetAsync(ctl.sims_left, 0, G * 4, stream));
  }
  SPB_CUDA(this, cudaMemsetAsync(T.live, 0, G, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.buf, 0, G, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.n_nodes, 0, G * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.leaf_info, 0, slots * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.leaf_state, 0, slots * sizeof(PState), stream));
  SPB_CUDA(this, cudaMemsetAsync(T.eval_count, 0, 16, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.eval_out, 0, slots * eval_stride * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.counters, 0, CTR_COUNT * 8, stream));
  SPB_CUDA(this, cudaMemsetAsync(T.error, 0, 4, stream));
  return alloc_trajectories((uint32_t)max_ply);   // self-play buffers, allocated with the engine
}

void spb_engine::release() {
  HostEngine::release();
  drop_step_graph();
}

// The reference's arena is a Vec that grows without bound (mcts.rs:19,151-157).  Here every tree owns a fixed
// slice of the pools, so before a search the slices are widened if the largest live tree could outgrow them:
// one simulation appends at most A children (mcts.rs:131-158).  Growth is a strided device copy; it happens
// before any tree is touched, so a failure leaves the engine as it was.
int32_t spb_engine::ensure_capacity(uint32_t num_searches) {
  unsigned long long mx = 0;
  SPB_CUDA(this, cudaMemsetAsync(d_misc, 0, 8, stream));
  k_max_nodes<<<(T.G + 127) / 128, 128, 0, stream>>>(T, d_misc);
  SPB_CUDA(this, cudaGetLastError());
  ++launches;
  SPB_CUDA(this, cudaMemcpyAsync(&mx, d_misc, 8, cudaMemcpyDeviceToHost, stream));
  SPB_CUDA(this, cudaStreamSynchronize(stream));
  const unsigned long long need = mx + (unsigned long long)num_searches * (unsigned long long)A;
  if (need <= T.cap || (cfg.flags & SPB_FLAG_FIXED_POOL)) return SPB_OK;   // fixed pool: the device flag reports exhaustion
  unsigned long long ncap = std::max<unsigned long long>(need, 2ull * T.cap);
  ncap = (ncap + 1023ull) & ~1023ull;
  if (ncap > MAX_CAP) ncap = MAX_CAP;
  if (need > ncap) { set_error("node pool exhausted: a tree would exceed 2^24 nodes"); return SPB_ERR_POOL; }
  const size_t pool = (size_t)T.G * (size_t)ncap;
  NodeRec* nrec[2] = {nullptr, nullptr};
  uint32_t* npar[2] = {nullptr, nullptr};
  cudaError_t ce = cudaSuccess;
  for (int b = 0; b < 2 && ce == cudaSuccess; ++b) {
    ce = cudaMalloc((void**)&nrec[b], pool * sizeof(NodeRec));
    if (ce == cudaSuccess) ce = cudaMalloc((void**)&npar[b], pool * sizeof(uint32_t));
  }
  for (int b = 0; b < 2 && ce == cudaSuccess; ++b) {
    ce = cudaMemcpy2DAsync(nrec[b], ncap * sizeof(NodeRec), T.rec[b], (size_t)T.cap * sizeof(NodeRec), (size_t)T.cap * sizeof(NodeRec), T.G,
                           cudaMemcpyDeviceToDevice, stream);
    if (ce == cudaSuccess)
      ce = cudaMemcpy2DAsync(npar[b], ncap * sizeof(uint32_t), T.par[b], (size_t)T.cap * sizeof(uint32_t), (size_t)T.cap * sizeof(uint32_t), T.G,
                             cudaMemcpyDeviceToDevice, stream);
  }
  if (ce == cudaSuccess) ce = cudaStreamSynchronize(stream);
  if (ce != cudaSuccess) {
    for (int b = 0; b < 2; ++b) { if (nrec[b]) cudaFree(nrec[b]); if (npar[b]) cudaFree(npar[b]); }
    cudaGetLastError();
    set_error(std::string("node pool exhausted: cannot grow the pools to ") + std::to_string(ncap) + " nodes per tree (" + cudaGetErrorString(ce) + ")");
    return SPB_ERR_POOL;
  }
  for (int b = 0; b < 2; ++b) {
    for (void* old : {(void*)T.rec[b], (void*)T.par[b]}) {
      allocs.erase(std::find(allocs.begin(), allocs.end(), old));
      cudaFree(old);
    }
    T.rec[b] = nrec[b]; T.par[b] = npar[b];
    allocs.push_back(nrec[b]); allocs.push_back(npar[b]);
  }
  T.cap = (uint32_t)ncap;
  cfg.max_nodes_per_tree = T.cap;
  drop_step_graph();   // the graph captured the old pointers
  return SPB_OK;
}

template <class G>
int32_t spb_engine::launch_eval_step(uint32_t parity) {
  const uint32_t slots = T.G * T.K;
  if (cfg.evaluator == SPB_EVAL_NET) {
    SPB_CUDA(this, evaluator.launch(T.leaf_state, T.eval_list, &T.eval_count[parity & 1], slots, T.eval_out, G::EVAL_STRIDE, nullptr,
                                    (cfg.flags & SPB_FLAG_EVAL_SIMT) != 0, stream));
  } else {
    with_builtin_eval(cfg.evaluator, [&](auto ev) {
      k_eval_builtin<G, decltype(ev)::value><<<(slots + 255) / 256, 256, 0, stream>>>(T.leaf_state, T.eval_list, &T.eval_count[parity & 1], T.eval_out);
    });
  }
  ++launches;
  return SPB_OK;
}

// Launch with programmatic stream serialization: the grid may begin before its predecessor in the stream has drained
// (it blocks in griddepcontrol.wait before touching anything the predecessor writes).  Only for kernels that contain
// that wait.
template <class... P, class... A>
static cudaError_t launch_pdl(void (*kernel)(P...), uint32_t blocks, uint32_t threads, cudaStream_t stream, A... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(blocks);
  cfg.blockDim = dim3(threads);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<P>(args)...);
}

template <class G>
int32_t spb_engine::search_t(uint32_t num_searches) {
  if (num_searches == 0) return SPB_OK;
  const uint32_t blocks = (T.G + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  const bool split = cfg.evaluator == SPB_EVAL_NET || (cfg.flags & SPB_FLAG_FORCE_SPLIT) || T.K > 1;
  if (cfg.evaluator == SPB_EVAL_NET && !evaluator.loaded()) { set_error("no weights loaded: call spb_load_weights first"); return SPB_ERR_STATE; }
  { int32_t rc = ensure_capacity(num_searches); if (rc != SPB_OK) return rc; }
  // The network evaluator (and the built-in evaluators under SPB_FLAG_FORCE_SPLIT) run through the asynchronous
  // pipeline unless the lock-step pipeline is asked for; K > 1 leaves per tree is a lock-step extension.
  const bool async = split && T.K == 1 && !(cfg.flags & SPB_FLAG_LOCKSTEP);
  SPB_CUDA(this, cudaEventRecord(ev0, stream));
  last_eval_launches = 0;
  if (T.root_noise) { int32_t rc = launch_root_noise(); if (rc != SPB_OK) return rc; }   // eta of every root, before any descent
  if (async) {
    int32_t rc = search_async<G>(num_searches);
    if (rc != SPB_OK) return rc;
  } else if (!split) {
    with_builtin_eval(cfg.evaluator, [&](auto ev) { k_search_fused<G, decltype(ev)::value><<<blocks, THREADS, 0, stream>>>(T, num_searches); });
    SPB_CUDA(this, cudaGetLastError());
    ++launches;
  } else if (T.K > 1) {
    // EXTENSION: K leaves per tree per step with virtual loss (see k_tree_step_multi).
    const uint32_t K = T.K, steps = (num_searches + K - 1) / K;
    SPB_CUDA(this, cudaMemsetAsync(T.eval_count, 0, 8, stream));
    k_tree_step_multi<G><<<blocks, THREADS, 0, stream>>>(T, 0, std::min(K, num_searches), 0u);
    SPB_CUDA(this, cudaGetLastError());
    ++launches;
    for (uint32_t j = 0; j < steps; ++j) {
      const bool last = (j == steps - 1);
      if (last) {
        SPB_CUDA(this, cudaMemcpyAsync(&T.eval_count[2], &T.eval_count[j & 1u], 4, cudaMemcpyDeviceToDevice, stream));
        last_eval_parity = 2;
      }
      int32_t rc = launch_eval_step<G>(j);
      if (rc != SPB_OK) return rc;
      SPB_CUDA(this, cudaGetLastError());
      ++last_eval_launches;
      const uint32_t done_after = std::min(num_searches, (j + 1) * K);
      const uint32_t k_next = last ? 0u : std::min(K, num_searches - done_after);
      k_tree_step_multi<G><<<blocks, THREADS, 0, stream>>>(T, 1, k_next, j + 1);
      SPB_CUDA(this, cudaGetLastError());
      ++launches;
    }
  } else {
    // step j: select writes eval_count[j&1]; the kernel also zeroes eval_count[(j+1)&1].
    SPB_CUDA(this, cudaMemsetAsync(T.eval_count, 0, 8, stream));
    SPB_CUDA(this, launch_pdl(k_tree_step<G>, blocks, THREADS, stream, T, 0, 1, 0u));
    ++launches;
    uint32_t j = 0;
    const bool use_graph = !(cfg.flags & SPB_FLAG_NO_GRAPH) && num_searches > 2;
    if (use_graph) {
      // One graph = two steps (parities 0,1): eval(0) step(1) eval(1) step(0).
      if (!step_graph) {
        cudaGraph_t graph;
        SPB_CUDA(this, cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        int32_t rc = launch_eval_step<G>(0u);
        cudaError_t pe = launch_pdl(k_tree_step<G>, blocks, THREADS, stream, T, 1, 1, 1u);
        if (rc == SPB_OK) rc = launch_eval_step<G>(1u);
        if (pe == cudaSuccess) pe = launch_pdl(k_tree_step<G>, blocks, THREADS, stream, T, 1, 1, 0u);
        cudaError_t ce = cudaStreamEndCapture(stream, &graph);
        launches -= 2;
        if (rc != SPB_OK) return rc;
        if (ce == cudaSuccess) ce = pe;
        if (ce != cudaSuccess) { set_error(std::string("graph capture: ") + cudaGetErrorString(ce)); return SPB_ERR_CUDA; }
        SPB_CUDA(this, cudaGraphInstantiate(&step_graph, graph, 0));
        cudaGraphDestroy(graph);
      }
      while (j + 2 <= num_searches - 1) {
        SPB_CUDA(this, cudaGraphLaunch(step_graph, stream));
        launches += 4;
        last_eval_launches += 2;
        j += 2;
      }
    }
    for (; j < num_searches; ++j) {
      int32_t rc = launch_eval_step<G>(j);
      if (rc != SPB_OK) return rc;
      SPB_CUDA(this, cudaGetLastError());
      ++last_eval_launches;
      const int last = (j == num_searches - 1);
      if (last) {   // keep the size of the last work list: the final tree step clears the ping-pong counter
        SPB_CUDA(this, cudaMemcpyAsync(&T.eval_count[2], &T.eval_count[j & 1u], 4, cudaMemcpyDeviceToDevice, stream));
        last_eval_parity = 2;
      }
      SPB_CUDA(this, launch_pdl(k_tree_step<G>, blocks, THREADS, stream, T, 1, last ? 0 : 1, j + 1));
      ++launches;
    }
  }
  SPB_CUDA(this, cudaEventRecord(ev1, stream));
  uint32_t ctl_host[CTL_WORDS];
  if (async) SPB_CUDA(this, cudaMemcpyAsync(ctl_host, d_ctl_words, sizeof ctl_host, cudaMemcpyDeviceToHost, stream));
  int32_t rc = check_device_errors();   // synchronises the stream
  SPB_CUDA(this, cudaEventElapsedTime(&last_search_ms, ev0, ev1));
  if (async) std::memcpy(last_async_stats, &ctl_host[7 * 32], sizeof(uint64_t) * ASTAT_COUNT);
  if (rc == SPB_OK && async && (ctl_host[6 * 32] != 0u || ctl_host[5 * 32] != ctl_host[4 * 32])) {
    char msg[256];
    std::snprintf(msg, sizeof msg, "asynchronous search pipeline stalled (abort=%u, trees done %u of %u, leaf ring %u/%u, ready ring %u/%u)",
                  ctl_host[6 * 32], ctl_host[5 * 32], ctl_host[4 * 32], ctl_host[0], ctl_host[32], ctl_host[64], ctl_host[96]);
    set_error(msg);
    return SPB_ERR_STATE;
  }
  return rc;
}

// EXTENSION (DESIGN.md §4.6): eta of every live root into T.root_noise (k_root_noise).
int32_t spb_engine::launch_root_noise() {
  const uint32_t blocks = (T.G + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  with_game(cfg.game, [&](auto g) {
    k_root_noise<typename decltype(g)::type><<<blocks, THREADS, 0, stream>>>(T, P.game_id, noise_alpha, noise_seed);
  });
  SPB_CUDA(this, cudaGetLastError());
  ++launches;
  return SPB_OK;
}

// The evaluation cache of the asynchronous pipeline: per tree the next power of two >= 2 x num_searches slots (at least
// one probe window, at most EVAL_CACHE_MAX_SLOTS), so that the <= num_searches records of one search fill at most half of
// it.  Grow-only like the node pools; zeroed once when allocated (epoch 0 = empty).  No result depends on the cache, so
// when the allocation fails the searches run without one.
int32_t spb_engine::ensure_eval_cache(uint32_t num_searches) {
  uint32_t want = EVAL_CACHE_WINDOW;
  while (want < 2ull * num_searches && want < EVAL_CACHE_MAX_SLOTS) want <<= 1;
  if (want <= ctl.cache.slots || want <= cache_tried) return SPB_OK;
  cache_tried = want;
  const size_t n = (size_t)T.G * want;
  EvalCache nc{nullptr, nullptr, nullptr, want};
  cudaError_t ce = cudaMalloc((void**)&nc.key, n * sizeof(ulonglong2));
  if (ce == cudaSuccess) ce = cudaMalloc((void**)&nc.epoch, n * sizeof(uint32_t));
  if (ce == cudaSuccess) ce = cudaMalloc((void**)&nc.rec, n * (size_t)eval_stride * sizeof(float));
  if (ce == cudaSuccess) ce = cudaMemsetAsync(nc.epoch, 0, n * sizeof(uint32_t), stream);
  if (ce != cudaSuccess) {
    for (void* p : {(void*)nc.key, (void*)nc.epoch, (void*)nc.rec}) if (p) cudaFree(p);
    cudaGetLastError();                                              // an allocation failure is not sticky: clear it
    return SPB_OK;                                                   // keep the smaller table (or none)
  }
  SPB_CUDA(this, cudaStreamSynchronize(stream));                     // no search of the old table is in flight
  for (void* old : {(void*)ctl.cache.key, (void*)ctl.cache.epoch, (void*)ctl.cache.rec}) {
    if (!old) continue;
    allocs.erase(std::find(allocs.begin(), allocs.end(), old));
    cudaFree(old);
  }
  for (void* p : {(void*)nc.key, (void*)nc.epoch, (void*)nc.rec}) allocs.push_back(p);
  ctl.cache = nc;
  return SPB_OK;
}

// One search through the asynchronous pipeline: rings reset, every live tree queued, ONE resident kernel until all trees
// have completed their simulations (network: evaluator CTAs + tree warps; built-in evaluators: evaluator warps + tree warps).
template <class G>
int32_t spb_engine::search_async(uint32_t num_searches) {
  { int32_t rc = ensure_eval_cache(num_searches); if (rc != SPB_OK) return rc; }
  if (++cache_epoch == 0u) {   // the epoch wrapped: entries of epoch 1 could look live again
    if (ctl.cache.epoch) SPB_CUDA(this, cudaMemsetAsync(ctl.cache.epoch, 0, (size_t)T.G * ctl.cache.slots * 4, stream));
    cache_epoch = 1u;
  }
  ctl.epoch = cache_epoch;
  SPB_CUDA(this, cudaMemsetAsync(d_ctl_words, 0, (size_t)CTL_WORDS * 4, stream));
  SPB_CUDA(this, cudaMemsetAsync(d_ring_slots, 0, 2 * (size_t)ring_size * 8, stream));
  k_async_init<<<(T.G + 127) / 128, 128, 0, stream>>>(T, ctl, num_searches);
  SPB_CUDA(this, cudaGetLastError());
  ++launches;
  if (cfg.evaluator == SPB_EVAL_NET) {
    SPB_CUDA(this, evaluator.launch_ring(T, ctl, stream));
    ++last_eval_launches;
  } else {
    const uint32_t grid = std::max(1u, std::min(592u, (T.G + 3u) / 4u));
    with_builtin_eval(cfg.evaluator, [&](auto ev) { k_async_builtin<G, decltype(ev)::value><<<grid, THREADS, 0, stream>>>(T, ctl); });
    SPB_CUDA(this, cudaGetLastError());
  }
  ++launches;
  last_eval_parity = -1;
  return SPB_OK;
}

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int32_t spb_abi_version(void) { return SPB_ABI_VERSION; }

int32_t spb_default_config(spb_config* cfg) {
  if (!cfg) return SPB_ERR_ARG;
  std::memset(cfg, 0, sizeof *cfg);
  cfg->abi_version = SPB_ABI_VERSION;
  cfg->game = SPB_GAME_CONNECT4;
  cfg->device = 0;
  cfg->num_games = 100;            // mcts.rs:54
  cfg->max_nodes_per_tree = 0;
  cfg->leaves_per_tree = 1;
  cfg->c = 2.0f;                   // mcts.rs:49
  cfg->evaluator = SPB_EVAL_NET;
  return SPB_OK;
}

// The checks of spb_create beyond HostEngine::config_error (max_nodes_per_tree 0 already replaced by its default).
static const char* config_error(const spb_config& c) {
  if (const char* m = spb_engine::config_error(c)) return m;
  if (c.game != SPB_GAME_CONNECT4 && c.game != SPB_GAME_TICTACTOE) return "unknown game";
  if (c.num_games == 0 || c.num_games > (1u << 22)) return "num_games out of range";
  if (c.leaves_per_tree < 1 || c.leaves_per_tree > 16) return "leaves_per_tree must be in 1..16";
  if (c.max_nodes_per_tree < 16 || c.max_nodes_per_tree > MAX_CAP) return "max_nodes_per_tree out of range";
  return nullptr;
}

int32_t spb_create(const spb_config* cfg, spb_engine** out) {
  if (!cfg || !out) { g_create_error = "null argument"; return SPB_ERR_ARG; }
  *out = nullptr;
  spb_config c = *cfg;
  if (c.max_nodes_per_tree == 0) c.max_nodes_per_tree = 16384;
  if (const char* m = config_error(c)) { g_create_error = m; return SPB_ERR_ARG; }
  return spb_engine::create(c, out);
}

int32_t spb_destroy(spb_engine* e) {
  if (!e) return SPB_ERR_ARG;
  spb_comm_destroy(e);
  e->release();
  delete e;
  return SPB_OK;
}

const char* spb_last_error(const spb_engine* e) { return spb_engine::last_error(e); }

int32_t spb_load_weights(spb_engine* e, const void* blob, size_t n) {
  SPB_GUARD(e);
  SPB_ARG(e, blob && n > 8, "null / empty weight blob");
  HostNet net;
  std::string err;
  if (!parse_safetensors_net(blob, n, e->cfg.game, &net, &err)) { e->set_error("spb_load_weights: " + err); return SPB_ERR_WEIGHTS; }
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (!e->evaluator.upload(net, &err)) { e->set_error("spb_load_weights: " + err); return SPB_ERR_CUDA; }
  // The captured step graph holds the address of the previous weight image in its kernel nodes (hot swap between
  // generations, learner_concurrent.rs:158-159): drop it, the next search captures the new one.
  e->drop_step_graph();
  e->last_eval_parity = -1;
  return SPB_OK;
}

int32_t spb_check_weights(int32_t game, const void* blob, size_t n, char* err, size_t err_cap) {
  if (err && err_cap) err[0] = 0;
  if (game != SPB_GAME_CONNECT4 && game != SPB_GAME_TICTACTOE) return SPB_ERR_ARG;
  if (!blob) return SPB_ERR_ARG;
  HostNet net;
  std::string msg;
  if (!parse_safetensors_net(blob, n, game, &net, &msg)) {
    if (err && err_cap) { std::strncpy(err, msg.c_str(), err_cap - 1); err[err_cap - 1] = 0; }
    return SPB_ERR_WEIGHTS;
  }
  return SPB_OK;
}

int32_t spb_reset_games(spb_engine* e, const uint32_t* slots, uint32_t n, const spb_state* roots) {
  SPB_GUARD(e);
  if (int32_t rc = e->check_slots(slots, n)) return rc;
  if (n == 0) return SPB_OK;
  StageLayout L;
  const size_t o_slots = L.take(slots ? (size_t)n * 4 : 0), o_roots = L.take(roots ? (size_t)n * sizeof(PState) : 0);
  if (int32_t rc = e->ensure_stage(L.bytes, L.bytes)) return rc;
  if (slots) std::memcpy(e->h_at<uint32_t>(o_slots), slots, (size_t)n * 4);
  if (roots) {
    PState* hp = e->h_at<PState>(o_roots);
    for (uint32_t i = 0; i < n; ++i) hp[i] = ps_from_abi(roots[i]);
  }
  if (L.bytes) SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, L.bytes, cudaMemcpyHostToDevice, e->stream));
  k_reset<<<(n + 127) / 128, 128, 0, e->stream>>>(e->T, e->P.hist_len, e->P.parked, slots ? e->d_at<uint32_t>(o_slots) : nullptr,
                                                  roots ? e->d_at<PState>(o_roots) : nullptr, n);
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));   // staging buffer is reused by the next call
  return SPB_OK;
}

int32_t spb_search(spb_engine* e, uint32_t num_searches) {
  SPB_GUARD(e);
  return with_game(e->cfg.game, [&](auto g) { return e->search_t<typename decltype(g)::type>(num_searches); });
}

static int32_t fetch_root_children(spb_engine* e) {
  k_root_children<<<(e->T.G + 127) / 128, 128, 0, e->stream>>>(e->T, e->d_rc_moves, e->d_rc_counts, e->d_rc_ids, e->d_rc_n);
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  return SPB_OK;
}

int32_t spb_root_children_all(spb_engine* e, uint8_t* actions, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children) {
  SPB_GUARD(e);
  return e->root_children(0, e->T.G, actions, visit_counts, child_ids, n_children, [e] { return fetch_root_children(e); });
}

int32_t spb_root_children(spb_engine* e, uint32_t slot, uint8_t* actions, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children) {
  SPB_GUARD(e);
  return e->root_children(slot, 1, actions, visit_counts, child_ids, n_children, [e] { return fetch_root_children(e); });
}

int32_t spb_root_policy(spb_engine* e, uint32_t slot, float* policy) {
  SPB_GUARD(e);
  SPB_ARG(e, policy, "null policy");
  uint8_t a[SPB_MAX_ACTIONS]; uint32_t c[SPB_MAX_ACTIONS], n = 0;
  int32_t rc = spb_root_children(e, slot, a, c, nullptr, &n);
  if (rc) return rc;
  // mcts.rs:315-328: zero policy, set_prob(action, count as f32), normalize (ndarray sum order; counts are
  // integers < 2^24 so every order gives the same f32 sum), f32 divide.
  float p[SPB_MAX_ACTIONS] = {0};
  for (uint32_t i = 0; i < n; ++i) p[a[i]] = (float)c[i];
  float s = 0.0f;
  for (int i = 0; i < e->A; ++i) s += p[i];
  for (int i = 0; i < e->A; ++i) policy[i] = p[i] / s;
  return SPB_OK;
}

int32_t spb_advance(spb_engine* e, const uint32_t* slots, const uint32_t* node_ids, uint32_t n, spb_state* out_states) {
  SPB_GUARD(e);
  SPB_ARG(e, node_ids, "null node_ids");
  if (int32_t rc = e->check_slots(slots, n)) return rc;
  if (n == 0) return SPB_OK;
  // validate against arena lengths (one D2H of n_nodes)
  std::vector<uint32_t> nn(e->T.G);
  SPB_CUDA(e, cudaMemcpyAsync(nn.data(), e->T.n_nodes, (size_t)e->T.G * 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  for (uint32_t i = 0; i < n; ++i) SPB_ARG(e, node_ids[i] < nn[slots ? slots[i] : i], "node id out of range");
  StageLayout L;
  const size_t o_slots = L.take(slots ? (size_t)n * 4 : 0), o_ids = L.take((size_t)n * 4), o_out = L.take((size_t)n * sizeof(PState));
  if (int32_t rc = e->ensure_stage(L.bytes, L.bytes)) return rc;
  if (slots) std::memcpy(e->h_at<uint32_t>(o_slots), slots, (size_t)n * 4);
  std::memcpy(e->h_at<uint32_t>(o_ids), node_ids, (size_t)n * 4);
  SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, o_out, cudaMemcpyHostToDevice, e->stream));   // the inputs: everything before o_out
  const uint32_t blocks = (n + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  const uint32_t* dsl = slots ? e->d_at<uint32_t>(o_slots) : nullptr;
  const uint32_t* dn = e->d_at<uint32_t>(o_ids);
  PState* dout = e->d_at<PState>(o_out);
  with_game(e->cfg.game, [&](auto g) { k_advance<typename decltype(g)::type><<<blocks, THREADS, 0, e->stream>>>(e->T, dsl, dn, n, dout); });
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(e->h_at<PState>(o_out), dout, (size_t)n * sizeof(PState), cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (out_states) {
    const PState* hp = e->h_at<PState>(o_out);
    for (uint32_t i = 0; i < n; ++i) out_states[i] = ps_to_abi(hp[i]);
  }
  return SPB_OK;
}

int32_t spb_arena_len(spb_engine* e, uint32_t slot, uint32_t* out) {
  SPB_GUARD(e);
  return e->arena_len(slot, out);
}

int32_t spb_get_state(spb_engine* e, uint32_t slot, uint32_t node_id, spb_state* out) {
  SPB_GUARD(e);
  SPB_ARG(e, slot < e->T.G && out, "bad argument");
  uint32_t len = 0;
  int32_t rc = spb_arena_len(e, slot, &len);
  if (rc) return rc;
  SPB_ARG(e, node_id < len, "node id out of range");
  rc = e->ensure_stage(sizeof(PState), 0);
  if (rc) return rc;
  with_game(e->cfg.game, [&](auto g) { k_get_state<typename decltype(g)::type><<<1, 1, 0, e->stream>>>(e->T, slot, node_id, e->d_at<PState>(0)); });
  ++e->launches;
  PState ps;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(&ps, e->d_stage, sizeof ps, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  *out = ps_to_abi(ps);
  return SPB_OK;
}

int32_t spb_set_root_noise(spb_engine* e, float alpha, float epsilon, uint64_t seed) {
  SPB_GUARD(e);
  const int32_t rc = e->set_root_noise(alpha, epsilon, seed);
  // the captured step graph holds the previous Trees (and with it the noise settings): the next search captures anew
  if (rc == SPB_OK) e->drop_step_graph();
  return rc;
}

int32_t spb_root_noise(spb_engine* e, uint32_t slot, float* eta, uint32_t* n) {
  SPB_GUARD(e);
  return e->root_noise(slot, eta, n, [e] { return e->launch_root_noise(); });
}

int32_t spb_node_stats(spb_engine* e, uint32_t slot, uint32_t node_id, uint32_t* visit_count, float* value_sum, float* prior,
                       uint32_t* first_child, uint32_t* n_children) {
  SPB_GUARD(e);
  SPB_ARG(e, slot < e->T.G, "slot out of range");
  uint32_t len = 0;
  int32_t rc = spb_arena_len(e, slot, &len);
  if (rc) return rc;
  SPB_ARG(e, node_id < len, "node id out of range");
  rc = e->ensure_stage(sizeof(NodeRec), 0);
  if (rc) return rc;
  k_node_stats<<<1, 1, 0, e->stream>>>(e->T, slot, node_id, e->d_at<NodeRec>(0));
  ++e->launches;
  NodeRec r;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(&r, e->d_stage, sizeof r, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (visit_count) *visit_count = r.N;
  if (value_sum) *value_sum = r.W;
  if (prior) *prior = r.P;
  if (first_child) *first_child = info_fc(r.info);
  if (n_children) *n_children = info_nc(r.info);
  return SPB_OK;
}

}  // extern "C"

// ---- predict ------------------------------------------------------------------------------------
template <class G>
static int32_t predict_t(spb_engine* e, const spb_state* states, uint32_t n, float* policies, float* values, float* raw_logits) {
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(PState)), o_cnt = L.take(4), o_out = L.take((size_t)n * G::EVAL_STRIDE * 4);
  const size_t o_pol = L.take((size_t)n * G::A * 4), o_val = L.take((size_t)n * 4), o_log = L.take((size_t)n * G::A * 4);
  if (int32_t rc = e->ensure_stage(L.bytes, L.bytes)) return rc;
  auto* hs = e->h_at<uint8_t>(0);
  PState* hp = e->h_at<PState>(o_states);
  for (uint32_t i = 0; i < n; ++i) hp[i] = ps_from_abi(states[i]);
  *e->h_at<uint32_t>(o_cnt) = n;
  SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, hs, o_cnt + 4, cudaMemcpyHostToDevice, e->stream));
  PState* dstates = e->d_at<PState>(o_states);
  uint32_t* dcnt = e->d_at<uint32_t>(o_cnt);
  float* dout = e->d_at<float>(o_out);
  float* dlog = e->d_at<float>(o_log);
  if (e->cfg.evaluator == SPB_EVAL_NET) {
    if (!e->evaluator.loaded()) { e->set_error("no weights loaded: call spb_load_weights first"); return SPB_ERR_STATE; }
    SPB_CUDA(e, cudaMemsetAsync(dlog, 0, (size_t)n * G::A * 4, e->stream));
    SPB_CUDA(e, e->evaluator.launch(dstates, nullptr, dcnt, n, dout, G::EVAL_STRIDE, raw_logits ? dlog : nullptr,
                                    (e->cfg.flags & SPB_FLAG_EVAL_SIMT) != 0, e->stream));
  } else {
    // identity work list: k_eval_builtin indexes states by list entry, so build 0..n-1 in the logits area
    std::vector<uint32_t> idl(n);
    for (uint32_t i = 0; i < n; ++i) idl[i] = i;
    SPB_CUDA(e, cudaMemcpyAsync(dlog, idl.data(), (size_t)n * 4, cudaMemcpyHostToDevice, e->stream));
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
    with_builtin_eval(e->cfg.evaluator, [&](auto ev) {
      k_eval_builtin<G, decltype(ev)::value><<<(n + 255) / 256, 256, 0, e->stream>>>(dstates, reinterpret_cast<uint32_t*>(dlog), dcnt, dout);
    });
    SPB_CUDA(e, cudaGetLastError());
  }
  ++e->launches;
  k_mask_policies<G><<<(n + 127) / 128, 128, 0, e->stream>>>(dstates, n, dout, e->d_at<float>(o_pol), e->d_at<float>(o_val));
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(hs + o_pol, e->d_at<uint8_t>(o_pol), L.bytes - o_pol, cudaMemcpyDeviceToHost, e->stream));   // policies, values, logits
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  if (policies) std::memcpy(policies, hs + o_pol, (size_t)n * G::A * 4);
  if (values) std::memcpy(values, hs + o_val, (size_t)n * 4);
  if (raw_logits && e->cfg.evaluator == SPB_EVAL_NET) std::memcpy(raw_logits, hs + o_log, (size_t)n * G::A * 4);
  return SPB_OK;
}

extern "C" {

int32_t spb_predict(spb_engine* e, const spb_state* states, uint32_t n, float* policies, float* values, float* raw_logits) {
  SPB_GUARD(e);
  SPB_ARG(e, states || n == 0, "null states");
  if (n == 0) return SPB_OK;
  return with_game(e->cfg.game, [&](auto g) { return predict_t<typename decltype(g)::type>(e, states, n, policies, values, raw_logits); });
}

// ---- game rules ---------------------------------------------------------------------------------
// Grows the stage and converts the n states into the pinned stage at offset 0: the states come first in every layout below.
static int32_t upload_states(spb_engine* e, const spb_state* states, uint32_t n, size_t d_bytes, size_t h_bytes) {
  const int32_t rc = e->ensure_stage(d_bytes, h_bytes);
  if (rc) return rc;
  PState* hp = e->h_at<PState>(0);
  for (uint32_t i = 0; i < n; ++i) hp[i] = ps_from_abi(states[i]);
  return SPB_OK;
}

int32_t spb_game_next_states(spb_engine* e, const spb_state* states, const uint8_t* actions, uint32_t n, spb_state* out_states, int32_t* err) {
  SPB_GUARD(e);
  SPB_ARG(e, states && actions && out_states && err, "null argument");
  if (n == 0) return SPB_OK;
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(PState)), o_act = L.take(n), o_out = L.take((size_t)n * sizeof(PState)), o_err = L.take((size_t)n * 4);
  if (int32_t rc = upload_states(e, states, n, L.bytes, L.bytes)) return rc;
  std::memcpy(e->h_at<uint8_t>(o_act), actions, n);
  SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, o_out, cudaMemcpyHostToDevice, e->stream));   // the inputs: everything before o_out
  with_game(e->cfg.game, [&](auto g) {
    k_game_next<typename decltype(g)::type><<<(n + 127) / 128, 128, 0, e->stream>>>(e->d_at<PState>(o_states), e->d_at<uint8_t>(o_act), n, e->d_at<PState>(o_out),
                                                                                   e->d_at<int32_t>(o_err));
  });
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(e->h_at<uint8_t>(o_out), e->d_at<uint8_t>(o_out), L.bytes - o_out, cudaMemcpyDeviceToHost, e->stream));   // states, errors
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  const PState* hp = e->h_at<PState>(o_out);
  const int32_t* he = e->h_at<int32_t>(o_err);
  for (uint32_t i = 0; i < n; ++i) { out_states[i] = ps_to_abi(hp[i]); err[i] = he[i]; }
  return SPB_OK;
}

int32_t spb_game_valid_actions(spb_engine* e, const spb_state* states, uint32_t n, uint32_t* masks) {
  SPB_GUARD(e);
  SPB_ARG(e, states && masks, "null argument");
  if (n == 0) return SPB_OK;
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(PState)), o_out = L.take((size_t)n * 4);
  if (int32_t rc = upload_states(e, states, n, L.bytes, o_out)) return rc;
  SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, o_out, cudaMemcpyHostToDevice, e->stream));
  with_game(e->cfg.game, [&](auto g) {
    k_game_valid<typename decltype(g)::type><<<(n + 127) / 128, 128, 0, e->stream>>>(e->d_at<PState>(o_states), n, e->d_at<uint32_t>(o_out));
  });
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(masks, e->d_at<uint32_t>(o_out), (size_t)n * 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

int32_t spb_game_encode(spb_engine* e, const spb_state* states, uint32_t n, float* out) {
  SPB_GUARD(e);
  SPB_ARG(e, states && out, "null argument");
  if (n == 0) return SPB_OK;
  const size_t total = (size_t)n * (e->cfg.game == SPB_GAME_CONNECT4 ? 3 * 6 * 7 : 27);
  StageLayout L;
  const size_t o_states = L.take((size_t)n * sizeof(PState)), o_out = L.take(total * 4);
  if (int32_t rc = upload_states(e, states, n, L.bytes, o_out)) return rc;
  SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, o_out, cudaMemcpyHostToDevice, e->stream));
  with_game(e->cfg.game, [&](auto g) {
    k_game_encode<typename decltype(g)::type><<<(unsigned)((total + 255) / 256), 256, 0, e->stream>>>(e->d_at<PState>(o_states), n, e->d_at<float>(o_out));
  });
  ++e->launches;
  SPB_CUDA(e, cudaGetLastError());
  SPB_CUDA(e, cudaMemcpyAsync(out, e->d_at<float>(o_out), total * 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

// ---- self-play ----------------------------------------------------------------------------------
int32_t spb_selfplay_step(spb_engine* e, int32_t rule, float temperature, uint64_t seed, const spb_state* restart_roots, uint32_t* n_finished) {
  SPB_GUARD(e);
  const uint32_t G = e->T.G;
  PState* droots = nullptr;
  if (restart_roots) {
    const size_t bytes = (size_t)G * sizeof(PState);
    if (int32_t rc = upload_states(e, restart_roots, G, bytes, bytes)) return rc;
    SPB_CUDA(e, cudaMemcpyAsync(e->d_stage, e->h_stage, bytes, cudaMemcpyHostToDevice, e->stream));
    droots = e->d_at<PState>(0);
  }
  const uint32_t blocks = (G + WARPS_PER_BLOCK - 1) / WARPS_PER_BLOCK;
  return e->selfplay_step(rule, n_finished, [&] {
    with_game(e->cfg.game, [&](auto g) {
      k_selfplay_step<typename decltype(g)::type><<<blocks, THREADS, 0, e->stream>>>(e->T, e->P, rule, temperature, seed, droots);
    });
  });
}

int32_t spb_drain_trajectories(spb_engine* e, spb_position* buf, size_t capacity, size_t* written, uint64_t* game_ids) {
  SPB_GUARD(e);
  return e->drain_trajectories(buf, capacity, written, game_ids);
}

int32_t spb_drain_trajectories_device(spb_engine* e, spb_position* buf_dev, size_t capacity, size_t* written, uint64_t* game_ids_dev) {
  SPB_GUARD(e);
  return e->drain_trajectories_device(buf_dev, capacity, written, game_ids_dev);
}

// ---- counters -----------------------------------------------------------------------------------
int32_t spb_get_counters(spb_engine* e, spb_counters* out) {
  SPB_GUARD(e);
  return e->get_counters(out, false, [e] { k_nodes_live<<<(e->T.G + 127) / 128, 128, 0, e->stream>>>(e->T, e->d_misc); });
}

int32_t spb_reset_counters(spb_engine* e) {
  SPB_GUARD(e);
  return e->reset_counters();
}

int32_t spb_last_search_timing(spb_engine* e, float* search_ms, float* evaluator_ms, uint32_t* evaluator_launches) {
  if (!e) return SPB_ERR_ARG;
  if (search_ms) *search_ms = e->last_search_ms;
  if (evaluator_ms) *evaluator_ms = e->last_eval_ms;
  if (evaluator_launches) *evaluator_launches = e->last_eval_launches;
  return SPB_OK;
}

int32_t spb_time_evaluator(spb_engine* e, uint32_t iters, float* avg_ms, uint32_t* n_positions, double* flops_per_position) {
  SPB_GUARD(e);
  SPB_ARG(e, iters > 0 && avg_ms, "bad argument");
  if (e->cfg.evaluator != SPB_EVAL_NET || !e->evaluator.loaded()) { e->set_error("needs the network evaluator with weights loaded"); return SPB_ERR_STATE; }
  const uint32_t slots = e->T.G * e->T.K;
  const uint32_t* cnt = &e->T.eval_count[2];
  const bool simt = (e->cfg.flags & SPB_FLAG_EVAL_SIMT) != 0;
  // Lock-step pipeline: the work list of the last simulation step.  Asynchronous pipeline (no step lists): the latest
  // evaluated leaf of every slot, as one static list of G positions.
  const uint32_t* list = e->T.eval_list;
  if (e->last_eval_parity < 0) {
    list = nullptr;
    SPB_CUDA(e, cudaMemcpyAsync(&e->T.eval_count[2], &slots, 4, cudaMemcpyHostToDevice, e->stream));
    SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  }
  for (int w = 0; w < 2; ++w)    // warm-up
    SPB_CUDA(e, e->evaluator.launch(e->T.leaf_state, list, cnt, slots, e->T.eval_out, e->eval_stride, nullptr, simt, e->stream, /*overlap=*/false));
  SPB_CUDA(e, cudaEventRecord(e->ev0, e->stream));
  for (uint32_t i = 0; i < iters; ++i)
    SPB_CUDA(e, e->evaluator.launch(e->T.leaf_state, list, cnt, slots, e->T.eval_out, e->eval_stride, nullptr, simt, e->stream, /*overlap=*/false));
  SPB_CUDA(e, cudaEventRecord(e->ev1, e->stream));
  uint32_t n = 0;
  SPB_CUDA(e, cudaMemcpyAsync(&n, cnt, 4, cudaMemcpyDeviceToHost, e->stream));
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  float ms = 0.f;
  SPB_CUDA(e, cudaEventElapsedTime(&ms, e->ev0, e->ev1));
  e->launches += iters + 2;
  *avg_ms = ms / (float)iters;
  if (n_positions) *n_positions = n;
  if (flops_per_position) *flops_per_position = e->evaluator.flops_per_position();
  return SPB_OK;
}

int32_t spb_last_async_stats(spb_engine* e, uint64_t* out, uint32_t n) {
  if (!e || !out) return SPB_ERR_ARG;
  for (uint32_t i = 0; i < n; ++i) out[i] = i < (uint32_t)ASTAT_COUNT ? e->last_async_stats[i] : 0;
  return SPB_OK;
}

int32_t spb_synchronize(spb_engine* e) {
  SPB_GUARD(e);
  SPB_CUDA(e, cudaStreamSynchronize(e->stream));
  return SPB_OK;
}

}  // extern "C"
