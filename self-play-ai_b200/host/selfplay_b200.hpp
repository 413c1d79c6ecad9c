// selfplay_b200.hpp — header-only C++ host mirror of the reference's search interface over the C ABI.
//
// The reference is compiled code (Rust) and no Rust toolchain exists in the build image, so the host side above
// include/selfplay_b200.h is provided in C++ with the reference's names, argument meaning and error behaviour
// (ref: src/mcts.rs:8-44, :86, :161, :196; src/game/mod.rs:9-33).  The Rust crates in rust/ are the same thing for
// cargo users.  Errors: where the reference returns Err(String) or panics, these functions throw spb::Error
// (nothing crosses the C ABI as an exception).
#pragma once
#include <algorithm>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/selfplay_b200.h"

namespace spb {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error("selfplay_b200 error " + std::to_string(c) + ": " + m), code(c) {}
};

// ref: enum Status, game/mod.rs:9-15
enum class Status : uint8_t { Ongoing = SPB_STATUS_ONGOING, Tied = SPB_STATUS_TIED, Won = SPB_STATUS_WON };

// ref: struct Args, mcts.rs:8-18 (defaults mcts.rs:46-59).  Only c (via the Tree) and num_searches are read by search.
struct Args {
  float c = 2.0f;
  uint32_t num_searches = 600;
  float temperature = 1.25f;
  uint32_t num_learn_iters = 10;
  uint32_t num_self_play_iters = 500;
  size_t num_parallel_self_play_games = 100;
  int64_t batch_size = 32;
  uint32_t num_epochs = 4;
};

// ref: the `State` values the learners read (game/mod.rs:21-33): current player, status, value_and_terminated.
struct State {
  spb_state raw{};
  int get_current_player() const { return raw.current_player; }                    // game/mod.rs:25
  Status get_status() const { return static_cast<Status>(raw.status); }            // game/mod.rs:28
  std::pair<float, bool> get_value_and_terminated() const {                        // connect_four.rs:231-240
    if (raw.status == SPB_STATUS_WON) return {-1.0f, true};
    if (raw.status == SPB_STATUS_TIED) return {0.0f, true};
    return {0.0f, false};
  }
  bool operator==(const State& o) const {
    return raw.stones[0] == o.raw.stones[0] && raw.stones[1] == o.raw.stones[1] && raw.current_player == o.raw.current_player &&
           raw.num_actions_played == o.raw.num_actions_played && raw.status == o.raw.status;
  }
};

class Mcts;

// ref: struct Tree<T>, mcts.rs:32-39 — a handle on one engine slot; histories stay on the host as in the reference.
class Tree {
 public:
  uint32_t slot;
  std::vector<State> state_history;               // mcts.rs:37
  std::vector<std::vector<float>> policy_history; // mcts.rs:38
 private:
  friend class Mcts;
  explicit Tree(uint32_t s) : slot(s) {}
};

// ref: struct Mcts<T> { args, model }, mcts.rs:41-44.  Owns the engine (node pools + evaluator weights) of one GPU.
class Mcts {
 public:
  Args args;
  Mcts(const Args& a, int game, int device = 0, int evaluator = SPB_EVAL_NET, uint32_t flags = 0) : args(a) {
    spb_config cfg;
    spb_default_config(&cfg);
    cfg.game = game; cfg.device = device; cfg.evaluator = evaluator; cfg.flags = flags; cfg.c = a.c;
    cfg.num_games = (uint32_t)a.num_parallel_self_play_games;
    actions_ = game == SPB_GAME_CONNECT4 ? 7 : 9;
    int rc = spb_create(&cfg, &e_);
    if (rc != SPB_OK) throw Error(rc, spb_last_error(nullptr));
  }
  ~Mcts() { if (e_) spb_destroy(e_); }
  Mcts(const Mcts&) = delete;
  Mcts& operator=(const Mcts&) = delete;

  // ref: VarStore::load, main.rs:61 — the bytes of the safetensors file VarStore::save wrote (learner.rs:192).
  void load_weights(const std::vector<uint8_t>& safetensors) { check(spb_load_weights(e_, safetensors.data(), safetensors.size())); }
  // The learner's device tensors, named as in the checkpoint (spb_load_weights_device); they may change once this returns.
  void load_weights_device(const std::vector<spb_tensor>& tensors) { check(spb_load_weights_device(e_, tensors.data(), (uint32_t)tensors.size())); }
  // COLLECTIVE: every rank takes root_rank's weights.
  void broadcast_weights(int32_t root_rank) { check(spb_broadcast_weights(e_, root_rank)); }

  // ref: Tree::default (mcts.rs:67) / Tree::with_root_state (mcts.rs:86)
  Tree make_tree(uint32_t slot) { check(spb_reset_games(e_, &slot, 1, nullptr)); return Tree(slot); }
  Tree with_root_state(uint32_t slot, const State& s) { check(spb_reset_games(e_, &slot, 1, &s.raw)); return Tree(slot); }

  // ref: Mcts::search, mcts.rs:196-332.  Result i belongs to trees[i]: (root visit counts scattered by action and
  // normalised, [(child arena id, visit count as f32)] in child order).
  std::vector<std::pair<std::vector<float>, std::vector<std::pair<size_t, float>>>> search(std::vector<Tree*>& trees) {
    check(spb_search(e_, args.num_searches));
    std::vector<std::pair<std::vector<float>, std::vector<std::pair<size_t, float>>>> out;
    for (Tree* t : trees) {
      uint8_t a[SPB_MAX_ACTIONS]; uint32_t c[SPB_MAX_ACTIONS], ids[SPB_MAX_ACTIONS], n = 0;
      check(spb_root_children(e_, t->slot, a, c, ids, &n));
      std::vector<float> policy(actions_, 0.0f);
      check(spb_root_policy(e_, t->slot, policy.data()));
      std::vector<std::pair<size_t, float>> pairs;
      for (uint32_t i = 0; i < n; ++i) pairs.emplace_back(ids[i], (float)c[i]);
      out.emplace_back(std::move(policy), std::move(pairs));
    }
    return out;
  }

  // ref: Tree::use_subtree, mcts.rs:161-192; returns tree.arena[0].state of the re-rooted tree.
  State use_subtree(Tree& tree, size_t new_root_id) {
    uint32_t id = (uint32_t)new_root_id;
    State s;
    check(spb_advance(e_, &tree.slot, &id, 1, &s.raw));
    return s;
  }
  // ref: tree.arena[id].state (learner_concurrent.rs:184,195; main.rs:92) and tree.arena.len()
  State node_state(const Tree& tree, size_t id) { State s; check(spb_get_state(e_, tree.slot, (uint32_t)id, &s.raw)); return s; }
  size_t arena_len(const Tree& tree) { uint32_t n = 0; check(spb_arena_len(e_, tree.slot, &n)); return n; }
  // EXTENSION (DESIGN.md §4.6): Dirichlet noise on the root priors; epsilon = 0 turns it off.
  void set_root_noise(float alpha, float epsilon, uint64_t seed) { check(spb_set_root_noise(e_, alpha, epsilon, seed)); }
  std::vector<float> root_noise(const Tree& tree) {
    float eta[SPB_MAX_ACTIONS];
    uint32_t n = 0;
    check(spb_root_noise(e_, tree.slot, eta, &n));
    return std::vector<float>(eta, eta + n);
  }
  uint8_t action_taken(const Tree& tree, size_t child_index) {     // node.action_taken of the root's child_index-th child (mcts.rs:25)
    uint8_t a[SPB_MAX_ACTIONS]; uint32_t n = 0;
    check(spb_root_children(e_, tree.slot, a, nullptr, nullptr, &n));
    if (child_index >= n) throw Error(SPB_ERR_ARG, "child index out of range");
    return a[child_index];
  }
  spb_engine* raw() { return e_; }

  // The learner hand-off in device memory.  Pointers ending in _dev are device memory of this engine's GPU (e.g. a slice
  // of a replay buffer); a null buf_dev is the size query.  Each returns the number of records held / written.
  // Finished games' positions ordered by (game id, ply), with their global game ids (game_ids_dev nullable).
  size_t drain_trajectories_device(spb_position* buf_dev, size_t capacity, uint64_t* game_ids_dev = nullptr) {
    size_t n = 0;
    check(spb_drain_trajectories_device(e_, buf_dev, capacity, &n, game_ids_dev));
    return n;
  }
  // COLLECTIVE: every rank's records to learner_rank (0 elsewhere); a null or short buffer keeps them staged on the device.
  size_t gather_trajectories_device(int32_t learner_rank, spb_position* buf_dev, size_t capacity, uint64_t* game_ids_dev = nullptr) {
    size_t n = 0;
    check(spb_gather_trajectories_device(e_, learner_rank, buf_dev, capacity, &n, game_ids_dev));
    return n;
  }
  // The training tensors of spb_positions_to_training for this engine's game, built on the device; row i from
  // positions_dev[indices_dev ? indices_dev[i] : i], each output nullable.
  void positions_to_training_device(const spb_position* positions_dev, size_t n_positions, const uint64_t* indices_dev, size_t n,
                                    float* encodings_dev, float* policies_dev, float* values_dev) {
    check(spb_positions_to_training_device(e_, positions_dev, n_positions, indices_dev, n, encodings_dev, policies_dev, values_dev));
  }

 private:
  void check(int rc) { if (rc != SPB_OK) throw Error(rc, spb_last_error(e_)); }
  spb_engine* e_ = nullptr;
  int actions_ = 7;
};

// ---- chess (ref: src/game/chess.rs, src/model/chess.rs) ---------------------------------------------------------------
// ref: chess::State {game, transposition_table, fifty_move_rule_halfmove_counter} (chess.rs:24-29): the position and, beside
// it, one hash per ply of game history.  A move is from | to << 6 | promotion << 12.
struct ChessState {
  spb_chess_state raw{};
  std::vector<uint64_t> history;                                                   // transposition_table as list hashes
  int get_current_player() const { return raw.side; }                              // chess.rs:108-110
  static ChessState start() { ChessState s; spb_chess_start_position(&s.raw); return s; }   // State::default(), chess.rs:94-102
};

class ChessTree {
 public:
  uint32_t slot;
 private:
  friend class ChessMcts;
  explicit ChessTree(uint32_t s) : slot(s) {}
};

// ref: Mcts<chess Net>, mcts.rs:41-44 over model/chess.rs.
class ChessMcts {
 public:
  Args args;
  ChessMcts(const Args& a, int device = 0, int evaluator = SPB_EVAL_NET) : args(a) {
    spb_config cfg;
    spb_default_config(&cfg);
    cfg.game = SPB_GAME_CHESS; cfg.device = device; cfg.evaluator = evaluator; cfg.c = a.c;
    cfg.num_games = (uint32_t)a.num_parallel_self_play_games;
    int rc = spb_chess_create(&cfg, &e_);
    if (rc != SPB_OK) throw Error(rc, spb_chess_last_error(nullptr));
  }
  ~ChessMcts() { if (e_) spb_chess_destroy(e_); }
  ChessMcts(const ChessMcts&) = delete;
  ChessMcts& operator=(const ChessMcts&) = delete;

  void load_weights(const std::vector<uint8_t>& safetensors) { check(spb_chess_load_weights(e_, safetensors.data(), safetensors.size())); }
  void load_weights_device(const std::vector<spb_tensor>& tensors) { check(spb_chess_load_weights_device(e_, tensors.data(), (uint32_t)tensors.size())); }
  void broadcast_weights(int32_t root_rank) { check(spb_chess_broadcast_weights(e_, root_rank)); }
  // ref: Tree::with_root_state, mcts.rs:86
  ChessTree with_root_state(uint32_t slot, const ChessState& s) {
    std::vector<uint64_t> h(SPB_CHESS_MAX_HISTORY, 0);
    for (size_t i = 0; i < s.history.size() && i < h.size(); ++i) h[i] = s.history[i];
    spb_chess_state st = s.raw;
    st.hist_len = (uint32_t)std::min<size_t>(s.history.size(), SPB_CHESS_MAX_HISTORY);
    check(spb_chess_reset_games(e_, &slot, 1, &st, h.data()));
    return ChessTree(slot);
  }
  // get_valid_actions / get_status (chess.rs:150-166) of one state
  std::vector<uint16_t> get_valid_actions(const ChessState& s, Status* status = nullptr) {
    std::vector<uint64_t> h(SPB_CHESS_MAX_HISTORY, 0);
    for (size_t i = 0; i < s.history.size() && i < h.size(); ++i) h[i] = s.history[i];
    std::vector<uint16_t> mv(SPB_CHESS_MAX_MOVES);
    uint32_t n = 0; uint8_t st = 0;
    spb_chess_state raw = s.raw;
    raw.hist_len = (uint32_t)std::min<size_t>(s.history.size(), SPB_CHESS_MAX_HISTORY);
    check(spb_chess_legal_moves(e_, &raw, h.data(), 1, mv.data(), &n, nullptr, &st, nullptr));
    mv.resize(n);
    if (status) *status = static_cast<Status>(st);
    return mv;
  }
  uint64_t perft(const ChessState& s, uint32_t depth) { uint64_t n = 0; check(spb_chess_perft(e_, &s.raw, depth, &n)); return n; }
  // EXTENSION (DESIGN.md §4.6): Dirichlet noise on the root priors, as Mcts::set_root_noise.
  void set_root_noise(float alpha, float epsilon, uint64_t seed) { check(spb_chess_set_root_noise(e_, alpha, epsilon, seed)); }
  std::vector<float> root_noise(const ChessTree& tree) {
    std::vector<float> eta(SPB_CHESS_MAX_MOVES);
    uint32_t n = 0;
    check(spb_chess_root_noise(e_, tree.slot, eta.data(), &n));
    eta.resize(n);
    return eta;
  }
  // ref: Mcts::search, mcts.rs:196-332: per tree [(child arena id, visit count)] with the children's moves.
  struct Result { std::vector<uint16_t> moves; std::vector<std::pair<size_t, float>> child_id_to_probs; };
  std::vector<Result> search(std::vector<ChessTree*>& trees) {
    check(spb_chess_search(e_, args.num_searches));
    std::vector<Result> out;
    for (ChessTree* t : trees) {
      std::vector<uint16_t> mv(SPB_CHESS_MAX_MOVES);
      std::vector<uint32_t> cnt(SPB_CHESS_MAX_MOVES), ids(SPB_CHESS_MAX_MOVES);
      uint32_t n = 0;
      check(spb_chess_root_children(e_, t->slot, mv.data(), cnt.data(), ids.data(), &n));
      Result r;
      r.moves.assign(mv.begin(), mv.begin() + n);
      for (uint32_t i = 0; i < n; ++i) r.child_id_to_probs.emplace_back(ids[i], (float)cnt[i]);
      out.push_back(std::move(r));
    }
    return out;
  }
  // ref: Tree::use_subtree, mcts.rs:161-192 (a child of the root); returns the new root position.
  spb_chess_state use_subtree(ChessTree& tree, size_t child_id) {
    uint32_t id = (uint32_t)child_id;
    spb_chess_state s{};
    check(spb_chess_advance(e_, &tree.slot, &id, 1, &s));
    return s;
  }
  size_t arena_len(const ChessTree& tree) { uint32_t n = 0; check(spb_chess_arena_len(e_, tree.slot, &n)); return n; }

  // ref: learner_concurrent.rs:179-238 — one self-play ply for every live game on the device (rule SPB_MOVE_*); finished
  // slots restart from restart_roots[slot] (num_parallel_self_play_games entries) or retire.  Returns the games finished.
  // Throws Error(SPB_ERR_STATE) when the trajectory buffer is full: drain and call again, nothing is lost.
  uint32_t self_play_step(int rule, float temperature, uint64_t seed, const std::vector<ChessState>* restart_roots = nullptr) {
    std::vector<spb_chess_state> roots;
    std::vector<uint64_t> hist;
    if (restart_roots) {
      for (const ChessState& s : *restart_roots) {
        spb_chess_state st = s.raw;
        st.hist_len = (uint32_t)std::min<size_t>(s.history.size(), SPB_CHESS_MAX_HISTORY);
        roots.push_back(st);
        std::vector<uint64_t> h(SPB_CHESS_MAX_HISTORY, 0);
        std::copy(s.history.begin(), s.history.begin() + st.hist_len, h.begin());
        hist.insert(hist.end(), h.begin(), h.end());
      }
    }
    uint32_t finished = 0;
    check(spb_chess_selfplay_step(e_, rule, temperature, seed, restart_roots ? roots.data() : nullptr, restart_roots ? hist.data() : nullptr,
                                  &finished));
    return finished;
  }
  // Finished games' positions ordered by (game id, ply), with their global game ids.
  std::pair<std::vector<spb_chess_position>, std::vector<uint64_t>> drain_trajectories() {
    size_t n = 0;
    check(spb_chess_drain_trajectories(e_, nullptr, 0, &n, nullptr));
    std::vector<spb_chess_position> pos(n);
    std::vector<uint64_t> ids(n);
    if (n) check(spb_chess_drain_trajectories(e_, pos.data(), n, &n, ids.data()));
    pos.resize(n);
    ids.resize(n);
    return {std::move(pos), std::move(ids)};
  }
  // The device forms (as Mcts::drain_trajectories_device / gather_trajectories_device), chess records.
  size_t drain_trajectories_device(spb_chess_position* buf_dev, size_t capacity, uint64_t* game_ids_dev = nullptr) {
    size_t n = 0;
    check(spb_chess_drain_trajectories_device(e_, buf_dev, capacity, &n, game_ids_dev));
    return n;
  }
  size_t gather_trajectories_device(int32_t learner_rank, spb_chess_position* buf_dev, size_t capacity, uint64_t* game_ids_dev = nullptr) {
    size_t n = 0;
    check(spb_chess_gather_trajectories_device(e_, learner_rank, buf_dev, capacity, &n, game_ids_dev));
    return n;
  }
  // The training tensors of chess records (host only): encodings [n][19][8][8], policies [n][4672], values [n].
  struct TrainingBatch { std::vector<float> encodings, policies, values; };
  static TrainingBatch positions_to_training(const std::vector<spb_chess_position>& positions) {
    const size_t n = positions.size();
    TrainingBatch b{std::vector<float>(n * SPB_CHESS_PLANES * 64), std::vector<float>(n * SPB_CHESS_POLICY_SIZE), std::vector<float>(n)};
    const int rc = spb_chess_positions_to_training(positions.data(), n, b.encodings.data(), b.policies.data(), b.values.data());
    if (rc != SPB_OK) throw Error(rc, "spb_chess_positions_to_training: bad argument");
    return b;
  }

 private:
  void check(int rc) { if (rc != SPB_OK) throw Error(rc, spb_chess_last_error(e_)); }
  spb_chess_engine* e_ = nullptr;
};

}  // namespace spb
