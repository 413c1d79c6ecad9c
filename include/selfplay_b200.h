/*
 * selfplay_b200.h — C ABI of the B200-native self-play engine.
 *
 * This is the drop-in boundary for the reference's self-play hot path
 * (joshua16266261/self-play-ai): src/mcts.rs (Mcts::search, Tree, use_subtree),
 * src/game/{mod,connect_four,tictactoe}.rs (State / Policy traits) and
 * src/model/mod.rs (Model::predict / Net::forward).  The reference has no FFI
 * of its own (100 % safe Rust); a Rust `-sys` crate binds exactly these symbols
 * (see INTEGRATION.md and rust/selfplay-b200-sys/).  Every entry point cites the
 * reference interface it replaces as `ref: file:line`.
 *
 * Conventions
 *   - every function returns int32_t: 0 = SPB_OK, negative = error.  The text of
 *     the last error on a handle is spb_last_error(handle) (spb_last_error(NULL)
 *     returns the text of the last spb_create failure on this thread).
 *   - no panics / aborts cross the ABI; node-pool exhaustion is SPB_ERR_POOL.
 *   - the caller owns every buffer it passes; pointers are HOST pointers unless
 *     the parameter name ends in `_dev`.
 *   - a handle is NOT thread-safe: one handle per host thread per GPU, which is
 *     how the reference uses one `Mcts` per worker thread (ref: main.rs:169).
 *   - there is no CPU fallback: spb_create fails with SPB_ERR_CUDA when no
 *     sm_100 device is present.
 */
#ifndef SELFPLAY_B200_H
#define SELFPLAY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPB_ABI_VERSION 2

/* ---- status codes ------------------------------------------------------- */
#define SPB_OK             0
#define SPB_ERR_ARG       -1   /* bad argument (null pointer, slot out of range, ...) */
#define SPB_ERR_CUDA      -2   /* CUDA runtime error / no sm_100 device */
#define SPB_ERR_POOL      -3   /* a tree's node pool is full and cannot grow (SPB_FLAG_FIXED_POOL, HBM, 2^24) */
#define SPB_ERR_ILLEGAL   -4   /* illegal move / game already ended (ref: connect_four.rs:193,209) */
#define SPB_ERR_WEIGHTS   -5   /* weight blob malformed / tensor missing / shape mismatch */
#define SPB_ERR_STATE     -6   /* call not valid in the engine's current state */
#define SPB_ERR_NOMEM     -7   /* host or device allocation failed */

/* ---- games (ref: src/game/mod.rs:1-3) ----------------------------------- */
#define SPB_GAME_TICTACTOE 0   /* ref: src/game/tictactoe.rs   A = 9, board 3x3 */
#define SPB_GAME_CONNECT4  1   /* ref: src/game/connect_four.rs A = 7, board 6x7 */
#define SPB_MAX_ACTIONS    9

/* ---- Status (ref: src/game/mod.rs:9-15) --------------------------------- */
#define SPB_STATUS_ONGOING 0
#define SPB_STATUS_TIED    1
#define SPB_STATUS_WON     2

/* ---- evaluators --------------------------------------------------------- */
#define SPB_EVAL_NET       0   /* fused bf16 tcgen05 conv ResNet (ref: model/connect_four.rs:50-81) */
#define SPB_EVAL_DET       1   /* deterministic hash evaluator, SURVEY.md §8(c) — parity harness */
#define SPB_EVAL_UNIFORM   2   /* raw p = 1.0 for every action, v = 0 — parity harness */

/*
 * A game position.  Replaces `State` (ref: connect_four.rs:20-26, tictactoe.rs:20-26):
 * board + current_player + num_actions_played + status.
 *   Connect4   : bit (col*7 + row) of stones[p], row 0 = bottom (ref: connect_four.rs:17-18, :52-65)
 *   Tic-tac-toe: bit (row*3 + col) of stones[p]
 * stones[0] = Player::X (moves first), stones[1] = Player::O.
 */
typedef struct spb_state {
  uint64_t stones[2];
  uint8_t  current_player;      /* 0 = X, 1 = O        (ref: connect_four.rs:23)  */
  uint8_t  num_actions_played;  /*                     (ref: connect_four.rs:24)  */
  uint8_t  status;              /* SPB_STATUS_*        (ref: connect_four.rs:25)  */
  uint8_t  reserved[5];         /* must be zero */
} spb_state;

/*
 * Engine configuration.  Mirrors the fields of `Args` that the hot path reads
 * (ref: mcts.rs:8-18): `c` (read from the Tree, mcts.rs:99, default 2.0 mcts.rs:49).
 * `num_searches` is an argument of spb_search.
 */
typedef struct spb_config {
  uint32_t abi_version;          /* SPB_ABI_VERSION */
  int32_t  game;                 /* SPB_GAME_* */
  int32_t  device;               /* CUDA device ordinal */
  uint32_t num_games;            /* G: concurrent trees ("slots"); ref: mcts.rs:54 num_parallel_self_play_games */
  uint32_t max_nodes_per_tree;   /* initial arena capacity per tree; 0 = default (16384); grows on demand */
  uint32_t leaves_per_tree;      /* K in-flight leaves per tree per step (1..16); 1 = the reference algorithm.
                                    K > 1 is an EXTENSION (virtual loss, defined in DESIGN.md §4.4): not in the reference */
  float    c;                    /* PUCT constant; ref: mcts.rs:49 (2.0) */
  int32_t  evaluator;            /* SPB_EVAL_* */
  uint32_t flags;                /* SPB_FLAG_* */
  uint32_t game_id_base;         /* id of slot 0's first self-play game (rank offset when games are sharded over GPUs) */
  uint32_t game_id_stride;       /* id increment when a slot starts its next game; 0 = num_games */
  uint32_t trajectory_capacity;  /* records of the finished-trajectory buffer drained by spb_drain_trajectories;
                                    0 = default (4 * num_games * max plies, at most 2^26) */
  uint32_t reserved[4];          /* must be zero */
} spb_config;

#define SPB_FLAG_NO_GRAPH   1u   /* launch kernels directly instead of through a CUDA graph */
#define SPB_FLAG_EVAL_SIMT  2u   /* use the CUDA-core evaluator kernel instead of tcgen05 (debug / cross-check) */
#define SPB_FLAG_LOCKSTEP   32u  /* network evaluator: run the reference's loop literally — per simulation step one evaluator
                                    launch for the leaves of all trees, then one tree-step launch (mcts.rs:214-286) — instead of
                                    the asynchronous pipeline (DESIGN.md §4.2), whose results are bit-identical.  Chess engine:
                                    one lock-step loop over all trees instead of two half-loops on two streams (DESIGN.md §4.5) */
#define SPB_FLAG_FIXED_POOL 16u  /* never grow the node pools: a tree that would pass max_nodes_per_tree makes spb_search return
                                    SPB_ERR_POOL.  Without the flag the pools grow before a search that could outgrow them, like
                                    the reference's Vec arena (mcts.rs:19) */
#define SPB_FLAG_FORCE_SPLIT 4u  /* run DetEval / uniform through the pipeline of the network evaluator (asynchronous, or lock-step
                                    with SPB_FLAG_LOCKSTEP) instead of the fused single-kernel search: parity harness */

typedef struct spb_engine spb_engine;

/* Exact integer counters; feed the roofline formulas of SURVEY.md §8(d). */
typedef struct spb_counters {
  uint64_t simulations;          /* iterations of mcts.rs:214 summed over trees */
  uint64_t evaluations;          /* leaves sent to the evaluator (mcts.rs:268) */
  uint64_t terminal_leaves;      /* simulations that ended on a terminal node (mcts.rs:245) */
  uint64_t path_length_sum;      /* sum over simulations of select() calls (mcts.rs:239-241) */
  uint64_t children_created;     /* nodes appended by expand (mcts.rs:116-143) */
  uint64_t nodes_live;           /* sum of arena lengths over slots, now */
  uint64_t kernel_launches;      /* kernels of this library launched since create/reset_counters */
  uint64_t reserved[5];
} spb_counters;

/* ---- lifecycle ---------------------------------------------------------- */

/* Fill `cfg` with defaults: Connect4, device 0, 100 games (mcts.rs:54), c = 2.0, K = 1, SPB_EVAL_NET. */
int32_t spb_default_config(spb_config* cfg);

/* ref: Mcts{args, model} construction, main.rs:43-44 / learner_concurrent.rs:30-34. */
int32_t spb_create(const spb_config* cfg, spb_engine** out);
int32_t spb_destroy(spb_engine* e);
const char* spb_last_error(const spb_engine* e);
int32_t spb_abi_version(void);

/* ---- weights (ref: VarStore::save learner.rs:192, ::load main.rs:61) ----- */

/*
 * Load a safetensors blob exported from the reference's VarStore.  BatchNorm (eval
 * mode, eps 1e-5) is folded into the preceding conv, weights are cast to bf16 and
 * packed into the evaluator's shared-memory layout.  Tensors are matched by
 * creation order of model/connect_four.rs:50-73 (see INTEGRATION.md for the name table).
 */
int32_t spb_load_weights(spb_engine* e, const void* safetensors_blob, size_t num_bytes);

/*
 * Host-only validation of a checkpoint (no GPU needed): parses the blob for `game` exactly like
 * spb_load_weights and reports SPB_OK or SPB_ERR_WEIGHTS with the reason in err[0..err_cap).
 */
int32_t spb_check_weights(int32_t game, const void* safetensors_blob, size_t num_bytes, char* err, size_t err_cap);

/*
 * Weights straight from a learner's device tensors, with no file in between.  One table entry per tensor, named by either
 * scheme spb_load_weights accepts (explicit names, or the tch VarStore names that VarStore::variables() returns, e.g.
 * "weight__12"); tensors no role needs are ignored, as in a blob.  data is device memory of the engine's GPU (or managed
 * memory), contiguous, row-major, aligned to its element size.  The accepted dtypes are those of the blob: F32, BF16, F64
 * (SPB_DTYPE_F16 is rejected with the blob's message).
 */
#define SPB_DTYPE_F32  0
#define SPB_DTYPE_BF16 1
#define SPB_DTYPE_F64  2
#define SPB_DTYPE_F16  3
typedef struct spb_tensor {
  const char* name;
  const void* data;
  int32_t dtype;                 /* SPB_DTYPE_* */
  int32_t ndim;                  /* 0..4 */
  int64_t shape[4];
} spb_tensor;                    /* 56 bytes */
/*
 * BatchNorm is folded and the image packed on the device, byte for byte the image spb_load_weights writes for the same
 * tensors.  Ordering: the caller has finished writing the tensors before the call (e.g. a stream synchronisation); the call
 * synchronises the engine's stream before it returns, after which it no longer reads them (the next optimizer step may
 * update them in place).  Names, shapes, dtypes and pointers are checked before anything is written: a bad table returns
 * SPB_ERR_WEIGHTS (as the blob would) or SPB_ERR_ARG (NULL table or name, ndim outside 0..4, a pointer that is not device
 * memory of the engine's GPU or is misaligned) and leaves the loaded net as it was.  The image is rewritten in place (no
 * device allocation after the engine's first load); a CUDA error while writing it leaves the engine without weights.
 */
int32_t spb_load_weights_device(spb_engine* e, const spb_tensor* tensors, uint32_t n);

/* ---- trees (ref: Tree::default mcts.rs:67, Tree::with_root_state mcts.rs:86) ---- */

/*
 * (Re)start the trees in `slots[0..n)` from `roots[i]`; roots == NULL means the
 * default state (empty board, X to move).  slots == NULL means slots 0..n-1.
 */
int32_t spb_reset_games(spb_engine* e, const uint32_t* slots, uint32_t n, const spb_state* roots);

/*
 * ref: Mcts::search mcts.rs:196-332.  Runs `num_searches` lock-step simulations
 * (mcts.rs:214) for every slot.  Statistics accumulate on top of whatever the tree
 * already holds (subtree reuse, mcts.rs:161-192).
 */
int32_t spb_search(spb_engine* e, uint32_t num_searches);

/*
 * ref: mcts.rs:310-331 — the second element of search()'s result for one tree:
 * for each root child in child (= legal action) order: action taken, visit count,
 * arena id.  Any output pointer may be NULL.  Arrays need SPB_MAX_ACTIONS entries.
 */
int32_t spb_root_children(spb_engine* e, uint32_t slot, uint8_t* actions,
                          uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children);

/*
 * Batched form for all G slots in one device->host copy.  Row i belongs to slot i;
 * visit_counts / child_ids are [G][SPB_MAX_ACTIONS] indexed by CHILD ORDER,
 * actions likewise; n_children is [G].
 */
int32_t spb_root_children_all(spb_engine* e, uint8_t* actions, uint32_t* visit_counts,
                              uint32_t* child_ids, uint32_t* n_children);

/*
 * ref: mcts.rs:315-328 — the first element of search()'s result: root child visit
 * counts scattered by action then divided by their sum (f32).  `policy` has A floats
 * (7 for Connect4, 9 for tic-tac-toe, row-major).
 */
int32_t spb_root_policy(spb_engine* e, uint32_t slot, float* policy);

/*
 * ref: Tree::use_subtree mcts.rs:161-192.  Re-roots slot[i] at arena node
 * node_ids[i] (BFS compaction that keeps visit_count / value_sum / prior and child
 * order).  out_states (nullable) receives the new root state of each slot.
 */
int32_t spb_advance(spb_engine* e, const uint32_t* slots, const uint32_t* node_ids,
                    uint32_t n, spb_state* out_states);

/* ref: `tree.arena[id].state` (learner_concurrent.rs:184,195; main.rs:92). */
int32_t spb_get_state(spb_engine* e, uint32_t slot, uint32_t node_id, spb_state* out);

/* ref: `tree.arena.len()`; also the per-node statistics the reference keeps private (mcts.rs:26-29). */
int32_t spb_arena_len(spb_engine* e, uint32_t slot, uint32_t* out);
int32_t spb_node_stats(spb_engine* e, uint32_t slot, uint32_t node_id, uint32_t* visit_count,
                       float* value_sum, float* prior, uint32_t* first_child, uint32_t* n_children);

/* EXTENSION (not in the reference, mcts.rs:204-207 is a TODO): Dirichlet noise on the root priors; DESIGN.md §4.6.
 * epsilon = 0 disables it (the default); otherwise 0 < epsilon <= 1 and alpha finite > 0, else SPB_ERR_ARG.
 * Only the PUCT score of the root's children sees P' = (1 - epsilon) * P + epsilon * eta; stored priors never change.
 * eta is a pure function of (seed, game id, root ply, number of root children). */
int32_t spb_set_root_noise(spb_engine* e, float alpha, float epsilon, uint64_t seed);
/* The eta the next search of `slot`'s current root uses (drawn if needed): eta[SPB_MAX_ACTIONS] in child order,
 * *n = number of root children.  SPB_ERR_STATE while noise is off. */
int32_t spb_root_noise(spb_engine* e, uint32_t slot, float* eta, uint32_t* n);

/* ---- evaluator at the predict boundary (ref: Model::predict model/mod.rs:36-98) ---- */

/*
 * Evaluates `n` states: policies[n][A] = softmax(logits) masked by legal moves and
 * renormalised (connect_four.rs:261-279), values[n].  With SPB_EVAL_NET this is the
 * fused conv ResNet; raw_logits (nullable, [n][A]) receives the pre-softmax logits
 * (Net::forward, model/connect_four.rs:75-81).
 */
int32_t spb_predict(spb_engine* e, const spb_state* states, uint32_t n,
                    float* policies, float* values, float* raw_logits);

/* ---- game rules, batched on the device (ref: State trait game/mod.rs:21-33) ---- */

/* get_next_state (connect_four.rs:190-211 / tictactoe.rs:135-167).  err[i] = 0 or SPB_ERR_ILLEGAL. */
int32_t spb_game_next_states(spb_engine* e, const spb_state* states, const uint8_t* actions,
                             uint32_t n, spb_state* out_states, int32_t* err);
/* get_valid_actions (connect_four.rs:213-225): bit a of masks[i] set = action a legal. */
int32_t spb_game_valid_actions(spb_engine* e, const spb_state* states, uint32_t n, uint32_t* masks);
/* get_encoding (connect_four.rs:242-259): out[n][3][rows][cols] f32. */
int32_t spb_game_encode(spb_engine* e, const spb_state* states, uint32_t n, float* out);

/* ---- self-play driver (ref: SelfPlayWorker::self_play learner_concurrent.rs:169-242) ---- */

#define SPB_MOVE_GREEDY_LAST_MAX 0  /* ref: main.rs:108-112 (arg-max visit count, last max wins) */
#define SPB_MOVE_TEMPERATURE     1  /* ref: learner_concurrent.rs:189-194 (sample ∝ N^temperature), counter-based RNG */

/* One position record of a finished trajectory (compact form of `Payload`, learner_concurrent.rs:13-18). */
typedef struct spb_position {
  uint64_t stones[2];            /* position the search was run from (root state) */
  uint32_t visit_counts[SPB_MAX_ACTIONS]; /* root child visit counts scattered BY ACTION (policy target before normalising) */
  uint8_t  current_player;
  uint8_t  ply;                  /* index of this position inside its game */
  int8_t   outcome;              /* value target for this position: +1 / 0 / -1 (learner_concurrent.rs:214-226) */
  uint8_t  reserved;
} spb_position;                  /* 56 bytes */

/*
 * One self-play ply for every live slot, entirely on the device: pick a child of
 * the root by `rule`, record (root state, visit counts), then either finish the
 * game (terminal child: emit the trajectory with outcomes, restart the slot from
 * a fresh root if `restart_roots` != NULL, else leave it idle) or re-root
 * (use_subtree).  `seed` feeds the counter-based RNG of SPB_MOVE_TEMPERATURE.
 * n_finished (nullable) receives the number of games whose trajectory was emitted in this call.
 * When the trajectory buffer cannot take a finished game the call returns SPB_ERR_STATE: nothing is lost or
 * half-written — the game's slot is parked (idle, skipped by spb_search) with its history kept; drain with
 * spb_drain_trajectories and carry on: the next spb_selfplay_step emits the parked games first.
 */
int32_t spb_selfplay_step(spb_engine* e, int32_t rule, float temperature, uint64_t seed,
                          const spb_state* restart_roots, uint32_t* n_finished);

/* Copies finished positions (ordered by game sequence number, then ply) to `buf`. */
int32_t spb_drain_trajectories(spb_engine* e, spb_position* buf, size_t capacity, size_t* written,
                               uint64_t* game_ids /* nullable, [capacity] global game id per position */);
/*
 * The learner hand-off in device memory: the records spb_drain_trajectories returns, byte for byte and in the same order,
 * written to buf_dev (e.g. a slice of a replay buffer on the GPU) and game_ids_dev (nullable).  buf_dev == NULL: size
 * query, *written = the number held.  capacity < *written is SPB_ERR_ARG and nothing is drained.  When there are records
 * to write, buf_dev and game_ids_dev must be device (or managed) memory of e's GPU, 8-byte aligned, else SPB_ERR_ARG naming
 * the argument and nothing is drained.  The records are ordered on the device
 * (whole trajectories are moved as runs); scratch comes from the engine's grow-only staging.  Enqueued on the engine's
 * stream; returns once the outputs are written.
 */
int32_t spb_drain_trajectories_device(spb_engine* e, spb_position* buf_dev, size_t capacity, size_t* written,
                                      uint64_t* game_ids_dev /* nullable */);

/* ---- chess (ref: src/game/chess.rs, src/model/chess.rs; BASELINE config 5) ------------------------------------------ */
/*
 * The chess engine is a handle type of its own: `Mcts<chess Net>` + its `Vec<Tree<chess::State>>` on one GPU.  It is
 * created from the same spb_config with game = SPB_GAME_CHESS (leaves_per_tree must be 1; max_nodes_per_tree 0 = 32,768).
 * Everything the reference computes itself is reproduced exactly; what it delegates to the un-vendored crate `chess 3.2.0`
 * — the ORDER of the legal moves, hence of a node's children — is defined here as sorted by (from, to, promotion):
 * PARITY UNPINNED for that order (DESIGN.md §2); the legal-move SETS are pinned by the published perft counts.
 */
#define SPB_GAME_CHESS         2
#define SPB_CHESS_MAX_MOVES    256    /* capacity of a legal-move list (218 is the known maximum) */
#define SPB_CHESS_MAX_HISTORY  512    /* plies of game history a state may carry (repetition rule, chess.rs:51-62) */
#define SPB_CHESS_PLANES       19     /* get_encoding, chess.rs:176-249 */
#define SPB_CHESS_POLICY_SIZE  4672   /* 73 move planes x 8 x 8, chess.rs:311-493 */
#define SPB_CHESS_NO_SQUARE    64

typedef struct spb_chess_engine spb_chess_engine;

/*
 * A chess position.  Replaces `State{game, transposition_table, fifty_move_rule_halfmove_counter}` (chess.rs:24-29):
 * bitboards with square = rank*8 + file (a1 = 0, h8 = 63, as Square::to_index of the `chess` crate); the game history the
 * repetition rule needs travels beside the state as one 64-bit hash per ply (history[i] = hash of the legal-move list of
 * the position before ply i; the reference compares those lists, chess.rs:51-62,121-122).
 * A move is uint16: from | to << 6 | promotion << 12 (0 none, 1 knight, 2 bishop, 3 rook, 4 queen).
 */
typedef struct spb_chess_state {
  uint64_t piece[6];             /* pawns, knights, bishops, rooks, queens, kings (both colours) */
  uint64_t color[2];             /* white, black */
  uint8_t  side;                 /* side to move: 0 white, 1 black */
  uint8_t  castle;               /* bit 0 white king side, 1 white queen side, 2 black king side, 3 black queen side */
  uint8_t  ep;                   /* en-passant target square or SPB_CHESS_NO_SQUARE */
  uint8_t  reserved0;
  uint16_t fifty;                /* fifty_move_rule_halfmove_counter (chess.rs:124-143) */
  uint16_t plies;                /* moves played in the game (get_encoding plane 18) */
  uint32_t hist_len;             /* plies of history that travel with this state (<= SPB_CHESS_MAX_HISTORY) */
  uint32_t reserved1;
} spb_chess_state;               /* 80 bytes */

/* lifecycle (ref: Mcts{args, model} construction, main.rs:43-44); errors as for spb_create, text via spb_chess_last_error(NULL) */
int32_t spb_chess_create(const spb_config* cfg, spb_chess_engine** out);
int32_t spb_chess_destroy(spb_chess_engine* e);
const char* spb_chess_last_error(const spb_chess_engine* e);
/* VarStore::load (main.rs:61) for model/chess.rs:50-73: safetensors bytes, BatchNorm folded, bf16 packed for tcgen05. */
int32_t spb_chess_load_weights(spb_chess_engine* e, const void* blob, size_t n);
int32_t spb_chess_check_weights(const void* blob, size_t n, char* err, size_t err_cap);   /* host only */
/* spb_load_weights_device for the chess net (the names of spb_chess_load_weights); the network is created on first use. */
int32_t spb_chess_load_weights_device(spb_chess_engine* e, const spb_tensor* tensors, uint32_t n);

/* State::default(), chess.rs:94-102 (host only). */
int32_t spb_chess_start_position(spb_chess_state* out);
/*
 * get_valid_actions (chess.rs:150-152) + get_status (:154-166) for n states in one kernel.  history is [n][SPB_CHESS_MAX_HISTORY]
 * (nullable when every hist_len is 0).  Outputs (each nullable): moves[n][SPB_CHESS_MAX_MOVES] sorted by (from, to, promotion),
 * counts[n], policy_index[n][SPB_CHESS_MAX_MOVES] = position of each move in the flat 73x8x8 policy (Policy::get_prob,
 * chess.rs:495-502), status[n] (SPB_STATUS_*; Won = the side to move is checkmated, value +1.0 by chess.rs:172),
 * repetitions[n] (get_num_repetitions, chess.rs:51-62).
 */
int32_t spb_chess_legal_moves(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, uint16_t* moves,
                              uint32_t* counts, uint16_t* policy_index, uint8_t* status, uint32_t* repetitions);
/*
 * get_next_state (chess.rs:112-148).  err[i] = SPB_OK, or SPB_ERR_ILLEGAL (move not legal / game already over: the state
 * is copied unchanged), or SPB_ERR_STATE (history full).  history (nullable only if no state moves) is updated in place:
 * the hash of the legal-move list of states[i] is appended and out_states[i].hist_len = hist_len + 1.
 */
int32_t spb_chess_next_states(spb_chess_engine* e, const spb_chess_state* states, uint64_t* history, const uint16_t* moves, uint32_t n,
                              spb_chess_state* out_states, int32_t* err);
/* get_encoding (chess.rs:176-249): out[n][19][8][8] f32. */
int32_t spb_chess_encode(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, float* out);
/* perft(depth) of one position on the device (the standard move-generator test): leaf count of the legal-move tree. */
int32_t spb_chess_perft(spb_chess_engine* e, const spb_chess_state* state, uint32_t depth, uint64_t* nodes);
/* Policy::get_channel (chess.rs:311-390), the flat policy index, Policy::get_action (:392-493, 0xFFFF = off the board): host only. */
int32_t spb_chess_move_channel(int32_t side, uint16_t move);
int32_t spb_chess_policy_index(int32_t side, uint16_t move);
uint16_t spb_chess_action(int32_t side, int32_t channel, int32_t row, int32_t col);

/* Tree::with_root_state (mcts.rs:86-89) for n slots (slots NULL = 0..n-1; roots NULL = the start position; history
 * [n][SPB_CHESS_MAX_HISTORY], NULL = games that start at their root). */
int32_t spb_chess_reset_games(spb_chess_engine* e, const uint32_t* slots, uint32_t n, const spb_chess_state* roots, const uint64_t* history);
/* Mcts::search (mcts.rs:196-332): num_searches simulations for every live tree.  SPB_EVAL_NET runs the reference's loop
 * literally — per simulation one select over all trees, one network batch, one expand + backup. */
int32_t spb_chess_search(spb_chess_engine* e, uint32_t num_searches);
int32_t spb_chess_last_search_ms(spb_chess_engine* e, float* ms);   /* device time of the last spb_chess_search */
/* Result of search for one tree / all trees (mcts.rs:315-328), child order: moves, visit counts, arena ids; arrays of
 * SPB_CHESS_MAX_MOVES entries per tree. */
int32_t spb_chess_root_children(spb_chess_engine* e, uint32_t slot, uint16_t* moves, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children);
int32_t spb_chess_root_children_all(spb_chess_engine* e, uint16_t* moves, uint32_t* visit_counts, uint32_t* child_ids, uint32_t* n_children);
/* The Policy half of the result: visit counts scattered by set_prob and normalised, out[SPB_CHESS_POLICY_SIZE]. */
int32_t spb_chess_root_policy(spb_chess_engine* e, uint32_t slot, float* out);
/* Tree::use_subtree(child id) (mcts.rs:161-192) for n trees; the root position advances, the game history grows by one
 * ply.  out_states (nullable) receives the new root states.  SPB_ERR_ARG if an id is not a child of its root. */
int32_t spb_chess_advance(spb_chess_engine* e, const uint32_t* slots, const uint32_t* child_ids, uint32_t n, spb_chess_state* out_states);
/* arena[node_id].state (mcts.rs:22). */
int32_t spb_chess_get_state(spb_chess_engine* e, uint32_t slot, uint32_t node_id, spb_chess_state* out);
int32_t spb_chess_arena_len(spb_chess_engine* e, uint32_t slot, uint32_t* out);
/* Node fields (mcts.rs:20-30); status = SPB_STATUS_* (Ongoing until the node has been reached as a leaf). */
int32_t spb_chess_node_stats(spb_chess_engine* e, uint32_t slot, uint32_t node_id, uint32_t* visit_count, float* value_sum, float* prior,
                             uint32_t* first_child, uint32_t* n_children, uint16_t* move, uint8_t* status);
/* EXTENSION: spb_set_root_noise / spb_root_noise for chess trees (DESIGN.md §4.6).  The eta buffer (SPB_CHESS_MAX_MOVES floats
 * per game) is allocated by the first call with epsilon > 0.  The game id is spb_config.game_id_base + slot until the first
 * self-play step, then the slot's current game id; the root ply is spb_chess_state.plies. */
int32_t spb_chess_set_root_noise(spb_chess_engine* e, float alpha, float epsilon, uint64_t seed);
int32_t spb_chess_root_noise(spb_chess_engine* e, uint32_t slot, float* eta /* [SPB_CHESS_MAX_MOVES] */, uint32_t* n);
/* Model::predict (model/mod.rs:36-98): policies[n][4672] = softmax masked to the legal moves and renormalised
 * (chess.rs:251-271), values[n], raw_logits[n][4672] (each nullable).  n <= num_games. */
int32_t spb_chess_predict(spb_chess_engine* e, const spb_chess_state* states, const uint64_t* history, uint32_t n, float* policies, float* values,
                          float* raw_logits);
/*
 * Re-runs the dominant kernel — one 256 -> 256 3x3 residual convolution over the evaluator batch of the most recent
 * spb_chess_search, still resident in HBM — `iters` times between CUDA events on the engine's stream: average launch
 * duration, positions in the batch, algorithmic FLOPs of one launch (2*MAC) and of a whole network evaluation per position.
 * Used by bench.py for the tensor roofline.
 */
int32_t spb_chess_time_conv(spb_chess_engine* e, uint32_t iters, float* avg_ms, uint32_t* n_positions, double* flops_per_launch,
                            double* flops_per_position);
int32_t spb_chess_get_counters(spb_chess_engine* e, spb_counters* out);   /* reserved[0] = largest arena */
int32_t spb_chess_reset_counters(spb_chess_engine* e);

/* ---- chess self-play driver (ref: SelfPlayWorker::self_play learner_concurrent.rs:169-242, over chess::State) --------------
 * The contract of spb_selfplay_step / spb_drain_trajectories for chess trees.  spb_config.game_id_base, game_id_stride and
 * trajectory_capacity take effect as for the Connect4 engine (capacity 0 = 4 * num_games * SPB_CHESS_MAX_HISTORY records, at
 * most 2^26; never less than one whole game, SPB_CHESS_MAX_HISTORY records).  The device buffers of the trajectories are
 * allocated by the first spb_chess_selfplay_step (SPB_CHESS_MAX_HISTORY records per slot plus the output buffer, 1,624 bytes a
 * record); an engine that never plays keeps its search footprint.  Outcomes follow the value the chess search uses (chess.rs:172:
 * Won = +1.0 for the side to move in the terminal state, i.e. the CHECKMATED side), signed per position by
 * learner_concurrent.rs:214-226: every position of the mated side gets +1, of the mating side -1 (DESIGN.md §7).
 * A game whose next position would pass SPB_CHESS_MAX_HISTORY plies of history or SPB_CHESS_MAX_HISTORY records ends as a
 * tie with SPB_CHESS_POS_ADJUDICATED set on every record (the reference has no such cap).
 */
#define SPB_CHESS_POS_ADJUDICATED 1u   /* spb_chess_position.flags: the game was ended as a tie at the history cap */

typedef struct spb_chess_position {
  spb_chess_state state;                            /* root the search ran from; hist_len as at that root */
  uint32_t visit_counts[SPB_CHESS_MAX_MOVES];       /* root children in child order; 0 past n_moves */
  uint16_t moves[SPB_CHESS_MAX_MOVES];              /* their moves; 0xFFFF past n_moves */
  uint16_t n_moves;
  uint16_t ply;                                     /* index of this position inside its trajectory */
  uint8_t  repetitions;                             /* get_num_repetitions of the root (chess.rs:51-62), encoding plane 16 */
  int8_t   outcome;                                 /* value target: +1 / 0 / -1 from this position's side to move */
  uint8_t  flags;                                   /* SPB_CHESS_POS_* */
  uint8_t  reserved;
} spb_chess_position;                               /* 1,624 bytes */

/*
 * One self-play ply for every live slot on the device: pick a root child by `rule` (SPB_MOVE_*; temperature: sample
 * ∝ N^temperature with the counter-based RNG keyed by (seed, game id, ply)), record the root, then end the game (terminal
 * child or history cap: emit the trajectory; restart the slot from restart_roots[slot] / restart_history[slot] when
 * restart_roots != NULL — the rules of spb_chess_reset_games, arrays of num_games entries — else leave it idle) or re-root
 * (use_subtree, exactly as spb_chess_advance).  n_finished (nullable): games emitted by this call.  A full output buffer
 * parks the game's slot with its history and the call returns SPB_ERR_STATE; nothing is lost: drain and call again.
 */
int32_t spb_chess_selfplay_step(spb_chess_engine* e, int32_t rule, float temperature, uint64_t seed, const spb_chess_state* restart_roots,
                                const uint64_t* restart_history, uint32_t* n_finished);
/* Copies the finished positions (ordered by game id, then ply) to buf; buf == NULL: *written = the number held. */
int32_t spb_chess_drain_trajectories(spb_chess_engine* e, spb_chess_position* buf, size_t capacity, size_t* written,
                                     uint64_t* game_ids /* nullable, [capacity] */);
/* spb_drain_trajectories_device for chess records; an engine that never played holds 0 records and allocates nothing. */
int32_t spb_chess_drain_trajectories_device(spb_chess_engine* e, spb_chess_position* buf_dev, size_t capacity, size_t* written,
                                            uint64_t* game_ids_dev /* nullable */);
/*
 * The training tensors of n records (host only, no GPU needed), each output nullable: encodings[n][19][8][8] (get_encoding of
 * the recorded root with its recorded repetitions, chess.rs:176-249), policies[n][4672] (visit counts scattered by the policy
 * index of each move and divided by their f32 sum: what spb_chess_root_policy returned for that root), values[n] (outcome).
 * SPB_ERR_ARG for a malformed record (n_moves outside 1..256, side > 1, a move outside the policy).
 */
int32_t spb_chess_positions_to_training(const spb_chess_position* positions, size_t n, float* encodings, float* policies, float* values);
/*
 * The same tensors built on the device, per minibatch, from records held in device memory (ref: the replay buffer the
 * learner pops batch_size positions from, learner_concurrent.rs:87-165; the tensors of :126-146).  Output row i comes
 * from positions[indices ? indices[i] : i]; without indices n <= n_positions.  Every pointer is device (or managed) memory
 * of e's GPU (records and indices 8-byte aligned, outputs 4-byte aligned), each output nullable: encodings[n][19][8][8], policies[n][4672], values[n].  The results are bit-identical
 * to spb_chess_positions_to_training of the same records (a record whose counts sum to 0 gives NaN policies on both
 * sides, with the NaN bit pattern of each processor).  Validation is that of the host function, plus indices[i] <
 * n_positions: a malformed row gives SPB_ERR_ARG, nothing is written, and spb_chess_last_error names the first bad row.
 * Enqueued on the engine's stream; returns once the outputs are written.
 */
int32_t spb_chess_positions_to_training_device(spb_chess_engine* e, const spb_chess_position* positions, size_t n_positions,
                                               const uint64_t* indices /* nullable */, size_t n,
                                               float* encodings, float* policies, float* values);

/* ---- multi-GPU: trajectories to the learner rank; learner hand-off ------- */

/*
 * Games are sharded over GPUs: one engine per rank, global game ids by spb_config.game_id_base / game_id_stride, no
 * exchange while searching.  The one exchange is the gather of finished trajectories to the learner rank — the role of the
 * replay-buffer push of the reference's workers (ref: learner_concurrent.rs:281-288).  Transport: NCCL, bound at run time
 * (libnccl.so.2).  Rank 0 creates an id, the host distributes its 128 bytes by any means, every rank joins:
 */
#define SPB_COMM_ID_BYTES 128
int32_t spb_comm_unique_id(uint8_t* id /* [SPB_COMM_ID_BYTES] */);
int32_t spb_comm_init(spb_engine* e, const uint8_t* id, int32_t rank, int32_t world_size);
int32_t spb_comm_destroy(spb_engine* e);
/*
 * COLLECTIVE over the communicator: every rank hands over the trajectories it would otherwise return from
 * spb_drain_trajectories (all-gather of counts, grouped send/recv into device memory of the learner rank).  On the learner
 * rank *written = total records, ordered by (global game id, ply): the result of R ranks is byte-identical to the same
 * games played on one rank.  If buf is NULL or capacity < *written the records stay staged and the next call (no
 * collective) delivers them.  On the other ranks *written = 0.
 */
int32_t spb_gather_trajectories(spb_engine* e, int32_t learner_rank, spb_position* buf, size_t capacity, size_t* written,
                                uint64_t* game_ids /* nullable */);
/*
 * The device form of the gather, with its contract (COLLECTIVE; *written = 0 on the other ranks): on the learner rank the
 * ordered records go to buf_dev / game_ids_dev (nullable), with the pointer rules of spb_drain_trajectories_device.  If
 * buf_dev is NULL or capacity < *written the gathered records stay staged in device memory and the next call (no
 * collective) delivers them; the pointers are checked at that delivery, after the collective, and a bad one returns
 * SPB_ERR_ARG with the records still staged.  *written == 0 stages nothing: the next call is a new collective, so a
 * learner makes its delivering call only when *written > 0.  A gather staged by one form cannot be claimed by the
 * other: that call returns SPB_ERR_STATE, naming the call to make, and the records stay staged.
 */
int32_t spb_gather_trajectories_device(spb_engine* e, int32_t learner_rank, spb_position* buf_dev, size_t capacity,
                                       size_t* written, uint64_t* game_ids_dev /* nullable */);
/*
 * COLLECTIVE over the communicator: the weight image of root_rank, as it stands, replaces every other rank's (a rank needs
 * no weights beforehand).  First every rank learns what every rank holds (all-gather of a small descriptor): if the root
 * has no weights (SPB_ERR_STATE), a rank cannot hold the image (SPB_ERR_NOMEM) or the ranks' games differ (SPB_ERR_ARG),
 * every rank returns that error, no second collective is issued and every net stays as it was.  Then the image is
 * broadcast on the engine's stream; a non-root rank whose image did not arrive is left without weights.  No communicator:
 * SPB_ERR_STATE; root_rank out of range: SPB_ERR_ARG.  Trajectory staging is not touched.
 */
int32_t spb_broadcast_weights(spb_engine* e, int32_t root_rank);
/*
 * The same for chess engines (ref: learner_concurrent.rs:281-288), with the contract of spb_comm_init, spb_comm_destroy and
 * spb_gather_trajectories; the id comes from spb_comm_unique_id.  The gather hands over what spb_chess_drain_trajectories
 * would return; an engine that never played (no trajectory buffers yet) takes part with 0 records.  spb_chess_destroy
 * releases a live communicator.
 */
int32_t spb_chess_comm_init(spb_chess_engine* e, const uint8_t* id, int32_t rank, int32_t world_size);
int32_t spb_chess_comm_destroy(spb_chess_engine* e);
int32_t spb_chess_gather_trajectories(spb_chess_engine* e, int32_t learner_rank, spb_chess_position* buf, size_t capacity,
                                      size_t* written, uint64_t* game_ids /* nullable */);
int32_t spb_chess_gather_trajectories_device(spb_chess_engine* e, int32_t learner_rank, spb_chess_position* buf_dev,
                                             size_t capacity, size_t* written, uint64_t* game_ids_dev /* nullable */);
int32_t spb_chess_broadcast_weights(spb_chess_engine* e, int32_t root_rank);   /* spb_broadcast_weights for chess */
/*
 * ref: learner_concurrent.rs:126-146, learner.rs:162-182 — the tensors the learners train on, from n compact records
 * (host only, no GPU needed): encodings[n][3][R][C] (get_encoding of the recorded root state, connect_four.rs:242-259),
 * policies[n][A] (root visit counts / their sum, mcts.rs:315-328), values[n] (+-1 / 0 from the position's side to move,
 * learner_concurrent.rs:214-226).  Any output may be NULL.
 */
int32_t spb_positions_to_training(int32_t game, const spb_position* positions, size_t n, float* encodings, float* policies,
                                  float* values);
/*
 * The same tensors built on the device for the engine's game, per minibatch, from records held in device memory.  Output
 * row i comes from positions_dev[indices_dev ? indices_dev[i] : i]; without indices n <= n_positions.  Every pointer is
 * device (or managed) memory of e's GPU, the records and indices 8-byte aligned and the outputs 4-byte aligned (else
 * SPB_ERR_ARG naming the argument, nothing written), each output nullable: encodings_dev[n][3][R][C], policies_dev[n][A],
 * values_dev[n].  The results are bit-identical to spb_positions_to_training(game, ...) of the same records, which reads
 * current_player & 1 (a record whose counts sum to 0 gives NaN policies on both sides, with the NaN bit pattern of each
 * processor).  An index >= n_positions gives SPB_ERR_ARG, nothing is written, and spb_last_error names the first bad row.
 * Enqueued on the engine's stream; returns once the outputs are written.
 */
int32_t spb_positions_to_training_device(spb_engine* e, const spb_position* positions_dev, size_t n_positions,
                                         const uint64_t* indices_dev /* nullable */, size_t n,
                                         float* encodings_dev, float* policies_dev, float* values_dev);

/* ---- counters / timing -------------------------------------------------- */
int32_t spb_get_counters(spb_engine* e, spb_counters* out);
int32_t spb_reset_counters(spb_engine* e);
/*
 * Device time (CUDA events on the engine's stream) of the most recent spb_search and the number of evaluator
 * launches inside it.  evaluator_ms is reserved and reads 0: the steps run as one CUDA graph of programmatically
 * dependent launches, so there is no per-launch event — spb_time_evaluator measures the evaluator's launch time.
 */
int32_t spb_last_search_timing(spb_engine* e, float* search_ms, float* evaluator_ms,
                               uint32_t* evaluator_launches);
int32_t spb_synchronize(spb_engine* e);
/*
 * Statistics of the most recent search through the asynchronous pipeline (zeros for the other pipelines), out[0..n):
 * [0] evaluator batches, [1] boards in them, [2] ns the evaluator CTAs waited for leaves (sum over CTAs), [3] ns the tree
 * warps spent on trees (sum over warps), [4] tree visits, [5] tree warps, [6] evaluator CTAs.
 */
int32_t spb_last_async_stats(spb_engine* e, uint64_t* out, uint32_t n);
/*
 * Re-runs the evaluator kernel `iters` times on the work list of the most recent lock-step search (the leaves of
 * its last simulation step, still resident in HBM) and reports the average launch duration, measured with CUDA
 * events on the engine's stream, the number of positions per launch and the FLOPs per position (2*MAC).
 * Used by bench.py for the tensor roofline of the dominant kernel.
 */
int32_t spb_time_evaluator(spb_engine* e, uint32_t iters, float* avg_ms, uint32_t* n_positions, double* flops_per_position);

#ifdef __cplusplus
}
#endif
#endif /* SELFPLAY_B200_H */
