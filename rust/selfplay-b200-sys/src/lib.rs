//! 1:1 mirror of `include/selfplay_b200.h` (ABI version 2).  NOT compiled in the build image
//! (no rustc/cargo there); kept line-for-line with the header so it can be checked by eye.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub const SPB_ABI_VERSION: u32 = 2;
pub const SPB_OK: i32 = 0;
pub const SPB_ERR_ARG: i32 = -1;
pub const SPB_ERR_CUDA: i32 = -2;
pub const SPB_ERR_POOL: i32 = -3;
pub const SPB_ERR_ILLEGAL: i32 = -4;
pub const SPB_ERR_WEIGHTS: i32 = -5;
pub const SPB_ERR_STATE: i32 = -6;
pub const SPB_ERR_NOMEM: i32 = -7;
pub const SPB_GAME_TICTACTOE: i32 = 0;
pub const SPB_GAME_CONNECT4: i32 = 1;
pub const SPB_GAME_CHESS: i32 = 2;
pub const SPB_CHESS_MAX_MOVES: usize = 256;
pub const SPB_CHESS_MAX_HISTORY: usize = 512;
pub const SPB_CHESS_PLANES: usize = 19;
pub const SPB_CHESS_POLICY_SIZE: usize = 4672;
pub const SPB_CHESS_NO_SQUARE: u8 = 64;
pub const SPB_CHESS_POS_ADJUDICATED: u8 = 1;
pub const SPB_COMM_ID_BYTES: usize = 128;
pub const SPB_MAX_ACTIONS: usize = 9;
pub const SPB_STATUS_ONGOING: u8 = 0;
pub const SPB_STATUS_TIED: u8 = 1;
pub const SPB_STATUS_WON: u8 = 2;
pub const SPB_EVAL_NET: i32 = 0;
pub const SPB_EVAL_DET: i32 = 1;
pub const SPB_EVAL_UNIFORM: i32 = 2;
pub const SPB_FLAG_NO_GRAPH: u32 = 1;
pub const SPB_FLAG_EVAL_SIMT: u32 = 2;
pub const SPB_FLAG_FORCE_SPLIT: u32 = 4;
pub const SPB_FLAG_LOCKSTEP: u32 = 32;
pub const SPB_FLAG_FIXED_POOL: u32 = 16;
pub const SPB_MOVE_GREEDY_LAST_MAX: i32 = 0;
pub const SPB_MOVE_TEMPERATURE: i32 = 1;

#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct spb_state {
    pub stones: [u64; 2],
    pub current_player: u8,
    pub num_actions_played: u8,
    pub status: u8,
    pub reserved: [u8; 5],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct spb_config {
    pub abi_version: u32,
    pub game: i32,
    pub device: i32,
    pub num_games: u32,
    pub max_nodes_per_tree: u32,
    pub leaves_per_tree: u32,
    pub c: f32,
    pub evaluator: i32,
    pub flags: u32,
    pub game_id_base: u32,
    pub game_id_stride: u32,
    pub trajectory_capacity: u32,
    pub reserved: [u32; 4],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct spb_counters {
    pub simulations: u64,
    pub evaluations: u64,
    pub terminal_leaves: u64,
    pub path_length_sum: u64,
    pub children_created: u64,
    pub nodes_live: u64,
    pub kernel_launches: u64,
    pub reserved: [u64; 5],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct spb_position {
    pub stones: [u64; 2],
    pub visit_counts: [u32; SPB_MAX_ACTIONS],
    pub current_player: u8,
    pub ply: u8,
    pub outcome: i8,
    pub reserved: u8,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default, PartialEq, Eq)]
pub struct spb_chess_state {
    pub piece: [u64; 6],
    pub color: [u64; 2],
    pub side: u8,
    pub castle: u8,
    pub ep: u8,
    pub reserved0: u8,
    pub fifty: u16,
    pub plies: u16,
    pub hist_len: u32,
    pub reserved1: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct spb_chess_position {
    pub state: spb_chess_state,
    pub visit_counts: [u32; SPB_CHESS_MAX_MOVES],
    pub moves: [u16; SPB_CHESS_MAX_MOVES],
    pub n_moves: u16,
    pub ply: u16,
    pub repetitions: u8,
    pub outcome: i8,
    pub flags: u8,
    pub reserved: u8,
}

#[repr(C)]
pub struct spb_engine {
    _private: [u8; 0],
}

#[repr(C)]
pub struct spb_chess_engine {
    _private: [u8; 0],
}

extern "C" {
    pub fn spb_abi_version() -> i32;
    pub fn spb_default_config(cfg: *mut spb_config) -> i32;
    pub fn spb_create(cfg: *const spb_config, out: *mut *mut spb_engine) -> i32;
    pub fn spb_destroy(e: *mut spb_engine) -> i32;
    pub fn spb_last_error(e: *const spb_engine) -> *const c_char;
    pub fn spb_load_weights(e: *mut spb_engine, blob: *const c_void, num_bytes: usize) -> i32;
    pub fn spb_check_weights(game: i32, blob: *const c_void, num_bytes: usize, err: *mut c_char, err_cap: usize) -> i32;
    pub fn spb_reset_games(e: *mut spb_engine, slots: *const u32, n: u32, roots: *const spb_state) -> i32;
    pub fn spb_search(e: *mut spb_engine, num_searches: u32) -> i32;
    pub fn spb_root_children(e: *mut spb_engine, slot: u32, actions: *mut u8, visit_counts: *mut u32, child_ids: *mut u32, n_children: *mut u32) -> i32;
    pub fn spb_root_children_all(e: *mut spb_engine, actions: *mut u8, visit_counts: *mut u32, child_ids: *mut u32, n_children: *mut u32) -> i32;
    pub fn spb_root_policy(e: *mut spb_engine, slot: u32, policy: *mut f32) -> i32;
    pub fn spb_advance(e: *mut spb_engine, slots: *const u32, node_ids: *const u32, n: u32, out_states: *mut spb_state) -> i32;
    pub fn spb_get_state(e: *mut spb_engine, slot: u32, node_id: u32, out: *mut spb_state) -> i32;
    pub fn spb_arena_len(e: *mut spb_engine, slot: u32, out: *mut u32) -> i32;
    pub fn spb_node_stats(e: *mut spb_engine, slot: u32, node_id: u32, visit_count: *mut u32, value_sum: *mut f32, prior: *mut f32, first_child: *mut u32, n_children: *mut u32) -> i32;
    /// EXTENSION (DESIGN.md §4.6): Dirichlet noise on the root priors; epsilon = 0 turns it off.
    pub fn spb_set_root_noise(e: *mut spb_engine, alpha: f32, epsilon: f32, seed: u64) -> i32;
    /// eta[SPB_MAX_ACTIONS] of the slot's current root (child order), *n = number of root children.
    pub fn spb_root_noise(e: *mut spb_engine, slot: u32, eta: *mut f32, n: *mut u32) -> i32;
    pub fn spb_predict(e: *mut spb_engine, states: *const spb_state, n: u32, policies: *mut f32, values: *mut f32, raw_logits: *mut f32) -> i32;
    pub fn spb_game_next_states(e: *mut spb_engine, states: *const spb_state, actions: *const u8, n: u32, out_states: *mut spb_state, err: *mut i32) -> i32;
    pub fn spb_game_valid_actions(e: *mut spb_engine, states: *const spb_state, n: u32, masks: *mut u32) -> i32;
    pub fn spb_game_encode(e: *mut spb_engine, states: *const spb_state, n: u32, out: *mut f32) -> i32;
    pub fn spb_selfplay_step(e: *mut spb_engine, rule: i32, temperature: f32, seed: u64, restart_roots: *const spb_state, n_finished: *mut u32) -> i32;
    pub fn spb_drain_trajectories(e: *mut spb_engine, buf: *mut spb_position, capacity: usize, written: *mut usize, game_ids: *mut u64) -> i32;
    pub fn spb_drain_trajectories_device(e: *mut spb_engine, buf_dev: *mut spb_position, capacity: usize, written: *mut usize, game_ids_dev: *mut u64) -> i32;
    pub fn spb_chess_create(cfg: *const spb_config, out: *mut *mut spb_chess_engine) -> i32;
    pub fn spb_chess_destroy(e: *mut spb_chess_engine) -> i32;
    pub fn spb_chess_last_error(e: *const spb_chess_engine) -> *const c_char;
    pub fn spb_chess_load_weights(e: *mut spb_chess_engine, blob: *const c_void, num_bytes: usize) -> i32;
    pub fn spb_chess_check_weights(blob: *const c_void, num_bytes: usize, err: *mut c_char, err_cap: usize) -> i32;
    pub fn spb_chess_start_position(out: *mut spb_chess_state) -> i32;
    pub fn spb_chess_legal_moves(e: *mut spb_chess_engine, states: *const spb_chess_state, history: *const u64, n: u32, moves: *mut u16, counts: *mut u32, policy_index: *mut u16, status: *mut u8, repetitions: *mut u32) -> i32;
    pub fn spb_chess_next_states(e: *mut spb_chess_engine, states: *const spb_chess_state, history: *mut u64, moves: *const u16, n: u32, out_states: *mut spb_chess_state, err: *mut i32) -> i32;
    pub fn spb_chess_encode(e: *mut spb_chess_engine, states: *const spb_chess_state, history: *const u64, n: u32, out: *mut f32) -> i32;
    pub fn spb_chess_perft(e: *mut spb_chess_engine, state: *const spb_chess_state, depth: u32, nodes: *mut u64) -> i32;
    pub fn spb_chess_move_channel(side: i32, mv: u16) -> i32;
    pub fn spb_chess_policy_index(side: i32, mv: u16) -> i32;
    pub fn spb_chess_action(side: i32, channel: i32, row: i32, col: i32) -> u16;
    pub fn spb_chess_reset_games(e: *mut spb_chess_engine, slots: *const u32, n: u32, roots: *const spb_chess_state, history: *const u64) -> i32;
    pub fn spb_chess_search(e: *mut spb_chess_engine, num_searches: u32) -> i32;
    pub fn spb_chess_last_search_ms(e: *mut spb_chess_engine, ms: *mut f32) -> i32;
    pub fn spb_chess_root_children(e: *mut spb_chess_engine, slot: u32, moves: *mut u16, visit_counts: *mut u32, child_ids: *mut u32, n_children: *mut u32) -> i32;
    pub fn spb_chess_root_children_all(e: *mut spb_chess_engine, moves: *mut u16, visit_counts: *mut u32, child_ids: *mut u32, n_children: *mut u32) -> i32;
    pub fn spb_chess_root_policy(e: *mut spb_chess_engine, slot: u32, out: *mut f32) -> i32;
    pub fn spb_chess_advance(e: *mut spb_chess_engine, slots: *const u32, child_ids: *const u32, n: u32, out_states: *mut spb_chess_state) -> i32;
    pub fn spb_chess_get_state(e: *mut spb_chess_engine, slot: u32, node_id: u32, out: *mut spb_chess_state) -> i32;
    pub fn spb_chess_arena_len(e: *mut spb_chess_engine, slot: u32, out: *mut u32) -> i32;
    pub fn spb_chess_node_stats(e: *mut spb_chess_engine, slot: u32, node_id: u32, visit_count: *mut u32, value_sum: *mut f32, prior: *mut f32, first_child: *mut u32, n_children: *mut u32, mv: *mut u16, status: *mut u8) -> i32;
    pub fn spb_chess_set_root_noise(e: *mut spb_chess_engine, alpha: f32, epsilon: f32, seed: u64) -> i32;
    /// eta[SPB_CHESS_MAX_MOVES] of the slot's current root (child order), *n = number of legal moves of the root.
    pub fn spb_chess_root_noise(e: *mut spb_chess_engine, slot: u32, eta: *mut f32, n: *mut u32) -> i32;
    pub fn spb_chess_predict(e: *mut spb_chess_engine, states: *const spb_chess_state, history: *const u64, n: u32, policies: *mut f32, values: *mut f32, raw_logits: *mut f32) -> i32;
    pub fn spb_chess_time_conv(e: *mut spb_chess_engine, iters: u32, avg_ms: *mut f32, n_positions: *mut u32, flops_per_launch: *mut f64, flops_per_position: *mut f64) -> i32;
    pub fn spb_chess_get_counters(e: *mut spb_chess_engine, out: *mut spb_counters) -> i32;
    pub fn spb_chess_reset_counters(e: *mut spb_chess_engine) -> i32;
    pub fn spb_chess_selfplay_step(e: *mut spb_chess_engine, rule: i32, temperature: f32, seed: u64, restart_roots: *const spb_chess_state, restart_history: *const u64, n_finished: *mut u32) -> i32;
    pub fn spb_chess_drain_trajectories(e: *mut spb_chess_engine, buf: *mut spb_chess_position, capacity: usize, written: *mut usize, game_ids: *mut u64) -> i32;
    pub fn spb_chess_drain_trajectories_device(e: *mut spb_chess_engine, buf_dev: *mut spb_chess_position, capacity: usize, written: *mut usize, game_ids_dev: *mut u64) -> i32;
    pub fn spb_chess_positions_to_training(positions: *const spb_chess_position, n: usize, encodings: *mut f32, policies: *mut f32, values: *mut f32) -> i32;
    pub fn spb_chess_positions_to_training_device(e: *mut spb_chess_engine, positions: *const spb_chess_position, n_positions: usize, indices: *const u64, n: usize, encodings: *mut f32, policies: *mut f32, values: *mut f32) -> i32;
    pub fn spb_comm_unique_id(id: *mut u8) -> i32;
    pub fn spb_comm_init(e: *mut spb_engine, id: *const u8, rank: i32, world_size: i32) -> i32;
    pub fn spb_comm_destroy(e: *mut spb_engine) -> i32;
    pub fn spb_gather_trajectories(e: *mut spb_engine, learner_rank: i32, buf: *mut spb_position, capacity: usize, written: *mut usize, game_ids: *mut u64) -> i32;
    pub fn spb_gather_trajectories_device(e: *mut spb_engine, learner_rank: i32, buf_dev: *mut spb_position, capacity: usize, written: *mut usize, game_ids_dev: *mut u64) -> i32;
    pub fn spb_chess_comm_init(e: *mut spb_chess_engine, id: *const u8, rank: i32, world_size: i32) -> i32;
    pub fn spb_chess_comm_destroy(e: *mut spb_chess_engine) -> i32;
    pub fn spb_chess_gather_trajectories(e: *mut spb_chess_engine, learner_rank: i32, buf: *mut spb_chess_position, capacity: usize, written: *mut usize, game_ids: *mut u64) -> i32;
    pub fn spb_chess_gather_trajectories_device(e: *mut spb_chess_engine, learner_rank: i32, buf_dev: *mut spb_chess_position, capacity: usize, written: *mut usize, game_ids_dev: *mut u64) -> i32;
    pub fn spb_positions_to_training(game: i32, positions: *const spb_position, n: usize, encodings: *mut f32, policies: *mut f32, values: *mut f32) -> i32;
    pub fn spb_positions_to_training_device(e: *mut spb_engine, positions_dev: *const spb_position, n_positions: usize, indices_dev: *const u64, n: usize, encodings_dev: *mut f32, policies_dev: *mut f32, values_dev: *mut f32) -> i32;
    pub fn spb_get_counters(e: *mut spb_engine, out: *mut spb_counters) -> i32;
    pub fn spb_reset_counters(e: *mut spb_engine) -> i32;
    pub fn spb_last_search_timing(e: *mut spb_engine, search_ms: *mut f32, evaluator_ms: *mut f32, evaluator_launches: *mut u32) -> i32;
    pub fn spb_synchronize(e: *mut spb_engine) -> i32;
    pub fn spb_last_async_stats(e: *mut spb_engine, out: *mut u64, n: u32) -> i32;
    pub fn spb_time_evaluator(e: *mut spb_engine, iters: u32, avg_ms: *mut f32, n_positions: *mut u32, flops_per_position: *mut f64) -> i32;
}
