//! Safe wrapper with the signatures `learner.rs` / `learner_concurrent.rs` use today
//! (ref: src/mcts.rs:32-44, :86, :161, :196; src/game/mod.rs:21-44; src/model/mod.rs:36).  The trees live on the GPU; a
//! `Tree` is a handle on one engine slot.  1:1 with include/selfplay_b200.h through `selfplay-b200-sys`.
//! NOT compiled in the build image (no rustc/cargo there).
use selfplay_b200_sys as sys;
use std::ffi::CStr;
use std::marker::PhantomData;

#[derive(Debug)]
pub struct Error { pub code: i32, pub message: String }
pub type Result<T> = std::result::Result<T, Error>;

/// Conversion between the reference's game states and the ABI's bitboard state.
/// Implemented in the reference crate for `game::connect_four::State` (bit = col*7+row) and
/// `game::tictactoe::State` (bit = row*3+col); see INTEGRATION.md.
pub trait AbiState: Sized {
    const GAME: i32;
    const NUM_ACTIONS: usize;
    const ROWS: usize;
    const COLS: usize;
    fn to_abi(&self) -> sys::spb_state;
    fn from_abi(s: &sys::spb_state) -> Self;
}

/// The `spb_tensor` table of a device load; owns the NUL-terminated names for the call.
struct TensorTable { _names: Vec<std::ffi::CString>, raw: Vec<sys::spb_tensor> }
impl TensorTable {
    fn new(tensors: &[(&str, *const std::os::raw::c_void, i32, &[i64])]) -> Result<Self> {
        let mut names = Vec::with_capacity(tensors.len());
        let mut raw = Vec::with_capacity(tensors.len());
        for (name, data, dtype, shape) in tensors {
            if shape.len() > 4 { return Err(Error { code: sys::SPB_ERR_ARG, message: format!("{}: more than 4 dimensions", name) }); }
            let c = std::ffi::CString::new(*name).map_err(|_| Error { code: sys::SPB_ERR_ARG, message: format!("{}: NUL in the name", name) })?;
            let mut s = [0i64; 4];
            s[..shape.len()].copy_from_slice(shape);
            raw.push(sys::spb_tensor { name: c.as_ptr(), data: *data, dtype: *dtype, ndim: shape.len() as i32, shape: s });
            names.push(c);
        }
        Ok(TensorTable { _names: names, raw })
    }
}

/// ref: `Args` mcts.rs:8-18 — only `c` and `num_searches` are read on the search path.
#[derive(Clone, Copy)]
pub struct Args { pub c: f32, pub num_searches: u32, pub num_parallel_self_play_games: usize }
impl Default for Args {
    fn default() -> Self { Args { c: 2.0, num_searches: 600, num_parallel_self_play_games: 100 } }
}

/// How `self_play_step` picks the move (ref: main.rs:108-112 greedy last-max; learner_concurrent.rs:189-194 temperature).
#[derive(Clone, Copy)]
pub enum MoveRule { GreedyLastMax, Temperature { temperature: f32, seed: u64 } }

/// One recorded position of a finished game (ref: `Payload`, learner_concurrent.rs:13-18, in compact form).
pub type Position = sys::spb_position;

/// The tensors the learners train on (ref: learner_concurrent.rs:126-146): row-major `[n,3,R,C]`, `[n,A]`, `[n,1]`.
pub struct TrainingBatch { pub n: usize, pub encodings: Vec<f32>, pub policies: Vec<f32>, pub values: Vec<f32> }

/// ref: `Mcts<T>` mcts.rs:41-44.  Owns the engine (node pools, weights) of one GPU; one per host thread.
pub struct Mcts<S: AbiState> { raw: *mut sys::spb_engine, pub args: Args, _s: PhantomData<S> }
unsafe impl<S: AbiState> Send for Mcts<S> {}

/// ref: `Tree<T>` mcts.rs:32-39: a handle on slot `slot`; histories stay on the host like in the reference.
pub struct Tree<S: AbiState> { pub slot: u32, pub state_history: Vec<S>, pub policy_history: Vec<Vec<f32>> }

impl<S: AbiState> Mcts<S> {
    pub fn new(args: Args, device: i32, evaluator: i32) -> Result<Self> {
        Self::with_shard(args, device, evaluator, 0, 0)
    }
    /// Multi-GPU: rank r of R passes `game_id_base = r * games`, `game_id_stride = R * games` (SURVEY §8e).
    pub fn with_shard(args: Args, device: i32, evaluator: i32, game_id_base: u32, game_id_stride: u32) -> Result<Self> {
        let mut cfg = sys::spb_config::default();
        unsafe { sys::spb_default_config(&mut cfg) };
        cfg.game = S::GAME; cfg.device = device; cfg.c = args.c; cfg.evaluator = evaluator;
        cfg.num_games = args.num_parallel_self_play_games as u32;
        cfg.game_id_base = game_id_base; cfg.game_id_stride = game_id_stride;
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::spb_create(&cfg, &mut raw) };
        if rc != sys::SPB_OK { return Err(Error { code: rc, message: last_error(std::ptr::null()) }); }
        Ok(Mcts { raw, args, _s: PhantomData })
    }
    fn check(&self, rc: i32) -> Result<()> {
        if rc == sys::SPB_OK { Ok(()) } else { Err(Error { code: rc, message: last_error(self.raw) }) }
    }
    /// ref: `VarStore::load` main.rs:61 — bytes of the safetensors file `var_store.save` wrote (learner.rs:192).
    /// May be called again on a live engine (hot swap between generations, learner_concurrent.rs:158-159).
    pub fn load_weights(&mut self, safetensors: &[u8]) -> Result<()> {
        self.check(unsafe { sys::spb_load_weights(self.raw, safetensors.as_ptr() as *const _, safetensors.len()) })
    }
    /// The learner's live parameters, with no file in between: `(name, device pointer, dtype, shape)` per tensor, named as
    /// `VarStore::variables()` names them (e.g. `tensor.data_ptr()`, `SPB_DTYPE_F32`, `tensor.size()`).  The caller has
    /// finished writing the tensors (e.g. synchronised its stream); once this returns they may change.
    /// # Safety
    /// Each pointer must be a contiguous tensor of that dtype and shape in device memory of this engine's GPU.
    pub unsafe fn load_weights_device(&mut self, tensors: &[(&str, *const std::os::raw::c_void, i32, &[i64])]) -> Result<()> {
        let table = TensorTable::new(tensors)?;
        self.check(sys::spb_load_weights_device(self.raw, table.raw.as_ptr(), table.raw.len() as u32))
    }
    /// COLLECTIVE over the communicator: every rank takes `root_rank`'s weights.
    pub fn broadcast_weights(&mut self, root_rank: i32) -> Result<()> {
        self.check(unsafe { sys::spb_broadcast_weights(self.raw, root_rank) })
    }
    /// EXTENSION (not in the reference, mcts.rs:204-207 is a TODO; DESIGN.md §4.6): Dirichlet noise on the root priors of
    /// every search, P' = (1 - epsilon) P + epsilon eta with eta ~ Dir(alpha).  epsilon = 0 turns it off (the default).
    pub fn set_root_noise(&mut self, alpha: f32, epsilon: f32, seed: u64) -> Result<()> {
        self.check(unsafe { sys::spb_set_root_noise(self.raw, alpha, epsilon, seed) })
    }
    /// The eta the next search of `tree`'s root uses, one entry per root child (child order).
    pub fn root_noise(&mut self, tree: &Tree<S>) -> Result<Vec<f32>> {
        let (mut eta, mut n) = ([0f32; sys::SPB_MAX_ACTIONS], 0u32);
        self.check(unsafe { sys::spb_root_noise(self.raw, tree.slot, eta.as_mut_ptr(), &mut n) })?;
        Ok(eta[..n as usize].to_vec())
    }
    /// ref: `Tree::with_root_state` mcts.rs:86 / `Tree::default` mcts.rs:67.
    pub fn new_tree(&mut self, slot: u32, root: Option<&S>) -> Result<Tree<S>> {
        let abi = root.map(|s| s.to_abi());
        let p = abi.as_ref().map_or(std::ptr::null(), |s| s as *const _);
        self.check(unsafe { sys::spb_reset_games(self.raw, &slot, 1, p) })?;
        Ok(Tree { slot, state_history: Vec::new(), policy_history: Vec::new() })
    }
    /// ref: `Mcts::search` mcts.rs:196 — result i belongs to trees[i]:
    /// (root visit counts scattered by action and normalised, [(child arena id, visit count as f32)] in child order).
    pub fn search(&mut self, trees: &mut Vec<&mut Tree<S>>) -> Result<Vec<(Vec<f32>, Vec<(usize, f32)>)>> {
        self.check(unsafe { sys::spb_search(self.raw, self.args.num_searches) })?;
        let mut out = Vec::with_capacity(trees.len());
        for t in trees.iter() {
            let (mut a, mut c, mut ids, mut n) = ([0u8; sys::SPB_MAX_ACTIONS], [0u32; sys::SPB_MAX_ACTIONS], [0u32; sys::SPB_MAX_ACTIONS], 0u32);
            self.check(unsafe { sys::spb_root_children(self.raw, t.slot, a.as_mut_ptr(), c.as_mut_ptr(), ids.as_mut_ptr(), &mut n) })?;
            let mut policy = vec![0f32; S::NUM_ACTIONS];
            self.check(unsafe { sys::spb_root_policy(self.raw, t.slot, policy.as_mut_ptr()) })?;
            out.push((policy, (0..n as usize).map(|i| (ids[i] as usize, c[i] as f32)).collect()));
        }
        Ok(out)
    }
    /// ref: `Tree::use_subtree` mcts.rs:161; returns the new root state (`tree.arena[0].state`).
    pub fn use_subtree(&mut self, tree: &mut Tree<S>, new_root_id: usize) -> Result<S> {
        let id = new_root_id as u32;
        let mut st = sys::spb_state::default();
        self.check(unsafe { sys::spb_advance(self.raw, &tree.slot, &id, 1, &mut st) })?;
        Ok(S::from_abi(&st))
    }
    /// ref: `tree.arena[id].state` (learner_concurrent.rs:184,195; main.rs:92).
    pub fn node_state(&mut self, tree: &Tree<S>, node_id: usize) -> Result<S> {
        let mut st = sys::spb_state::default();
        self.check(unsafe { sys::spb_get_state(self.raw, tree.slot, node_id as u32, &mut st) })?;
        Ok(S::from_abi(&st))
    }
    /// ref: `Model::predict` model/mod.rs:36-98 — (masked + renormalised policies `[n][A]`, values `[n]`), input order.
    pub fn predict(&mut self, states: &[&S]) -> Result<(Vec<Vec<f32>>, Vec<f32>)> {
        let abi: Vec<sys::spb_state> = states.iter().map(|s| s.to_abi()).collect();
        let n = abi.len();
        let mut pol = vec![0f32; n * S::NUM_ACTIONS];
        let mut val = vec![0f32; n];
        self.check(unsafe { sys::spb_predict(self.raw, abi.as_ptr(), n as u32, pol.as_mut_ptr(), val.as_mut_ptr(), std::ptr::null_mut()) })?;
        Ok((pol.chunks(S::NUM_ACTIONS).map(|c| c.to_vec()).collect(), val))
    }
    /// ref: `State::get_next_state` game/mod.rs:24 for a batch; `Err(String)` per state like the reference.
    pub fn next_states(&mut self, states: &[&S], actions: &[u8]) -> Result<Vec<std::result::Result<S, String>>> {
        let abi: Vec<sys::spb_state> = states.iter().map(|s| s.to_abi()).collect();
        let n = abi.len();
        let mut out = vec![sys::spb_state::default(); n];
        let mut err = vec![0i32; n];
        self.check(unsafe { sys::spb_game_next_states(self.raw, abi.as_ptr(), actions.as_ptr(), n as u32, out.as_mut_ptr(), err.as_mut_ptr()) })?;
        Ok((0..n).map(|i| if err[i] == sys::SPB_OK { Ok(S::from_abi(&out[i])) } else { Err("Invalid action or game already over".to_string()) }).collect())
    }
    /// ref: `State::get_valid_actions` game/mod.rs:25 for a batch: ascending action indices per state.
    pub fn valid_actions(&mut self, states: &[&S]) -> Result<Vec<Vec<usize>>> {
        let abi: Vec<sys::spb_state> = states.iter().map(|s| s.to_abi()).collect();
        let mut masks = vec![0u32; abi.len()];
        self.check(unsafe { sys::spb_game_valid_actions(self.raw, abi.as_ptr(), abi.len() as u32, masks.as_mut_ptr()) })?;
        Ok(masks.iter().map(|m| (0..S::NUM_ACTIONS).filter(|a| (m >> a) & 1 == 1).collect()).collect())
    }
    /// ref: `State::get_encoding` game/mod.rs:29 for a batch: `[n][3][R][C]` row-major.
    pub fn encode(&mut self, states: &[&S]) -> Result<Vec<f32>> {
        let abi: Vec<sys::spb_state> = states.iter().map(|s| s.to_abi()).collect();
        let mut out = vec![0f32; abi.len() * 3 * S::ROWS * S::COLS];
        self.check(unsafe { sys::spb_game_encode(self.raw, abi.as_ptr(), abi.len() as u32, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// One self-play ply for every live game on the device (ref: learner_concurrent.rs:179-238): pick the move, record the
    /// position, `use_subtree` or finish the game; finished slots restart from `restart_roots` (one per slot) or retire.
    /// Returns the number of games that finished.
    pub fn self_play_step(&mut self, rule: MoveRule, restart_roots: Option<&[S]>) -> Result<u32> {
        let (r, t, seed) = match rule {
            MoveRule::GreedyLastMax => (sys::SPB_MOVE_GREEDY_LAST_MAX, 0.0f32, 0u64),
            MoveRule::Temperature { temperature, seed } => (sys::SPB_MOVE_TEMPERATURE, temperature, seed),
        };
        let roots: Option<Vec<sys::spb_state>> = restart_roots.map(|v| v.iter().map(|s| s.to_abi()).collect());
        let p = roots.as_ref().map_or(std::ptr::null(), |v| v.as_ptr());
        let mut finished = 0u32;
        self.check(unsafe { sys::spb_selfplay_step(self.raw, r, t, seed, p, &mut finished) })?;
        Ok(finished)
    }
    /// Finished games' positions ordered by (game id, ply) with their global game ids (ref: learner_concurrent.rs:202-228).
    pub fn drain_trajectories(&mut self) -> Result<(Vec<Position>, Vec<u64>)> {
        let mut n = 0usize;
        self.check(unsafe { sys::spb_drain_trajectories(self.raw, std::ptr::null_mut(), 0, &mut n, std::ptr::null_mut()) })?;
        let mut pos = vec![Position::default(); n];
        let mut ids = vec![0u64; n];
        if n > 0 {
            self.check(unsafe { sys::spb_drain_trajectories(self.raw, pos.as_mut_ptr(), n, &mut n, ids.as_mut_ptr()) })?;
            pos.truncate(n); ids.truncate(n);
        }
        Ok((pos, ids))
    }
    /// Joins the NCCL communicator of the job (id from `comm_unique_id()` on rank 0, distributed by the host).
    pub fn comm_init(&mut self, id: &[u8; sys::SPB_COMM_ID_BYTES], rank: i32, world_size: i32) -> Result<()> {
        self.check(unsafe { sys::spb_comm_init(self.raw, id.as_ptr(), rank, world_size) })
    }
    /// COLLECTIVE: every rank's finished trajectories to `learner_rank`, ordered by (game id, ply) — the replay-buffer push of
    /// the reference's workers (learner_concurrent.rs:281-288).  Empty on the other ranks.
    pub fn gather_trajectories(&mut self, learner_rank: i32) -> Result<(Vec<Position>, Vec<u64>)> {
        let mut n = 0usize;
        self.check(unsafe { sys::spb_gather_trajectories(self.raw, learner_rank, std::ptr::null_mut(), 0, &mut n, std::ptr::null_mut()) })?;
        let mut pos = vec![Position::default(); n];
        let mut ids = vec![0u64; n];
        if n > 0 {
            self.check(unsafe { sys::spb_gather_trajectories(self.raw, learner_rank, pos.as_mut_ptr(), n, &mut n, ids.as_mut_ptr()) })?;
        }
        Ok((pos, ids))
    }
    /// The records of `drain_trajectories`, ordered on the device into `buf_dev[..capacity]` and `game_ids_dev` (nullable),
    /// e.g. a slice of a replay buffer on the GPU; a null `buf_dev` is the size query.  Returns the number of records.
    ///
    /// # Safety
    /// Every non-null pointer is 8-byte aligned device (or managed) memory of this engine's GPU holding `capacity` elements;
    /// no other work uses it during the call.
    pub unsafe fn drain_trajectories_device(&mut self, buf_dev: *mut Position, capacity: usize, game_ids_dev: *mut u64) -> Result<usize> {
        let mut n = 0usize;
        self.check(sys::spb_drain_trajectories_device(self.raw, buf_dev, capacity, &mut n, game_ids_dev))?;
        Ok(n)
    }
    /// COLLECTIVE: `gather_trajectories` into device memory of the learner rank (0 records elsewhere); a null or short
    /// buffer keeps the records staged on the device for the next call.  A result of 0 stages nothing: the next call is a
    /// new collective, so make the delivering call only when the size query returned more than 0.
    ///
    /// # Safety
    /// As for `drain_trajectories_device`.
    pub unsafe fn gather_trajectories_device(&mut self, learner_rank: i32, buf_dev: *mut Position, capacity: usize, game_ids_dev: *mut u64) -> Result<usize> {
        let mut n = 0usize;
        self.check(sys::spb_gather_trajectories_device(self.raw, learner_rank, buf_dev, capacity, &mut n, game_ids_dev))?;
        Ok(n)
    }
    /// The training tensors of `positions_to_training` for this engine's game, built on its GPU from records in its device
    /// memory: row i from `positions[indices[i]]`, or `positions[i]` when `indices` is null (then `n <= n_positions`).
    /// Outputs (each nullable) are bit-identical to the host builder; an index out of range is `SPB_ERR_ARG`, nothing written.
    ///
    /// # Safety
    /// As for `ChessMcts::positions_to_training_device`.
    pub unsafe fn positions_to_training_device(&mut self, positions: *const Position, n_positions: usize, indices: *const u64, n: usize,
                                               encodings: *mut f32, policies: *mut f32, values: *mut f32) -> Result<()> {
        self.check(sys::spb_positions_to_training_device(self.raw, positions, n_positions, indices, n, encodings, policies, values))
    }
    pub fn counters(&mut self) -> Result<sys::spb_counters> {
        let mut c = sys::spb_counters::default();
        self.check(unsafe { sys::spb_get_counters(self.raw, &mut c) })?;
        Ok(c)
    }
}

/// 128-byte NCCL id for `Mcts::comm_init` (rank 0 creates it).
pub fn comm_unique_id() -> Result<[u8; sys::SPB_COMM_ID_BYTES]> {
    let mut id = [0u8; sys::SPB_COMM_ID_BYTES];
    let rc = unsafe { sys::spb_comm_unique_id(id.as_mut_ptr()) };
    if rc == sys::SPB_OK { Ok(id) } else { Err(Error { code: rc, message: last_error(std::ptr::null()) }) }
}

/// ref: learner_concurrent.rs:126-146 / learner.rs:162-182 — compact records to the `(N,3,R,C) / (N,A) / (N,1)` tensors
/// (host only).  Wrap the vectors with `Tensor::of_slice(..).view(..)` on the tch side.
pub fn positions_to_training<S: AbiState>(positions: &[Position]) -> Result<TrainingBatch> {
    let n = positions.len();
    let mut b = TrainingBatch { n, encodings: vec![0f32; n * 3 * S::ROWS * S::COLS], policies: vec![0f32; n * S::NUM_ACTIONS], values: vec![0f32; n] };
    let rc = unsafe { sys::spb_positions_to_training(S::GAME, positions.as_ptr(), n, b.encodings.as_mut_ptr(), b.policies.as_mut_ptr(), b.values.as_mut_ptr()) };
    if rc == sys::SPB_OK { Ok(b) } else { Err(Error { code: rc, message: "spb_positions_to_training: bad argument".to_string() }) }
}

impl<S: AbiState> Drop for Mcts<S> {
    fn drop(&mut self) { unsafe { sys::spb_destroy(self.raw); } }
}

fn last_error(e: *const sys::spb_engine) -> String {
    unsafe { CStr::from_ptr(sys::spb_last_error(e)).to_string_lossy().into_owned() }
}

// ---- chess (ref: src/game/chess.rs, src/model/chess.rs) ---------------------------------------------------------------

/// Conversion between `game::chess::State` and the ABI's bitboards + per-ply history hashes.  A move is
/// `from | to << 6 | promotion << 12` (`ChessMove::new(Square::new(from), Square::new(to), promotion)`).
pub trait AbiChessState: Sized {
    fn to_abi(&self) -> (sys::spb_chess_state, Vec<u64>);
    fn from_abi(s: &sys::spb_chess_state) -> Self;
}

pub type ChessState = sys::spb_chess_state;

/// `Mcts<chess Net>` on one GPU.
pub struct ChessMcts { raw: *mut sys::spb_chess_engine, pub args: Args }
unsafe impl Send for ChessMcts {}

/// Handle on one chess tree.
pub struct ChessTree { pub slot: u32 }

impl ChessMcts {
    pub fn new(args: Args, device: i32, evaluator: i32) -> Result<Self> {
        let mut cfg = sys::spb_config::default();
        unsafe { sys::spb_default_config(&mut cfg) };
        cfg.game = sys::SPB_GAME_CHESS; cfg.device = device; cfg.c = args.c; cfg.evaluator = evaluator;
        cfg.num_games = args.num_parallel_self_play_games as u32;
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::spb_chess_create(&cfg, &mut raw) };
        if rc != sys::SPB_OK { return Err(Error { code: rc, message: chess_last_error(std::ptr::null()) }); }
        Ok(ChessMcts { raw, args })
    }
    fn check(&self, rc: i32) -> Result<()> {
        if rc == sys::SPB_OK { Ok(()) } else { Err(Error { code: rc, message: chess_last_error(self.raw) }) }
    }
    pub fn load_weights(&mut self, safetensors: &[u8]) -> Result<()> {
        self.check(unsafe { sys::spb_chess_load_weights(self.raw, safetensors.as_ptr() as *const _, safetensors.len()) })
    }
    /// # Safety
    /// As `Mcts::load_weights_device`.
    pub unsafe fn load_weights_device(&mut self, tensors: &[(&str, *const std::os::raw::c_void, i32, &[i64])]) -> Result<()> {
        let table = TensorTable::new(tensors)?;
        self.check(sys::spb_chess_load_weights_device(self.raw, table.raw.as_ptr(), table.raw.len() as u32))
    }
    pub fn broadcast_weights(&mut self, root_rank: i32) -> Result<()> {
        self.check(unsafe { sys::spb_chess_broadcast_weights(self.raw, root_rank) })
    }
    fn padded_history(history: &[u64]) -> Vec<u64> {
        let mut h = vec![0u64; sys::SPB_CHESS_MAX_HISTORY];
        let n = history.len().min(sys::SPB_CHESS_MAX_HISTORY);
        h[..n].copy_from_slice(&history[..n]);
        h
    }
    /// EXTENSION (DESIGN.md §4.6): Dirichlet noise on the root priors, as `Mcts::set_root_noise`.
    pub fn set_root_noise(&mut self, alpha: f32, epsilon: f32, seed: u64) -> Result<()> {
        self.check(unsafe { sys::spb_chess_set_root_noise(self.raw, alpha, epsilon, seed) })
    }
    /// The eta the next search of `tree`'s root uses, one entry per legal move of the root (child order).
    pub fn root_noise(&mut self, tree: &ChessTree) -> Result<Vec<f32>> {
        let (mut eta, mut n) = (vec![0f32; sys::SPB_CHESS_MAX_MOVES], 0u32);
        self.check(unsafe { sys::spb_chess_root_noise(self.raw, tree.slot, eta.as_mut_ptr(), &mut n) })?;
        eta.truncate(n as usize);
        Ok(eta)
    }
    /// ref: `Tree::with_root_state` mcts.rs:86.  `root = None`: the start position.
    pub fn new_tree(&mut self, slot: u32, root: Option<(&ChessState, &[u64])>) -> Result<ChessTree> {
        let rc = match root {
            None => unsafe { sys::spb_chess_reset_games(self.raw, &slot, 1, std::ptr::null(), std::ptr::null()) },
            Some((st, hist)) => {
                let h = Self::padded_history(hist);
                unsafe { sys::spb_chess_reset_games(self.raw, &slot, 1, st, h.as_ptr()) }
            }
        };
        self.check(rc)?;
        Ok(ChessTree { slot })
    }
    /// ref: `Mcts::search` mcts.rs:196: per tree (policy `[73*8*8]`, [(child arena id, visit count)], the children's moves).
    pub fn search(&mut self, trees: &mut Vec<&mut ChessTree>) -> Result<Vec<(Vec<f32>, Vec<(usize, f32)>, Vec<u16>)>> {
        self.check(unsafe { sys::spb_chess_search(self.raw, self.args.num_searches) })?;
        let mut out = Vec::with_capacity(trees.len());
        for t in trees.iter() {
            let mut mv = vec![0u16; sys::SPB_CHESS_MAX_MOVES];
            let mut cnt = vec![0u32; sys::SPB_CHESS_MAX_MOVES];
            let mut ids = vec![0u32; sys::SPB_CHESS_MAX_MOVES];
            let mut n = 0u32;
            self.check(unsafe { sys::spb_chess_root_children(self.raw, t.slot, mv.as_mut_ptr(), cnt.as_mut_ptr(), ids.as_mut_ptr(), &mut n) })?;
            let mut policy = vec![0f32; sys::SPB_CHESS_POLICY_SIZE];
            self.check(unsafe { sys::spb_chess_root_policy(self.raw, t.slot, policy.as_mut_ptr()) })?;
            mv.truncate(n as usize);
            out.push((policy, (0..n as usize).map(|i| (ids[i] as usize, cnt[i] as f32)).collect(), mv));
        }
        Ok(out)
    }
    /// ref: `Tree::use_subtree` mcts.rs:161 (child of the root); returns the new root state.
    pub fn use_subtree(&mut self, tree: &mut ChessTree, child_id: usize) -> Result<ChessState> {
        let id = child_id as u32;
        let mut st = ChessState::default();
        self.check(unsafe { sys::spb_chess_advance(self.raw, &tree.slot, &id, 1, &mut st) })?;
        Ok(st)
    }
    pub fn node_state(&mut self, tree: &ChessTree, node_id: usize) -> Result<ChessState> {
        let mut st = ChessState::default();
        self.check(unsafe { sys::spb_chess_get_state(self.raw, tree.slot, node_id as u32, &mut st) })?;
        Ok(st)
    }
    /// ref: `get_valid_actions` + `get_status` chess.rs:150-166 for a batch: (moves, status, repetitions) per state.
    pub fn legal_moves(&mut self, states: &[(ChessState, Vec<u64>)]) -> Result<Vec<(Vec<u16>, u8, u32)>> {
        let n = states.len();
        let st: Vec<ChessState> = states.iter().map(|s| s.0).collect();
        let hist: Vec<u64> = states.iter().flat_map(|s| Self::padded_history(&s.1)).collect();
        let mut mv = vec![0u16; n * sys::SPB_CHESS_MAX_MOVES];
        let (mut cnt, mut reps, mut status) = (vec![0u32; n], vec![0u32; n], vec![0u8; n]);
        self.check(unsafe { sys::spb_chess_legal_moves(self.raw, st.as_ptr(), hist.as_ptr(), n as u32, mv.as_mut_ptr(), cnt.as_mut_ptr(),
                                                       std::ptr::null_mut(), status.as_mut_ptr(), reps.as_mut_ptr()) })?;
        Ok((0..n).map(|i| (mv[i * sys::SPB_CHESS_MAX_MOVES..i * sys::SPB_CHESS_MAX_MOVES + cnt[i] as usize].to_vec(), status[i], reps[i])).collect())
    }
    /// ref: `get_next_state` chess.rs:112-148 for a batch; the history of a state that moved grows by one hash.
    pub fn next_states(&mut self, states: &[(ChessState, Vec<u64>)], moves: &[u16]) -> Result<Vec<std::result::Result<(ChessState, Vec<u64>), String>>> {
        let n = states.len();
        let st: Vec<ChessState> = states.iter().map(|s| s.0).collect();
        let mut hist: Vec<u64> = states.iter().flat_map(|s| Self::padded_history(&s.1)).collect();
        let mut out = vec![ChessState::default(); n];
        let mut err = vec![0i32; n];
        self.check(unsafe { sys::spb_chess_next_states(self.raw, st.as_ptr(), hist.as_mut_ptr(), moves.as_ptr(), n as u32, out.as_mut_ptr(), err.as_mut_ptr()) })?;
        Ok((0..n).map(|i| if err[i] == sys::SPB_OK {
            let h = &hist[i * sys::SPB_CHESS_MAX_HISTORY..i * sys::SPB_CHESS_MAX_HISTORY + out[i].hist_len as usize];
            Ok((out[i], h.to_vec()))
        } else if err[i] == sys::SPB_ERR_STATE { Err("game history full".to_string()) } else { Err("Failed to make move".to_string()) }).collect())
    }
    /// ref: `get_encoding` chess.rs:176-249 for a batch: `[n][19][8][8]`.
    pub fn encode(&mut self, states: &[(ChessState, Vec<u64>)]) -> Result<Vec<f32>> {
        let n = states.len();
        let st: Vec<ChessState> = states.iter().map(|s| s.0).collect();
        let hist: Vec<u64> = states.iter().flat_map(|s| Self::padded_history(&s.1)).collect();
        let mut out = vec![0f32; n * sys::SPB_CHESS_PLANES * 64];
        self.check(unsafe { sys::spb_chess_encode(self.raw, st.as_ptr(), hist.as_ptr(), n as u32, out.as_mut_ptr()) })?;
        Ok(out)
    }
    /// ref: `Model::predict` model/mod.rs:36-98: (policies `[n][4672]` masked + renormalised, values `[n]`).
    pub fn predict(&mut self, states: &[(ChessState, Vec<u64>)]) -> Result<(Vec<f32>, Vec<f32>)> {
        let n = states.len();
        let st: Vec<ChessState> = states.iter().map(|s| s.0).collect();
        let hist: Vec<u64> = states.iter().flat_map(|s| Self::padded_history(&s.1)).collect();
        let mut pol = vec![0f32; n * sys::SPB_CHESS_POLICY_SIZE];
        let mut val = vec![0f32; n];
        self.check(unsafe { sys::spb_chess_predict(self.raw, st.as_ptr(), hist.as_ptr(), n as u32, pol.as_mut_ptr(), val.as_mut_ptr(), std::ptr::null_mut()) })?;
        Ok((pol, val))
    }
    pub fn counters(&mut self) -> Result<sys::spb_counters> {
        let mut c = sys::spb_counters::default();
        self.check(unsafe { sys::spb_chess_get_counters(self.raw, &mut c) })?;
        Ok(c)
    }
    /// One self-play ply for every live chess game on the device (ref: learner_concurrent.rs:179-238): pick the move, record
    /// the root, `use_subtree` or finish the game; finished slots restart from `restart_roots` (one (state, history) per slot)
    /// or retire.  Returns the number of games that finished.  `Err` with `SPB_ERR_STATE`: the trajectory buffer is full —
    /// drain and call again, nothing is lost.
    pub fn self_play_step(&mut self, rule: MoveRule, restart_roots: Option<&[(ChessState, Vec<u64>)]>) -> Result<u32> {
        let (r, t, seed) = match rule {
            MoveRule::GreedyLastMax => (sys::SPB_MOVE_GREEDY_LAST_MAX, 0.0f32, 0u64),
            MoveRule::Temperature { temperature, seed } => (sys::SPB_MOVE_TEMPERATURE, temperature, seed),
        };
        let roots: Option<Vec<ChessState>> = restart_roots.map(|v| v.iter().map(|s| s.0).collect());
        let hist: Option<Vec<u64>> = restart_roots.map(|v| v.iter().flat_map(|s| Self::padded_history(&s.1)).collect());
        let p = roots.as_ref().map_or(std::ptr::null(), |v| v.as_ptr());
        let h = hist.as_ref().map_or(std::ptr::null(), |v| v.as_ptr());
        let mut finished = 0u32;
        self.check(unsafe { sys::spb_chess_selfplay_step(self.raw, r, t, seed, p, h, &mut finished) })?;
        Ok(finished)
    }
    /// Finished games' positions ordered by (game id, ply) with their global game ids (ref: learner_concurrent.rs:202-228).
    pub fn drain_trajectories(&mut self) -> Result<(Vec<ChessPosition>, Vec<u64>)> {
        let mut n = 0usize;
        self.check(unsafe { sys::spb_chess_drain_trajectories(self.raw, std::ptr::null_mut(), 0, &mut n, std::ptr::null_mut()) })?;
        // a record is plain integers: all-zero bytes are a valid value
        let mut pos: Vec<ChessPosition> = vec![unsafe { std::mem::zeroed() }; n];
        let mut ids = vec![0u64; n];
        if n > 0 {
            self.check(unsafe { sys::spb_chess_drain_trajectories(self.raw, pos.as_mut_ptr(), n, &mut n, ids.as_mut_ptr()) })?;
            pos.truncate(n); ids.truncate(n);
        }
        Ok((pos, ids))
    }
    /// Joins the NCCL communicator of the job (id from `comm_unique_id()` on rank 0, distributed by the host).
    pub fn comm_init(&mut self, id: &[u8; sys::SPB_COMM_ID_BYTES], rank: i32, world_size: i32) -> Result<()> {
        self.check(unsafe { sys::spb_chess_comm_init(self.raw, id.as_ptr(), rank, world_size) })
    }
    /// Leaves the communicator (dropping the engine does too).
    pub fn comm_destroy(&mut self) -> Result<()> {
        self.check(unsafe { sys::spb_chess_comm_destroy(self.raw) })
    }
    /// COLLECTIVE: every rank's finished chess trajectories to `learner_rank`, ordered by (game id, ply) — the replay-buffer
    /// push of the reference's workers (learner_concurrent.rs:281-288).  Empty on the other ranks.
    pub fn gather_trajectories(&mut self, learner_rank: i32) -> Result<(Vec<ChessPosition>, Vec<u64>)> {
        let mut n = 0usize;
        self.check(unsafe { sys::spb_chess_gather_trajectories(self.raw, learner_rank, std::ptr::null_mut(), 0, &mut n, std::ptr::null_mut()) })?;
        let mut pos: Vec<ChessPosition> = vec![unsafe { std::mem::zeroed() }; n];
        let mut ids = vec![0u64; n];
        if n > 0 {
            self.check(unsafe { sys::spb_chess_gather_trajectories(self.raw, learner_rank, pos.as_mut_ptr(), n, &mut n, ids.as_mut_ptr()) })?;
        }
        Ok((pos, ids))
    }
    /// The device form of `drain_trajectories` (see `Mcts::drain_trajectories_device`).
    ///
    /// # Safety
    /// As for `Mcts::drain_trajectories_device`.
    pub unsafe fn drain_trajectories_device(&mut self, buf_dev: *mut ChessPosition, capacity: usize, game_ids_dev: *mut u64) -> Result<usize> {
        let mut n = 0usize;
        self.check(sys::spb_chess_drain_trajectories_device(self.raw, buf_dev, capacity, &mut n, game_ids_dev))?;
        Ok(n)
    }
    /// COLLECTIVE: the device form of `gather_trajectories` (see `Mcts::gather_trajectories_device`).
    ///
    /// # Safety
    /// As for `Mcts::drain_trajectories_device`.
    pub unsafe fn gather_trajectories_device(&mut self, learner_rank: i32, buf_dev: *mut ChessPosition, capacity: usize,
                                             game_ids_dev: *mut u64) -> Result<usize> {
        let mut n = 0usize;
        self.check(sys::spb_chess_gather_trajectories_device(self.raw, learner_rank, buf_dev, capacity, &mut n, game_ids_dev))?;
        Ok(n)
    }
    /// The training tensors of `chess_positions_to_training`, built on this engine's GPU from records in its device memory
    /// (a replay buffer of `n_positions` records; ref: learner_concurrent.rs:87-165, :126-146).  Row i comes from
    /// `positions[indices[i]]`, or `positions[i]` when `indices` is null (then `n <= n_positions`).  Outputs (each nullable):
    /// `encodings[n][19][8][8]`, `policies[n][4672]`, `values[n]` f32, bit-identical to the host builder.  Returns once they are
    /// written; a malformed row is `SPB_ERR_ARG` and nothing is written.
    ///
    /// # Safety
    /// Every non-null pointer is device (or managed) memory of this engine's GPU, e.g. `Tensor::data_ptr` of CUDA tensors, and
    /// holds as many elements as stated; no other work writes the inputs or reads the outputs during the call.
    pub unsafe fn positions_to_training_device(&mut self, positions: *const ChessPosition, n_positions: usize, indices: *const u64, n: usize,
                                               encodings: *mut f32, policies: *mut f32, values: *mut f32) -> Result<()> {
        self.check(sys::spb_chess_positions_to_training_device(self.raw, positions, n_positions, indices, n, encodings, policies, values))
    }
}

pub type ChessPosition = sys::spb_chess_position;

/// Chess self-play records to the training tensors `[n][19][8][8]` / `[n][4672]` / `[n]` (host only): the encoding of the
/// recorded root, its visit counts / their sum at each move's policy index, the outcome.
pub fn chess_positions_to_training(positions: &[ChessPosition]) -> Result<TrainingBatch> {
    let n = positions.len();
    let mut b = TrainingBatch { n, encodings: vec![0f32; n * sys::SPB_CHESS_PLANES * 64], policies: vec![0f32; n * sys::SPB_CHESS_POLICY_SIZE], values: vec![0f32; n] };
    let rc = unsafe { sys::spb_chess_positions_to_training(positions.as_ptr(), n, b.encodings.as_mut_ptr(), b.policies.as_mut_ptr(), b.values.as_mut_ptr()) };
    if rc == sys::SPB_OK { Ok(b) } else { Err(Error { code: rc, message: "spb_chess_positions_to_training: bad argument".to_string() }) }
}

/// `State::default()` chess.rs:94-102.
pub fn chess_start_position() -> ChessState {
    let mut s = ChessState::default();
    unsafe { sys::spb_chess_start_position(&mut s) };
    s
}
/// `Policy::get_channel` chess.rs:311-390 and the flat index of `get_prob` / `set_prob` (:495-514).
pub fn chess_move_channel(side: i32, mv: u16) -> usize { unsafe { sys::spb_chess_move_channel(side, mv) as usize } }
pub fn chess_policy_index(side: i32, mv: u16) -> usize { unsafe { sys::spb_chess_policy_index(side, mv) as usize } }

impl Drop for ChessMcts {
    fn drop(&mut self) { unsafe { sys::spb_chess_destroy(self.raw); } }
}

fn chess_last_error(e: *const sys::spb_chess_engine) -> String {
    unsafe { CStr::from_ptr(sys::spb_chess_last_error(e)).to_string_lossy().into_owned() }
}
