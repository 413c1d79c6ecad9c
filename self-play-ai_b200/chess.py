"""Chess rules on the device: ctypes wrappers of the spb_chess_* entry points (include/selfplay_b200.h).

Mirror of the reference's chess adapter, src/game/chess.rs: `get_valid_actions` / `get_status` (:150-166),
`get_next_state` (:112-148), `get_encoding` (:176-249), `Policy::get_channel` / `get_action` (:311-493).
A move is uint16 `from | to << 6 | promotion << 12`; squares are rank*8 + file.  `ChessEngine` adds the trees:
`Mcts::search` (mcts.rs:196-332), `Tree::use_subtree` (:161-192), `Model::predict` (model/mod.rs:36-98).  No CPU fallback:
every batched call runs kernels on the engine's device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import engine as E

MAX_MOVES, MAX_HISTORY, PLANES, POLICY_SIZE, NO_SQUARE = 256, 512, 19, 4672, 64
MOVE_NONE = 0xFFFF

CHESS_STATE_DTYPE = np.dtype([("piece", "<u8", (6,)), ("color", "<u8", (2,)), ("side", "u1"), ("castle", "u1"), ("ep", "u1"),
                              ("reserved0", "u1"), ("fifty", "<u2"), ("plies", "<u2"), ("hist_len", "<u4"), ("reserved1", "<u4")])
assert CHESS_STATE_DTYPE.itemsize == 80
# spb_chess_position: one searched root of a self-play trajectory (compact form of `Payload`, learner_concurrent.rs:13-18)
CHESS_POSITION_DTYPE = np.dtype([("state", CHESS_STATE_DTYPE), ("visit_counts", "<u4", (MAX_MOVES,)), ("moves", "<u2", (MAX_MOVES,)),
                                 ("n_moves", "<u2"), ("ply", "<u2"), ("repetitions", "u1"), ("outcome", "i1"), ("flags", "u1"),
                                 ("reserved", "u1")])
assert CHESS_POSITION_DTYPE.itemsize == 1624
POS_ADJUDICATED = 1          # CHESS_POSITION_DTYPE["flags"]: the game was ended as a tie at the history cap


def start_position() -> np.ndarray:
    """State::default() (chess.rs:94-102) -> array of one CHESS_STATE_DTYPE record."""
    s = np.zeros(1, CHESS_STATE_DTYPE)
    rc = E.load_library().spb_chess_start_position(s.ctypes.data)
    if rc != 0:
        raise E.EngineError(rc, "spb_chess_start_position")
    return s


def move_channel(side: int, move: int) -> int:
    return E.load_library().spb_chess_move_channel(side, move)


def policy_index(side: int, move: int) -> int:
    return E.load_library().spb_chess_policy_index(side, move)


def action(side: int, channel: int, row: int, col: int) -> int:
    return E.load_library().spb_chess_action(side, channel, row, col)


def _states(states) -> np.ndarray:
    a = np.ascontiguousarray(states, dtype=CHESS_STATE_DTYPE)
    return a.reshape(-1)


def _history(history, n):
    if history is None:
        return None
    h = np.ascontiguousarray(history, dtype=np.uint64)
    assert h.shape == (n, MAX_HISTORY), h.shape
    return h


class ChessEngine:
    """The chess engine: `Mcts<chess Net>` + its trees on one GPU (ref: src/mcts.rs:41-44 over src/game/chess.rs and
    src/model/chess.rs) — batched `State` methods, search, re-rooting, `Model::predict`."""

    def __init__(self, num_games=64, evaluator=E.EVAL_NET, c=2.0, device=0, max_nodes_per_tree=0, flags=0, trajectory_capacity=0,
                 game_id_base=0, game_id_stride=0):
        L = E.load_library()
        cfg = E.Config()
        L.spb_default_config(C.byref(cfg))
        cfg.game, cfg.num_games, cfg.evaluator, cfg.c, cfg.device = E.GAME_CHESS, num_games, evaluator, c, device
        cfg.max_nodes_per_tree, cfg.flags, cfg.leaves_per_tree = max_nodes_per_tree, flags, 1
        cfg.trajectory_capacity, cfg.game_id_base, cfg.game_id_stride = trajectory_capacity, game_id_base, game_id_stride
        h = C.c_void_p()
        rc = L.spb_chess_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise E.EngineError(rc, L.spb_chess_last_error(None).decode())
        self._h, self._L, self.G, self.device = h, L, num_games, device

    def close(self):
        if getattr(self, "_h", None):
            self._L.spb_chess_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _chk(self, rc):
        if rc != 0:
            raise E.EngineError(rc, self._L.spb_chess_last_error(self._h).decode())

    # ---- State trait, batched ----------------------------------------------------------------------------------------
    def legal_moves(self, states, history=None):
        """-> (moves[n,256] u16 sorted by (from,to,promotion), counts[n], policy_index[n,256], status[n], repetitions[n])."""
        st = _states(states)
        n = len(st)
        h = _history(history, n)
        moves = np.zeros((n, MAX_MOVES), np.uint16)
        pidx = np.zeros((n, MAX_MOVES), np.uint16)
        counts, reps, status = np.zeros(n, np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.uint8)
        self._chk(self._L.spb_chess_legal_moves(self._h, st.ctypes.data, None if h is None else h.ctypes.data, n, moves.ctypes.data,
                                                counts.ctypes.data, pidx.ctypes.data, status.ctypes.data, reps.ctypes.data))
        return moves, counts, pidx, status, reps

    def next_states(self, states, history, moves):
        """get_next_state for n states -> (out_states, history (updated copy), err[n])."""
        st = _states(states)
        n = len(st)
        h = np.array(_history(history, n), copy=True)
        mv = np.ascontiguousarray(moves, dtype=np.uint16)
        out = np.zeros(n, CHESS_STATE_DTYPE)
        err = np.zeros(n, np.int32)
        self._chk(self._L.spb_chess_next_states(self._h, st.ctypes.data, h.ctypes.data, mv.ctypes.data, n, out.ctypes.data, err.ctypes.data))
        return out, h, err

    def encode(self, states, history=None) -> np.ndarray:
        st = _states(states)
        n = len(st)
        h = _history(history, n)
        out = np.zeros((n, PLANES, 8, 8), np.float32)
        self._chk(self._L.spb_chess_encode(self._h, st.ctypes.data, None if h is None else h.ctypes.data, n, out.ctypes.data))
        return out

    def perft(self, state, depth: int) -> int:
        st = _states(state)
        assert len(st) == 1
        nodes = C.c_uint64()
        self._chk(self._L.spb_chess_perft(self._h, st.ctypes.data, depth, C.byref(nodes)))
        return int(nodes.value)

    # ---- weights / Model::predict ------------------------------------------------------------------------------------
    def load_weights(self, blob: bytes):
        buf = (C.c_char * len(blob)).from_buffer_copy(blob)
        self._chk(self._L.spb_chess_load_weights(self._h, C.cast(buf, C.c_void_p), len(blob)))

    def predict(self, states, history=None, want_logits=False):
        st = _states(states)
        n = len(st)
        h = _history(history, n)
        pol = np.zeros((n, POLICY_SIZE), np.float32)
        val = np.zeros(n, np.float32)
        lg = np.zeros((n, POLICY_SIZE), np.float32) if want_logits else None
        self._chk(self._L.spb_chess_predict(self._h, st.ctypes.data, None if h is None else h.ctypes.data, n, pol.ctypes.data, val.ctypes.data,
                                            None if lg is None else lg.ctypes.data))
        return (pol, val, lg) if want_logits else (pol, val)

    # ---- trees -------------------------------------------------------------------------------------------------------
    def reset_games(self, roots=None, history=None, slots=None):
        n = self.G if slots is None else len(slots)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.uint32)
        st = None if roots is None else _states(roots)
        h = None if history is None else _history(history, n)
        if st is not None:
            assert len(st) == n
        self._chk(self._L.spb_chess_reset_games(self._h, None if sl is None else sl.ctypes.data, n, None if st is None else st.ctypes.data,
                                                None if h is None else h.ctypes.data))

    def search(self, num_searches: int):
        self._chk(self._L.spb_chess_search(self._h, num_searches))

    def last_search_ms(self) -> float:
        ms = C.c_float()
        self._chk(self._L.spb_chess_last_search_ms(self._h, C.byref(ms)))
        return ms.value

    def root_children(self, slot: int):
        mv, cnt, ids = np.zeros(MAX_MOVES, np.uint16), np.zeros(MAX_MOVES, np.uint32), np.zeros(MAX_MOVES, np.uint32)
        n = C.c_uint32()
        self._chk(self._L.spb_chess_root_children(self._h, slot, mv.ctypes.data, cnt.ctypes.data, ids.ctypes.data, C.byref(n)))
        k = n.value
        return mv[:k].tolist(), cnt[:k].tolist(), ids[:k].tolist()

    def root_children_all(self, out=None):
        """`out`: the four arrays of an earlier call (e.g. in pinned host memory), written in place."""
        if out is not None:
            mv, cnt, ids, n = out
            assert mv.shape == (self.G, MAX_MOVES) and mv.dtype == np.uint16 and cnt.dtype == np.uint32 and ids.dtype == np.uint32 and n.shape == (self.G,)
            assert all(x.flags.c_contiguous for x in out)
        else:
            mv = np.zeros((self.G, MAX_MOVES), np.uint16)
            cnt = np.zeros((self.G, MAX_MOVES), np.uint32)
            ids = np.zeros((self.G, MAX_MOVES), np.uint32)
            n = np.zeros(self.G, np.uint32)
        self._chk(self._L.spb_chess_root_children_all(self._h, mv.ctypes.data, cnt.ctypes.data, ids.ctypes.data, n.ctypes.data))
        return mv, cnt, ids, n

    def root_policy(self, slot: int) -> np.ndarray:
        p = np.zeros(POLICY_SIZE, np.float32)
        self._chk(self._L.spb_chess_root_policy(self._h, slot, p.ctypes.data))
        return p

    # ---- EXTENSION: Dirichlet noise at the root (DESIGN.md §4.6) ------------------------------
    def set_root_noise(self, alpha: float, epsilon: float, seed: int = 0):
        """P' = (1 - epsilon) P + epsilon eta, eta ~ Dir(alpha), at the root of every search; epsilon = 0 turns it off."""
        self._chk(self._L.spb_chess_set_root_noise(self._h, alpha, epsilon, seed))

    def root_noise(self, slot: int) -> np.ndarray:
        """The eta the next search of `slot`'s root uses, one entry per legal move of the root (child order)."""
        eta = np.zeros(MAX_MOVES, np.float32)
        n = C.c_uint32()
        self._chk(self._L.spb_chess_root_noise(self._h, slot, eta.ctypes.data_as(C.POINTER(C.c_float)), C.byref(n)))
        return eta[:n.value].copy()

    def advance(self, child_ids, slots=None) -> np.ndarray:
        ids = np.ascontiguousarray(child_ids, dtype=np.uint32)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.uint32)
        out = np.zeros(len(ids), CHESS_STATE_DTYPE)
        self._chk(self._L.spb_chess_advance(self._h, None if sl is None else sl.ctypes.data, ids.ctypes.data, len(ids), out.ctypes.data))
        return out

    # ---- self-play (ref: SelfPlayWorker::self_play, learner_concurrent.rs:169-242) --------------------------------------
    def selfplay_step(self, rule=E.MOVE_GREEDY_LAST_MAX, temperature=1.25, seed=0, restart_roots=None, restart_history=None) -> int:
        """One ply for every live slot on the device -> number of games finished (emitted) by this call.  restart_roots /
        restart_history: num_games entries, as for reset_games.  A full trajectory buffer raises EngineError(-6): drain and
        call again, nothing is lost."""
        st = None if restart_roots is None else _states(restart_roots)
        h = None if restart_history is None else _history(restart_history, self.G)
        if st is not None:
            assert len(st) == self.G
        fin = C.c_uint32()
        self._chk(self._L.spb_chess_selfplay_step(self._h, rule, temperature, seed, None if st is None else st.ctypes.data,
                                                  None if h is None else h.ctypes.data, C.byref(fin)))
        return fin.value

    def drain_trajectories(self):
        """-> (positions[CHESS_POSITION_DTYPE], game_ids[u64]) ordered by (game id, ply)."""
        n = C.c_size_t()
        self._chk(self._L.spb_chess_drain_trajectories(self._h, None, 0, C.byref(n), None))
        pos = np.zeros(n.value, dtype=CHESS_POSITION_DTYPE)
        ids = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            self._chk(self._L.spb_chess_drain_trajectories(self._h, pos.ctypes.data, n.value, C.byref(n), ids.ctypes.data))
        return pos[:n.value], ids[:n.value]

    def drain_trajectories_device(self, out=None, ids_out=None):
        """The records of drain_trajectories, ordered on the device -> (CUDA uint8 [n, 1624], CUDA int64 [n]); out / ids_out as
        for Engine.drain_trajectories_device."""
        return E._records_to_device(
            lambda b, cap, n, i: self._chk(self._L.spb_chess_drain_trajectories_device(self._h, b, cap, n, i)),
            self.device, CHESS_POSITION_DTYPE.itemsize, out, ids_out)

    # ---- multi-GPU: trajectories to the learner rank (the contract of Engine's methods) -------------------------------
    def comm_init(self, comm_id: bytes, rank: int, world_size: int):
        buf = (C.c_uint8 * E.COMM_ID_BYTES).from_buffer_copy(comm_id)
        self._chk(self._L.spb_chess_comm_init(self._h, C.cast(buf, C.c_void_p), rank, world_size))

    def comm_destroy(self):
        self._chk(self._L.spb_chess_comm_destroy(self._h))

    def gather_trajectories(self, learner_rank: int = 0):
        """COLLECTIVE: -> (positions[CHESS_POSITION_DTYPE], game_ids) ordered by (game id, ply) on the learner rank, empty
        elsewhere."""
        n = C.c_size_t()
        self._chk(self._L.spb_chess_gather_trajectories(self._h, learner_rank, None, 0, C.byref(n), None))
        pos = np.zeros(n.value, dtype=CHESS_POSITION_DTYPE)
        ids = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            self._chk(self._L.spb_chess_gather_trajectories(self._h, learner_rank, pos.ctypes.data, n.value, C.byref(n), ids.ctypes.data))
        return pos[:n.value], ids[:n.value]

    def gather_trajectories_device(self, learner_rank: int = 0, out=None, ids_out=None):
        """COLLECTIVE: gather_trajectories into device memory of the learner rank -> (CUDA uint8 [n, 1624], CUDA int64 [n]),
        empty elsewhere."""
        return E._records_to_device(
            lambda b, cap, n, i: self._chk(self._L.spb_chess_gather_trajectories_device(self._h, learner_rank, b, cap, n, i)),
            self.device, CHESS_POSITION_DTYPE.itemsize, out, ids_out)

    def get_state(self, slot: int, node_id: int) -> np.ndarray:
        out = np.zeros(1, CHESS_STATE_DTYPE)
        self._chk(self._L.spb_chess_get_state(self._h, slot, node_id, out.ctypes.data))
        return out[0]

    def arena_len(self, slot: int) -> int:
        n = C.c_uint32()
        self._chk(self._L.spb_chess_arena_len(self._h, slot, C.byref(n)))
        return n.value

    def node_stats(self, slot: int, node_id: int) -> dict:
        n, fc, nc = C.c_uint32(), C.c_uint32(), C.c_uint32()
        w, p = C.c_float(), C.c_float()
        mv, st = C.c_uint16(), C.c_uint8()
        self._chk(self._L.spb_chess_node_stats(self._h, slot, node_id, C.byref(n), C.byref(w), C.byref(p), C.byref(fc), C.byref(nc),
                                               C.byref(mv), C.byref(st)))
        return dict(visit_count=n.value, value_sum=w.value, prior=p.value, first_child=fc.value, n_children=nc.value, move=mv.value,
                    status=st.value)

    def time_conv(self, iters=20):
        """-> (avg launch ms, positions in the batch, FLOPs per launch, FLOPs per evaluated position) of the residual conv kernel
        re-run on the last evaluator batch (spb_chess_time_conv)."""
        ms, n, fl, fp = C.c_float(), C.c_uint32(), C.c_double(), C.c_double()
        self._chk(self._L.spb_chess_time_conv(self._h, iters, C.byref(ms), C.byref(n), C.byref(fl), C.byref(fp)))
        return ms.value, n.value, fl.value, fp.value

    def counters(self) -> dict:
        c = E.Counters()
        self._chk(self._L.spb_chess_get_counters(self._h, C.byref(c)))
        d = c.as_dict()
        d["largest_arena"] = int(c.reserved[0])
        return d

    def reset_counters(self):
        self._chk(self._L.spb_chess_reset_counters(self._h))


def positions_to_training(positions):
    """spb_chess_positions_to_training (host only): -> (encodings[n,19,8,8], policies[n,4672], values[n,1]) f32, the training
    tensors of chess self-play records."""
    L = E.load_library()
    pos = np.ascontiguousarray(positions, dtype=CHESS_POSITION_DTYPE).reshape(-1)
    n = len(pos)
    enc = np.zeros((n, PLANES, 8, 8), np.float32)
    pol = np.zeros((n, POLICY_SIZE), np.float32)
    val = np.zeros((n, 1), np.float32)
    rc = L.spb_chess_positions_to_training(pos.ctypes.data, n, enc.ctypes.data, pol.ctypes.data, val.ctypes.data)
    if rc != 0:
        raise E.EngineError(rc, "spb_chess_positions_to_training: bad argument")
    return enc, pol, val


def positions_to_training_device(engine: ChessEngine, positions, indices=None):
    """spb_chess_positions_to_training_device: the tensors of positions_to_training, built on the engine's GPU ->
    torch CUDA tensors (encodings[n,19,8,8], policies[n,4672], values[n,1]) f32, bit-identical to the host builder.
    positions: CHESS_POSITION_DTYPE numpy array (copied to the device) or a CUDA uint8 tensor [n_positions, 1624], e.g. a
    replay buffer kept in device memory.  indices (numpy or CUDA int64 / uint64 tensor): row i is built from
    positions[indices[i]]; without it every record is built.  A malformed row raises EngineError(-1) and nothing is written."""
    import torch
    dev = torch.device("cuda", engine.device)
    if isinstance(positions, torch.Tensor):
        assert positions.is_cuda and positions.dtype == torch.uint8 and positions.dim() == 2 and positions.shape[1] == CHESS_POSITION_DTYPE.itemsize, \
            (positions.device, positions.dtype, tuple(positions.shape))
        pos = positions.contiguous()
    else:
        a = np.ascontiguousarray(positions, dtype=CHESS_POSITION_DTYPE).reshape(-1)
        pos = torch.from_numpy(a.view(np.uint8).reshape(len(a), CHESS_POSITION_DTYPE.itemsize)).to(dev)
    idx = None
    if indices is not None:
        if isinstance(indices, torch.Tensor):
            assert indices.is_cuda and indices.dtype in (torch.int64, torch.uint64) and indices.dim() == 1, (indices.device, indices.dtype)
            idx = indices.contiguous()
        else:
            i = np.ascontiguousarray(indices).reshape(-1)
            assert i.dtype.kind in "iu", i.dtype
            idx = torch.from_numpy(i.astype(np.int64)).to(dev)
    n = len(pos) if idx is None else len(idx)
    enc = torch.empty((n, PLANES, 8, 8), dtype=torch.float32, device=dev)
    pol = torch.empty((n, POLICY_SIZE), dtype=torch.float32, device=dev)
    val = torch.empty((n, 1), dtype=torch.float32, device=dev)
    torch.cuda.current_stream(dev).synchronize()                       # the engine's stream reads the inputs
    engine._chk(engine._L.spb_chess_positions_to_training_device(
        engine._h, pos.data_ptr() if len(pos) else None, len(pos), None if idx is None else idx.data_ptr(), n,
        enc.data_ptr(), pol.data_ptr(), val.data_ptr()))
    return enc, pol, val


def check_weights(blob: bytes):
    """Host-only validation of a chess checkpoint -> (code, message)."""
    L = E.load_library()
    buf = (C.c_char * len(blob)).from_buffer_copy(blob)
    err = C.create_string_buffer(512)
    rc = L.spb_chess_check_weights(C.cast(buf, C.c_void_p), len(blob), err, 512)
    return rc, err.value.decode()
