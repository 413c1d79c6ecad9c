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


class ChessEngine(E.EngineBase):
    """The chess engine: `Mcts<chess Net>` + its trees on one GPU (ref: src/mcts.rs:41-44 over src/game/chess.rs and
    src/model/chess.rs) — batched `State` methods, search, re-rooting, `Model::predict`."""
    _PREFIX, _RECORD, _STATE, _ROOT_WIDTH, _MOVE = "spb_chess_", CHESS_POSITION_DTYPE, CHESS_STATE_DTYPE, MAX_MOVES, np.uint16
    A = POLICY_SIZE

    def __init__(self, num_games=64, evaluator=E.EVAL_NET, c=2.0, device=0, max_nodes_per_tree=0, flags=0, trajectory_capacity=0,
                 game_id_base=0, game_id_stride=0):
        super().__init__(game=E.GAME_CHESS, num_games=num_games, evaluator=evaluator, c=c, device=device,
                         max_nodes_per_tree=max_nodes_per_tree, flags=flags, leaves_per_tree=1,
                         trajectory_capacity=trajectory_capacity, game_id_base=game_id_base, game_id_stride=game_id_stride)

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

    # ---- Model::predict ----------------------------------------------------------------------------------------------
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

    def last_search_ms(self) -> float:
        ms = C.c_float()
        self._chk(self._L.spb_chess_last_search_ms(self._h, C.byref(ms)))
        return ms.value

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

    def get_state(self, slot: int, node_id: int) -> np.ndarray:
        out = np.zeros(1, CHESS_STATE_DTYPE)
        self._chk(self._L.spb_chess_get_state(self._h, slot, node_id, out.ctypes.data))
        return out[0]

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
        """Engine.counters, plus largest_arena: the largest arena_len of any tree."""
        c = self._read_counters()
        return dict(c.as_dict(), largest_arena=int(c.reserved[0]))


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
    positions: CHESS_POSITION_DTYPE numpy array (copied to the device) or a contiguous CUDA uint8 tensor [n_positions, 1624],
    e.g. a replay buffer kept in device memory.  indices (numpy or CUDA int64 / uint64 tensor): row i is built from
    positions[indices[i]]; without it every record is built.  A malformed row raises EngineError(-1) and nothing is written."""
    return E._positions_to_training_device(engine, positions, indices, (PLANES, 8, 8))


def check_weights(blob: bytes):
    """Host-only validation of a chess checkpoint -> (code, message)."""
    return E._check_weights(E.load_library().spb_chess_check_weights, blob)
