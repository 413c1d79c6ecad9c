"""ctypes binding of include/selfplay_b200.h (the C ABI a Rust `-sys` crate would bind, see INTEGRATION.md)."""
from __future__ import annotations

import ctypes as C
import functools
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "libselfplay_b200.so")

GAME_TTT, GAME_C4, GAME_CHESS = 0, 1, 2
EVAL_NET, EVAL_DET, EVAL_UNIFORM = 0, 1, 2
ONGOING, TIED, WON = 0, 1, 2
MAX_ACTIONS = 9
NUM_ACTIONS = {GAME_TTT: 9, GAME_C4: 7}
BOARD = {GAME_TTT: (3, 3), GAME_C4: (6, 7)}
FLAG_NO_GRAPH, FLAG_EVAL_SIMT, FLAG_FORCE_SPLIT, FLAG_FIXED_POOL, FLAG_LOCKSTEP = 1, 2, 4, 16, 32
MOVE_GREEDY_LAST_MAX, MOVE_TEMPERATURE = 0, 1
ABI_VERSION = 2


class EngineError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("selfplay_b200 error %d: %s" % (code, msg))
        self.code = code


class State(C.Structure):
    """spb_state — replaces `State` (connect_four.rs:20-26 / tictactoe.rs:20-26)."""
    _fields_ = [("stones", C.c_uint64 * 2), ("current_player", C.c_uint8), ("num_actions_played", C.c_uint8),
                ("status", C.c_uint8), ("reserved", C.c_uint8 * 5)]

    def key(self):
        return (int(self.stones[0]), int(self.stones[1]), int(self.current_player),
                int(self.num_actions_played), int(self.status))

    def __repr__(self):
        return "State(x=%#x,o=%#x,p=%d,n=%d,st=%d)" % self.key()


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("game", C.c_int32), ("device", C.c_int32), ("num_games", C.c_uint32),
                ("max_nodes_per_tree", C.c_uint32), ("leaves_per_tree", C.c_uint32), ("c", C.c_float),
                ("evaluator", C.c_int32), ("flags", C.c_uint32), ("game_id_base", C.c_uint32),
                ("game_id_stride", C.c_uint32), ("trajectory_capacity", C.c_uint32), ("reserved", C.c_uint32 * 4)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("simulations", "evaluations", "terminal_leaves", "path_length_sum",
                                          "children_created", "nodes_live", "kernel_launches")] + \
               [("reserved", C.c_uint64 * 5)]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_ if n != "reserved"}


class Position(C.Structure):
    _fields_ = [("stones", C.c_uint64 * 2), ("visit_counts", C.c_uint32 * MAX_ACTIONS), ("current_player", C.c_uint8),
                ("ply", C.c_uint8), ("outcome", C.c_int8), ("reserved", C.c_uint8)]


STATE_DTYPE = np.dtype([("stones", "<u8", (2,)), ("current_player", "u1"), ("num_actions_played", "u1"),
                        ("status", "u1"), ("reserved", "u1", (5,))])
POSITION_DTYPE = np.dtype([("stones", "<u8", (2,)), ("visit_counts", "<u4", (MAX_ACTIONS,)), ("current_player", "u1"),
                           ("ply", "u1"), ("outcome", "i1"), ("reserved", "u1")])
assert STATE_DTYPE.itemsize == C.sizeof(State) == 24
assert POSITION_DTYPE.itemsize == C.sizeof(Position) == 56

DTYPE_F32, DTYPE_BF16, DTYPE_F64, DTYPE_F16 = 0, 1, 2, 3


class Tensor(C.Structure):
    """spb_tensor: one entry of the table spb_load_weights_device reads (a device tensor and its checkpoint name)."""
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int32), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


assert C.sizeof(Tensor) == 56

# Every symbol include/selfplay_b200.h declares: name -> (restype, argtypes)
_u32p, _u8p, _f32p, _i32p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_int32)
_vp = C.c_void_p
ABI = {
    "spb_abi_version": (C.c_int32, []),
    "spb_default_config": (C.c_int32, [C.POINTER(Config)]),
    "spb_create": (C.c_int32, [C.POINTER(Config), C.POINTER(_vp)]),
    "spb_destroy": (C.c_int32, [_vp]),
    "spb_last_error": (C.c_char_p, [_vp]),
    "spb_load_weights": (C.c_int32, [_vp, _vp, C.c_size_t]),
    "spb_check_weights": (C.c_int32, [C.c_int32, _vp, C.c_size_t, C.c_char_p, C.c_size_t]),
    "spb_load_weights_device": (C.c_int32, [_vp, C.POINTER(Tensor), C.c_uint32]),
    "spb_broadcast_weights": (C.c_int32, [_vp, C.c_int32]),
    "spb_reset_games": (C.c_int32, [_vp, _vp, C.c_uint32, _vp]),
    "spb_search": (C.c_int32, [_vp, C.c_uint32]),
    "spb_root_children": (C.c_int32, [_vp, C.c_uint32, _u8p, _u32p, _u32p, _u32p]),
    "spb_root_children_all": (C.c_int32, [_vp, _vp, _vp, _vp, _vp]),
    "spb_root_policy": (C.c_int32, [_vp, C.c_uint32, _f32p]),
    "spb_advance": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp]),
    "spb_get_state": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.POINTER(State)]),
    "spb_arena_len": (C.c_int32, [_vp, C.c_uint32, _u32p]),
    "spb_node_stats": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _u32p, _f32p, _f32p, _u32p, _u32p]),
    "spb_set_root_noise": (C.c_int32, [_vp, C.c_float, C.c_float, C.c_uint64]),
    "spb_root_noise": (C.c_int32, [_vp, C.c_uint32, _f32p, _u32p]),
    "spb_predict": (C.c_int32, [_vp, _vp, C.c_uint32, _vp, _vp, _vp]),
    "spb_game_next_states": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp, _vp]),
    "spb_game_valid_actions": (C.c_int32, [_vp, _vp, C.c_uint32, _vp]),
    "spb_game_encode": (C.c_int32, [_vp, _vp, C.c_uint32, _vp]),
    "spb_selfplay_step": (C.c_int32, [_vp, C.c_int32, C.c_float, C.c_uint64, _vp, _u32p]),
    "spb_drain_trajectories": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_drain_trajectories_device": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_comm_unique_id": (C.c_int32, [_vp]),
    "spb_comm_init": (C.c_int32, [_vp, _vp, C.c_int32, C.c_int32]),
    "spb_comm_destroy": (C.c_int32, [_vp]),
    "spb_gather_trajectories": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_gather_trajectories_device": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_positions_to_training": (C.c_int32, [C.c_int32, _vp, C.c_size_t, _vp, _vp, _vp]),
    "spb_positions_to_training_device": (C.c_int32, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp, _vp, _vp]),
    # chess (ref: src/game/chess.rs, src/model/chess.rs); typed wrappers in chess.py
    "spb_chess_create": (C.c_int32, [C.POINTER(Config), C.POINTER(_vp)]),
    "spb_chess_destroy": (C.c_int32, [_vp]),
    "spb_chess_last_error": (C.c_char_p, [_vp]),
    "spb_chess_load_weights": (C.c_int32, [_vp, _vp, C.c_size_t]),
    "spb_chess_check_weights": (C.c_int32, [_vp, C.c_size_t, C.c_char_p, C.c_size_t]),
    "spb_chess_load_weights_device": (C.c_int32, [_vp, C.POINTER(Tensor), C.c_uint32]),
    "spb_chess_broadcast_weights": (C.c_int32, [_vp, C.c_int32]),
    "spb_chess_start_position": (C.c_int32, [_vp]),
    "spb_chess_legal_moves": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp]),
    "spb_chess_next_states": (C.c_int32, [_vp, _vp, _vp, _vp, C.c_uint32, _vp, _vp]),
    "spb_chess_encode": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp]),
    "spb_chess_perft": (C.c_int32, [_vp, _vp, C.c_uint32, C.POINTER(C.c_uint64)]),
    "spb_chess_move_channel": (C.c_int32, [C.c_int32, C.c_uint16]),
    "spb_chess_policy_index": (C.c_int32, [C.c_int32, C.c_uint16]),
    "spb_chess_action": (C.c_uint16, [C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "spb_chess_reset_games": (C.c_int32, [_vp, _vp, C.c_uint32, _vp, _vp]),
    "spb_chess_search": (C.c_int32, [_vp, C.c_uint32]),
    "spb_chess_last_search_ms": (C.c_int32, [_vp, _f32p]),
    "spb_chess_root_children": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, _vp, _u32p]),
    "spb_chess_root_children_all": (C.c_int32, [_vp, _vp, _vp, _vp, _vp]),
    "spb_chess_root_policy": (C.c_int32, [_vp, C.c_uint32, _vp]),
    "spb_chess_advance": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp]),
    "spb_chess_get_state": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp]),
    "spb_chess_arena_len": (C.c_int32, [_vp, C.c_uint32, _u32p]),
    "spb_chess_node_stats": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _u32p, _f32p, _f32p, _u32p, _u32p, C.POINTER(C.c_uint16), _u8p]),
    "spb_chess_set_root_noise": (C.c_int32, [_vp, C.c_float, C.c_float, C.c_uint64]),
    "spb_chess_root_noise": (C.c_int32, [_vp, C.c_uint32, _f32p, _u32p]),
    "spb_chess_predict": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, _vp, _vp, _vp]),
    "spb_chess_time_conv": (C.c_int32, [_vp, C.c_uint32, _f32p, _u32p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "spb_chess_get_counters": (C.c_int32, [_vp, C.POINTER(Counters)]),
    "spb_chess_reset_counters": (C.c_int32, [_vp]),
    "spb_chess_selfplay_step": (C.c_int32, [_vp, C.c_int32, C.c_float, C.c_uint64, _vp, _vp, _u32p]),
    "spb_chess_drain_trajectories": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_chess_drain_trajectories_device": (C.c_int32, [_vp, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_chess_positions_to_training": (C.c_int32, [_vp, C.c_size_t, _vp, _vp, _vp]),
    "spb_chess_positions_to_training_device": (C.c_int32, [_vp, _vp, C.c_size_t, _vp, C.c_size_t, _vp, _vp, _vp]),
    "spb_chess_comm_init": (C.c_int32, [_vp, _vp, C.c_int32, C.c_int32]),
    "spb_chess_comm_destroy": (C.c_int32, [_vp]),
    "spb_chess_gather_trajectories": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_chess_gather_trajectories_device": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, C.POINTER(C.c_size_t), _vp]),
    "spb_get_counters": (C.c_int32, [_vp, C.POINTER(Counters)]),
    "spb_reset_counters": (C.c_int32, [_vp]),
    "spb_last_search_timing": (C.c_int32, [_vp, _f32p, _f32p, _u32p]),
    "spb_synchronize": (C.c_int32, [_vp]),
    "spb_last_async_stats": (C.c_int32, [_vp, C.POINTER(C.c_uint64), C.c_uint32]),
    "spb_time_evaluator": (C.c_int32, [_vp, C.c_uint32, _f32p, _u32p, C.POINTER(C.c_double)]),
}


def library_path() -> str:
    return _LIB


def build_library(verbose: bool = False) -> str:
    """Compiles csrc/ for sm_100a with nvcc (cross-compiles without a GPU)."""
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc")] + ([] if verbose else ["-s"]),
                          stdout=None if verbose else subprocess.DEVNULL)
    return _LIB


_lib = None


def load_library():
    """Loads libselfplay_b200.so.  Raises (never falls back) when the CUDA library is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB):
            raise EngineError(-2, "libselfplay_b200.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                                  "there is no CPU fallback")
        L = C.CDLL(_LIB)
        for name, (res, args) in ABI.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def states_array(states) -> np.ndarray:
    if isinstance(states, np.ndarray):
        assert states.dtype == STATE_DTYPE
        return np.ascontiguousarray(states)
    arr = np.zeros(len(states), dtype=STATE_DTYPE)
    for i, s in enumerate(states):
        arr[i]["stones"] = (s.stones[0], s.stones[1])
        arr[i]["current_player"] = s.current_player
        arr[i]["num_actions_played"] = s.num_actions_played
        arr[i]["status"] = s.status
    return arr


def check_weights(game: int, blob: bytes):
    """Host-only checkpoint validation -> (code, message)."""
    return _check_weights(functools.partial(load_library().spb_check_weights, game), blob)


def _check_weights(call, blob: bytes):
    """check_weights and chess.check_weights: `call(blob, size, err, err_cap)` is the entry point, its game bound."""
    buf = (C.c_char * len(blob)).from_buffer_copy(blob)
    err = C.create_string_buffer(512)
    rc = call(C.cast(buf, _vp), len(blob), err, 512)
    return rc, err.value.decode()


COMM_ID_BYTES = 128


def comm_unique_id() -> bytes:
    """spb_comm_unique_id: the 128-byte NCCL id rank 0 creates and the host distributes to every rank."""
    L = load_library()
    buf = (C.c_uint8 * COMM_ID_BYTES)()
    rc = L.spb_comm_unique_id(C.cast(buf, _vp))
    if rc != 0:
        raise EngineError(rc, L.spb_last_error(None).decode())
    return bytes(buf)


def positions_to_training(game: int, positions: np.ndarray):
    """spb_positions_to_training (host only): -> (encodings[n,3,R,C], policies[n,A], values[n,1]) f32 — the tensors of
    learner_concurrent.rs:126-146."""
    L = load_library()
    pos = np.ascontiguousarray(positions, dtype=POSITION_DTYPE)
    n = len(pos)
    R, Cc = BOARD[game]
    enc = np.zeros((n, 3, R, Cc), np.float32)
    pol = np.zeros((n, NUM_ACTIONS[game]), np.float32)
    val = np.zeros((n, 1), np.float32)
    rc = L.spb_positions_to_training(game, pos.ctypes.data, n, enc.ctypes.data, pol.ctypes.data, val.ctypes.data)
    if rc != 0:
        raise EngineError(rc, "spb_positions_to_training: bad argument")
    return enc, pol, val


def _dtype_codes():
    import torch
    return {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float64: DTYPE_F64, torch.float16: DTYPE_F16}


def tensor_table(named, device):
    """(name, tensor) pairs (a mapping or an iterable, e.g. a module's state_dict() or tch's VarStore::variables()) ->
    (ctypes array of spb_tensor, n, the encoded names to keep alive for the call).  Every tensor must be a contiguous CUDA
    tensor on `device` of at most 4 dimensions, in f32, bf16 or f64 (f16 is passed on and refused by the library, as in a
    checkpoint)."""
    import torch
    items = list(named.items()) if hasattr(named, "items") else list(named)
    codes = _dtype_codes()
    table = (Tensor * max(len(items), 1))()
    names = []
    for i, (name, t) in enumerate(items):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise TypeError("%s must be a CUDA tensor" % name)
        if t.device.index != device:
            raise ValueError("%s is on %s, the engine on cuda:%d" % (name, t.device, device))
        if not t.is_contiguous():
            raise ValueError("%s must be contiguous" % name)
        if t.dim() > 4 or t.dtype not in codes:
            raise ValueError("%s: %d dimensions of %s (at most 4 of float32, bfloat16, float64)" % (name, t.dim(), t.dtype))
        names.append(name.encode())
        table[i].name, table[i].data = names[-1], t.data_ptr()
        table[i].dtype, table[i].ndim = codes[t.dtype], t.dim()
        for k, d in enumerate(t.shape):
            table[i].shape[k] = d
    return table, len(items), names


def _check_cuda_tensor(t, dtype, width, name):
    """Raises unless t is a contiguous CUDA tensor of `dtype`, [n, width] (width None: [n])."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a CUDA tensor, not %s" % (name, type(t).__name__))
    if t.dtype not in ((dtype,) if not isinstance(dtype, tuple) else dtype):
        raise TypeError("%s must be %s, not %s" % (name, dtype, t.dtype))
    if (width is None and t.dim() != 1) or (width is not None and (t.dim() != 2 or t.shape[1] != width)):
        raise ValueError("%s must be [n%s], not %s" % (name, "" if width is None else ", %d" % width, tuple(t.shape)))
    if not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor, not on %s" % (name, t.device))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)


def positions_to_training_device(engine: "Engine", positions, indices=None):
    """spb_positions_to_training_device: the tensors of positions_to_training(engine.game, ...), built on the engine's GPU
    -> torch CUDA tensors (encodings[n,3,R,C], policies[n,A], values[n,1]) f32, bit-identical to the host builder.
    positions: POSITION_DTYPE numpy array (copied to the device) or a CUDA uint8 tensor [n_positions, 56], e.g. a replay
    buffer kept in device memory.  indices (numpy or CUDA int64 / uint64 tensor): row i is built from
    positions[indices[i]]; without it every record is built.  An index out of range raises EngineError(-1) and nothing is
    written."""
    return _positions_to_training_device(engine, positions, indices, (3,) + BOARD[engine.game])


def _positions_to_training_device(engine, positions, indices, encoding_shape):
    """positions_to_training_device and chess.positions_to_training_device: records of the engine's record dtype, an
    encoding of `encoding_shape` and a policy of engine.A entries per row."""
    import torch
    width = engine._RECORD.itemsize
    if isinstance(positions, torch.Tensor):
        _check_cuda_tensor(positions, torch.uint8, width, "positions")
        pos = positions
    if indices is not None and isinstance(indices, torch.Tensor):
        _check_cuda_tensor(indices, (torch.int64, torch.uint64), None, "indices")
    dev = torch.device("cuda", engine.device)
    if not isinstance(positions, torch.Tensor):
        a = np.ascontiguousarray(positions, dtype=engine._RECORD).reshape(-1)
        pos = torch.from_numpy(a.view(np.uint8).reshape(len(a), width)).to(dev)
    idx = None
    if indices is not None:
        if isinstance(indices, torch.Tensor):
            idx = indices
        else:
            i = np.ascontiguousarray(indices).reshape(-1)
            if i.dtype.kind not in "iu":
                raise TypeError("indices must be integers, not %s" % i.dtype)
            idx = torch.from_numpy(i.astype(np.int64)).to(dev)
    n = len(pos) if idx is None else len(idx)
    enc = torch.empty((n,) + encoding_shape, dtype=torch.float32, device=dev)
    pol = torch.empty((n, engine.A), dtype=torch.float32, device=dev)
    val = torch.empty((n, 1), dtype=torch.float32, device=dev)
    torch.cuda.current_stream(dev).synchronize()                       # the engine's stream reads the inputs
    engine._chk(engine._fn("positions_to_training_device")(
        engine._h, pos.data_ptr() if len(pos) else None, len(pos), None if idx is None else idx.data_ptr(), n,
        enc.data_ptr(), pol.data_ptr(), val.data_ptr()))
    return enc, pol, val


class EngineBase:
    """The entry points Engine and ChessEngine share, each stated once.  What differs between the two is a class attribute
    of each:
      _PREFIX       the entry points' prefix, "spb_" or "spb_chess_";
      _RECORD       the numpy dtype of a trajectory record;
      _STATE        the numpy dtype of a state, as advance returns it;
      _ROOT_WIDTH   the children a root row holds, and _MOVE the numpy type of their moves;
      A             the width of a root_policy row."""

    def __init__(self, **config):
        """Creates the engine from `config`, fields of Config; the others keep spb_default_config's values."""
        L = load_library()
        cfg = Config()
        L.spb_default_config(C.byref(cfg))
        for k, v in config.items():
            setattr(cfg, k, v)
        h = _vp()
        rc = getattr(L, self._PREFIX + "create")(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise EngineError(rc, getattr(L, self._PREFIX + "last_error")(None).decode())
        self._h, self._L = h, L
        self.G, self.device = config["num_games"], config["device"]

    def _fn(self, name):
        """The entry point of this engine's prefix: "search" -> spb_search or spb_chess_search."""
        return getattr(self._L, self._PREFIX + name)

    def close(self):
        if getattr(self, "_h", None):
            self._fn("destroy")(self._h)
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
            raise EngineError(rc, self._fn("last_error")(self._h).decode())

    # ---- weights -----------------------------------------------------------------------------
    def load_weights(self, blob: bytes):
        buf = (C.c_char * len(blob)).from_buffer_copy(blob)
        self._chk(self._fn("load_weights")(self._h, C.cast(buf, _vp), len(blob)))

    def load_weights_device(self, named):
        """spb_load_weights_device: the net from (name, CUDA tensor) pairs on the engine's GPU, named as in a checkpoint
        (the names load_weights accepts); the same image as load_weights of a checkpoint of these tensors."""
        import torch
        # the caller's writes to the tensors finish before the engine reads them; `items` and `names` keep the tensors and
        # the table's names alive until the call has returned, after which the engine no longer reads them
        items = list(named.items()) if hasattr(named, "items") else list(named)
        table, n, names = tensor_table(items, self.device)
        torch.cuda.current_stream(torch.device("cuda", self.device)).synchronize()
        self._chk(self._fn("load_weights_device")(self._h, table, n))

    def broadcast_weights(self, root: int = 0):
        """COLLECTIVE: every rank takes root's weight image (spb_broadcast_weights)."""
        self._chk(self._fn("broadcast_weights")(self._h, root))

    # ---- trees -------------------------------------------------------------------------------
    def search(self, num_searches: int):
        self._chk(self._fn("search")(self._h, num_searches))

    def root_children(self, slot: int):
        """-> (moves, visit_counts, child_ids) of `slot`'s root as lists, child order."""
        mv = np.zeros(self._ROOT_WIDTH, self._MOVE)
        cnt, ids = np.zeros(self._ROOT_WIDTH, np.uint32), np.zeros(self._ROOT_WIDTH, np.uint32)
        n = C.c_uint32()
        self._chk(self._fn("root_children")(self._h, slot, *map(np.ctypeslib.as_ctypes, (mv, cnt, ids)), C.byref(n)))
        k = n.value
        return mv[:k].tolist(), cnt[:k].tolist(), ids[:k].tolist()

    def root_children_all(self, out=None):
        """-> (moves[G,W], visit_counts[G,W] u32, child_ids[G,W] u32, n_children[G] u32), child order; W and the move type
        are _ROOT_WIDTH and _MOVE (9 u8 actions, or 256 u16 chess moves).  `out`: the four arrays of an earlier call (e.g.
        in pinned host memory), written in place."""
        W = self._ROOT_WIDTH
        if out is not None:
            mv, cnt, ids, n = out
            assert mv.shape == (self.G, W) and mv.dtype == self._MOVE and cnt.dtype == np.uint32 and ids.dtype == np.uint32 and n.shape == (self.G,)
            assert all(x.flags.c_contiguous for x in out)
        else:
            mv = np.zeros((self.G, W), self._MOVE)
            cnt = np.zeros((self.G, W), np.uint32)
            ids = np.zeros((self.G, W), np.uint32)
            n = np.zeros(self.G, np.uint32)
        self._chk(self._fn("root_children_all")(self._h, mv.ctypes.data, cnt.ctypes.data, ids.ctypes.data, n.ctypes.data))
        return mv, cnt, ids, n

    def root_policy(self, slot: int) -> np.ndarray:
        p = np.zeros(self.A, np.float32)
        self._chk(self._fn("root_policy")(self._h, slot, p.ctypes.data_as(_f32p)))
        return p

    def advance(self, node_ids, slots=None) -> np.ndarray:
        ids = np.ascontiguousarray(node_ids, dtype=np.uint32)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.uint32)
        out = np.zeros(len(ids), dtype=self._STATE)
        self._chk(self._fn("advance")(self._h, None if sl is None else sl.ctypes.data, ids.ctypes.data, len(ids), out.ctypes.data))
        return out

    def arena_len(self, slot: int) -> int:
        n = C.c_uint32()
        self._chk(self._fn("arena_len")(self._h, slot, C.byref(n)))
        return n.value

    # ---- EXTENSION: Dirichlet noise at the root (DESIGN.md §4.6) ------------------------------
    def set_root_noise(self, alpha: float, epsilon: float, seed: int = 0):
        """P' = (1 - epsilon) P + epsilon eta, eta ~ Dir(alpha), at the root of every search; epsilon = 0 turns it off."""
        self._chk(self._fn("set_root_noise")(self._h, alpha, epsilon, seed))

    def root_noise(self, slot: int) -> np.ndarray:
        """The eta the next search of `slot`'s root uses, one entry per root child (child order)."""
        eta = np.zeros(self._ROOT_WIDTH, np.float32)
        n = C.c_uint32()
        self._chk(self._fn("root_noise")(self._h, slot, eta.ctypes.data_as(_f32p), C.byref(n)))
        return eta[:n.value].copy()

    # ---- trajectories ------------------------------------------------------------------------
    def drain_trajectories(self):
        """-> (positions[_RECORD], game_ids[u64]) ordered by (game id, ply)."""
        return self._records(functools.partial(self._fn("drain_trajectories"), self._h))

    def drain_trajectories_device(self, out=None, ids_out=None):
        """The records of drain_trajectories, ordered on the device -> (CUDA uint8 [n, record bytes], CUDA int64 [n]).
        out / ids_out: caller tensors to write into (e.g. replay[head:]); the [:n] views of them are returned."""
        return self._records_to_device(functools.partial(self._fn("drain_trajectories_device"), self._h), out, ids_out)

    def gather_trajectories(self, learner_rank: int = 0):
        """COLLECTIVE: -> (positions, game_ids) ordered by (game id, ply) on the learner rank, empty elsewhere."""
        return self._records(functools.partial(self._fn("gather_trajectories"), self._h, learner_rank))

    def gather_trajectories_device(self, learner_rank: int = 0, out=None, ids_out=None):
        """COLLECTIVE: gather_trajectories into device memory of the learner rank -> (CUDA uint8 [n, record bytes], CUDA
        int64 [n]), empty elsewhere; out / ids_out as for drain_trajectories_device."""
        return self._records_to_device(functools.partial(self._fn("gather_trajectories_device"), self._h, learner_rank),
                                       out, ids_out)

    def _records(self, call):
        """The host forms of drain / gather: `call(buf, capacity, n_ref, ids)` is the entry point with the engine's
        arguments bound.  Size query, then the records -> the [:n] the second call wrote."""
        n = C.c_size_t()
        self._chk(call(None, 0, C.byref(n), None))
        pos = np.zeros(n.value, dtype=self._RECORD)
        ids = np.zeros(n.value, dtype=np.uint64)
        if n.value:
            self._chk(call(pos.ctypes.data, n.value, C.byref(n), ids.ctypes.data))
        return pos[:n.value], ids[:n.value]

    def _records_to_device(self, call, out, ids_out):
        """The device forms of drain / gather, `call` as for _records: the records into `out` / `ids_out` (allocated when
        None) -> their [:n] views."""
        import torch
        width = self._RECORD.itemsize
        if out is not None:
            _check_cuda_tensor(out, torch.uint8, width, "out")
        if ids_out is not None:
            _check_cuda_tensor(ids_out, torch.int64, None, "ids_out")
        dev = torch.device("cuda", self.device)
        n = C.c_size_t()
        self._chk(call(None, 0, C.byref(n), None))
        k = n.value
        if out is None:
            out = torch.empty((k, width), dtype=torch.uint8, device=dev)
        if ids_out is None:
            ids_out = torch.empty(k, dtype=torch.int64, device=dev)
        if len(out) < k or len(ids_out) < k:
            raise ValueError("out / ids_out hold %d / %d records, %d are ready" % (len(out), len(ids_out), k))
        if k:
            torch.cuda.current_stream(dev).synchronize()                   # the caller's work on out / ids_out comes first
            self._chk(call(out.data_ptr(), len(out), C.byref(n), ids_out.data_ptr()))
        return out[:n.value], ids_out[:n.value]

    # ---- multi-GPU: trajectories to the learner rank --------------------------------------------
    def comm_init(self, comm_id: bytes, rank: int, world_size: int):
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(comm_id)
        self._chk(self._fn("comm_init")(self._h, C.cast(buf, _vp), rank, world_size))

    def comm_destroy(self):
        self._chk(self._fn("comm_destroy")(self._h))

    # ---- counters ----------------------------------------------------------------------------
    def counters(self) -> dict:
        return self._read_counters().as_dict()

    def _read_counters(self) -> Counters:
        c = Counters()
        self._chk(self._fn("get_counters")(self._h, C.byref(c)))
        return c

    def reset_counters(self):
        self._chk(self._fn("reset_counters")(self._h))


class Engine(EngineBase):
    """One engine = `Mcts` + its `Vec<Tree>` on one GPU (ref: mcts.rs:41-44, learner_concurrent.rs:174)."""
    _PREFIX, _RECORD, _STATE, _ROOT_WIDTH, _MOVE = "spb_", POSITION_DTYPE, STATE_DTYPE, MAX_ACTIONS, np.uint8
    A = property(lambda self: NUM_ACTIONS[self.game], doc="The game's actions: the width of a policy row.")

    def __init__(self, game=GAME_C4, num_games=100, evaluator=EVAL_NET, c=2.0, device=0, max_nodes_per_tree=0,
                 flags=0, leaves_per_tree=1, game_id_base=0, game_id_stride=0, trajectory_capacity=0):
        super().__init__(game=game, num_games=num_games, evaluator=evaluator, c=c, device=device,
                         max_nodes_per_tree=max_nodes_per_tree, flags=flags, leaves_per_tree=leaves_per_tree,
                         game_id_base=game_id_base, game_id_stride=game_id_stride, trajectory_capacity=trajectory_capacity)
        self.game = game

    # ---- trees -------------------------------------------------------------------------------
    def reset_games(self, roots=None, slots=None):
        n = self.G if slots is None else len(slots)
        sl = None if slots is None else np.ascontiguousarray(slots, dtype=np.uint32)
        arr = None if roots is None else states_array(roots)
        if arr is not None:
            assert len(arr) == n
        self._chk(self._L.spb_reset_games(self._h, None if sl is None else sl.ctypes.data, n,
                                          None if arr is None else arr.ctypes.data))

    def get_state(self, slot: int, node_id: int) -> State:
        s = State()
        self._chk(self._L.spb_get_state(self._h, slot, node_id, C.byref(s)))
        return s

    def node_stats(self, slot: int, node_id: int) -> dict:
        n, fc, nc = C.c_uint32(), C.c_uint32(), C.c_uint32()
        w, p = C.c_float(), C.c_float()
        self._chk(self._L.spb_node_stats(self._h, slot, node_id, C.byref(n), C.byref(w), C.byref(p), C.byref(fc), C.byref(nc)))
        return dict(visit_count=n.value, value_sum=w.value, prior=p.value, first_child=fc.value, n_children=nc.value)

    # ---- evaluator / game rules --------------------------------------------------------------
    def predict(self, states, want_logits=False):
        arr = states_array(states)
        n = len(arr)
        pol = np.zeros((n, self.A), np.float32)
        val = np.zeros(n, np.float32)
        lg = np.zeros((n, self.A), np.float32) if want_logits else None
        self._chk(self._L.spb_predict(self._h, arr.ctypes.data, n, pol.ctypes.data, val.ctypes.data,
                                      None if lg is None else lg.ctypes.data))
        return (pol, val, lg) if want_logits else (pol, val)

    def game_next_states(self, states, actions):
        arr = states_array(states)
        act = np.ascontiguousarray(actions, dtype=np.uint8)
        out = np.zeros(len(arr), dtype=STATE_DTYPE)
        err = np.zeros(len(arr), np.int32)
        self._chk(self._L.spb_game_next_states(self._h, arr.ctypes.data, act.ctypes.data, len(arr), out.ctypes.data, err.ctypes.data))
        return out, err

    def game_valid_actions(self, states) -> np.ndarray:
        arr = states_array(states)
        m = np.zeros(len(arr), np.uint32)
        self._chk(self._L.spb_game_valid_actions(self._h, arr.ctypes.data, len(arr), m.ctypes.data))
        return m

    def game_encode(self, states) -> np.ndarray:
        arr = states_array(states)
        R, Cc = BOARD[self.game]
        out = np.zeros((len(arr), 3, R, Cc), np.float32)
        self._chk(self._L.spb_game_encode(self._h, arr.ctypes.data, len(arr), out.ctypes.data))
        return out

    # ---- self-play ---------------------------------------------------------------------------
    def selfplay_step(self, rule=MOVE_GREEDY_LAST_MAX, temperature=1.25, seed=0, restart_roots=None) -> int:
        arr = None if restart_roots is None else states_array(restart_roots)
        if arr is not None:
            assert len(arr) == self.G
        fin = C.c_uint32()
        self._chk(self._L.spb_selfplay_step(self._h, rule, temperature, seed, None if arr is None else arr.ctypes.data, C.byref(fin)))
        return fin.value

    # ---- timing ------------------------------------------------------------------------------
    def last_search_timing(self):
        s, ev, n = C.c_float(), C.c_float(), C.c_uint32()
        self._chk(self._L.spb_last_search_timing(self._h, C.byref(s), C.byref(ev), C.byref(n)))
        return s.value, ev.value, n.value

    def time_evaluator(self, iters=20):
        """-> (avg launch ms, positions per launch, FLOPs per position) of the evaluator kernel on the last work list."""
        ms, n, fl = C.c_float(), C.c_uint32(), C.c_double()
        self._chk(self._L.spb_time_evaluator(self._h, iters, C.byref(ms), C.byref(n), C.byref(fl)))
        return ms.value, n.value, fl.value

    def async_stats(self) -> dict:
        """Statistics of the last search through the asynchronous pipeline (see spb_last_async_stats)."""
        v = (C.c_uint64 * 12)()
        self._chk(self._L.spb_last_async_stats(self._h, v, 12))
        names = ("batches", "boards", "claim_wait_ns", "tree_busy_ns", "tree_visits", "tree_warps", "eval_ctas",
                 "claims_found_empty", "ticket_wait_ns", "avail_sum", "ready_backlog_sum", "ready_pops_starved")
        return {k: int(x) for k, x in zip(names, v)}

    def synchronize(self):
        self._chk(self._L.spb_synchronize(self._h))
