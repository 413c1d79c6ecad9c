"""B200-native self-play engine: host-side mirror of the reference's search API over the C ABI.

The product is `libselfplay_b200.so` (CUDA, sm_100a) behind `include/selfplay_b200.h`; this package is
the thin Python host side used by tests and bench.py.  There is no CPU fallback: importing works
anywhere (so the ABI can be inspected), creating an Engine needs a B200.
"""
from .engine import (  # noqa: F401
    EVAL_DET, EVAL_NET, EVAL_UNIFORM, FLAG_EVAL_SIMT, FLAG_LOCKSTEP, FLAG_FIXED_POOL, FLAG_FORCE_SPLIT, FLAG_NO_GRAPH, GAME_C4, GAME_CHESS, GAME_TTT,
    MAX_ACTIONS, MOVE_GREEDY_LAST_MAX, MOVE_TEMPERATURE, NUM_ACTIONS, ONGOING, TIED, WON, Config, Counters,
    Engine, EngineError, Position, check_weights, comm_unique_id, positions_to_training, positions_to_training_device, COMM_ID_BYTES, State, STATE_DTYPE, POSITION_DTYPE, library_path, load_library, build_library,
)
from .mcts import Args, Mcts, Tree  # noqa: F401
from . import chess  # noqa: F401
from .chess import ChessEngine, CHESS_STATE_DTYPE, CHESS_POSITION_DTYPE  # noqa: F401
