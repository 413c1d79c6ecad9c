"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/selfplay_b200.h declares, and its host-only logic behaves (no compute calls without a GPU)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import selfplay_b200 as S
from oracle import torch_net

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "selfplay_b200.h")).read()


def declared_symbols():
    return sorted(set(re.findall(r"\b(spb_[a-z_0-9]+)\s*\(", HEADER)))


def test_library_exports_every_declared_symbol():
    L = S.load_library()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(L, n), "missing export: " + n
    assert set(names) == set(S.engine.ABI), set(names) ^ set(S.engine.ABI)
    assert L.spb_abi_version() == S.engine.ABI_VERSION == int(re.search(r"#define SPB_ABI_VERSION (\d+)", HEADER).group(1))


def test_struct_layouts_match_header():
    assert C.sizeof(S.State) == 24 and C.sizeof(S.Position) == 56
    assert C.sizeof(S.Config) == 16 * 4 and C.sizeof(S.Counters) == 12 * 8
    cfg = S.Config()
    assert S.load_library().spb_default_config(C.byref(cfg)) == 0
    # defaults mirror Args::default (mcts.rs:46-59)
    assert (cfg.game, cfg.num_games, cfg.c, cfg.leaves_per_tree, cfg.evaluator) == (S.GAME_C4, 100, 2.0, 1, S.EVAL_NET)


def test_create_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(S.EngineError) as ei:
        S.Engine(num_games=4, evaluator=S.EVAL_DET)
    assert ei.value.code == -2 and "no CPU fallback" in str(ei.value)


def test_create_rejects_bad_config():
    L = S.load_library()
    cfg = S.Config()
    L.spb_default_config(C.byref(cfg))
    h = C.c_void_p()
    for field, val in [("abi_version", 99), ("game", 7), ("num_games", 0), ("leaves_per_tree", 0), ("evaluator", 9),
                       ("c", float("nan")), ("max_nodes_per_tree", 8), ("num_games", 2**22 + 1), ("leaves_per_tree", 17)]:
        bad = S.Config.from_buffer_copy(cfg)
        setattr(bad, field, val)
        assert L.spb_create(C.byref(bad), C.byref(h)) == -1, field
        assert L.spb_last_error(None)
    assert L.spb_create(None, C.byref(h)) == -1
    assert L.spb_destroy(None) == -1 and L.spb_search(None, 1) == -1


def chess_config():
    cfg = S.Config()
    S.load_library().spb_default_config(C.byref(cfg))
    cfg.game, cfg.num_games, cfg.evaluator = S.GAME_CHESS, 4, S.EVAL_DET
    return cfg


def test_chess_create_rejects_bad_config():
    L = S.load_library()
    h = C.c_void_p()
    for field, val in [("abi_version", 99), ("game", S.GAME_C4), ("num_games", 0), ("num_games", 2**20 + 1),
                       ("leaves_per_tree", 2), ("evaluator", 9), ("c", float("nan")), ("max_nodes_per_tree", 100)]:
        bad = chess_config()
        setattr(bad, field, val)
        assert L.spb_chess_create(C.byref(bad), C.byref(h)) == -1, field
        assert L.spb_chess_last_error(None), field
    assert L.spb_chess_create(None, C.byref(h)) == -1


def test_chess_create_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = S.load_library()
    h = C.c_void_p()
    assert L.spb_chess_create(C.byref(chess_config()), C.byref(h)) == -2
    assert b"no CPU fallback" in L.spb_chess_last_error(None)


def test_every_entry_point_rejects_a_null_engine():
    # every function of the header whose first parameter is an engine handle, called with NULL, NULL pointers and zeros
    L = S.load_library()
    names = re.findall(r"\b(spb_[a-z_0-9]+)\s*\(\s*(?:const\s+)?(?:spb_engine|spb_chess_engine)\s*\*", HEADER)
    names = sorted(set(n for n in names if not n.endswith("last_error")))
    assert any(n.startswith("spb_chess_") for n in names) and len(names) > 50
    for name in names:
        f = getattr(L, name)
        assert f.argtypes is not None, name
        args = [None if t in (C.c_void_p, C.c_char_p) or issubclass(t, C._Pointer) else 0 for t in f.argtypes]
        assert f(*args) == -1, name


@pytest.mark.parametrize("game", [S.GAME_TTT, S.GAME_C4])
def test_check_weights_accepts_both_naming_schemes(game):
    net = torch_net.make_net(game, seed=3)
    for blob in (torch_net.to_safetensors_tch(net), torch_net.to_safetensors_explicit(net),
                 torch_net.to_safetensors_tch(net, shuffle_seed=5),
                 torch_net.to_safetensors_tch(net, bn_order=("running_mean", "running_var", "weight", "bias"))):
        rc, msg = S.check_weights(game, blob)
        assert rc == 0, msg


def test_check_weights_rejects_garbage():
    net = torch_net.make_net(S.GAME_C4, seed=3)
    blob = torch_net.to_safetensors_tch(net)
    assert S.check_weights(S.GAME_C4, b"\x00" * 4)[0] == -5
    assert S.check_weights(S.GAME_C4, blob[:1000])[0] == -5
    rc, msg = S.check_weights(S.GAME_TTT, blob)          # Connect4 checkpoint into the tic-tac-toe net
    assert rc == -5 and "shape" in msg
    import struct
    hdr_len = struct.unpack("<Q", blob[:8])[0]
    rc, msg = S.check_weights(S.GAME_C4, blob[:8] + b"{" + b"x" * (hdr_len - 1) + blob[8 + hdr_len:])
    assert rc == -5


def test_tch_names_look_like_a_varstore():
    names = [k for k in __import__("json").loads(torch_net.to_safetensors_tch(torch_net.make_net(1))[8:].split(b"}}")[0] + b"}}")]
    assert "bias" in names and "weight" in names and "running_mean" in names
    assert any(re.fullmatch(r"weight__\d+", n) for n in names)
    assert len(names) == 70     # SURVEY.md §2 row 8: 70 VarStore tensors


def test_flag_and_code_constants_agree_across_header_python_and_rust():
    """The header is the source of truth; the ctypes mirror and the Rust -sys crate must not drift from it."""
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "selfplay_b200.h")).read()
    defs = {m.group(1): int(m.group(2).rstrip("u"), 0) for m in re.finditer(r"#define\s+(SPB_[A-Z0-9_]+)\s+(-?\d+u?)\b", header)}
    py = {"SPB_FLAG_NO_GRAPH": S.FLAG_NO_GRAPH, "SPB_FLAG_EVAL_SIMT": S.FLAG_EVAL_SIMT, "SPB_FLAG_FORCE_SPLIT": S.FLAG_FORCE_SPLIT,
          "SPB_FLAG_FIXED_POOL": S.FLAG_FIXED_POOL, "SPB_FLAG_LOCKSTEP": S.FLAG_LOCKSTEP,
          "SPB_GAME_CONNECT4": S.GAME_C4, "SPB_GAME_TICTACTOE": S.GAME_TTT,
          "SPB_EVAL_NET": S.EVAL_NET, "SPB_EVAL_DET": S.EVAL_DET, "SPB_EVAL_UNIFORM": S.EVAL_UNIFORM}
    for name, value in py.items():
        assert defs[name] == value, name
    flags = [v for k, v in defs.items() if k.startswith("SPB_FLAG_")]
    assert len(set(flags)) == len(flags) and all(v & (v - 1) == 0 for v in flags)      # distinct single bits
    rust = open(os.path.join(root, "rust", "selfplay-b200-sys", "src", "lib.rs")).read()
    n_consts = 0
    for m in re.finditer(r"pub const (SPB_[A-Z0-9_]+): (?:[iu]32|u8|usize) = (-?\d+);", rust):
        assert defs[m.group(1)] == int(m.group(2)), m.group(1)
        n_consts += 1
    assert n_consts >= 30


def test_rust_sys_crate_mirrors_every_function_and_struct_of_the_header():
    """rust/selfplay-b200-sys cannot be compiled here (no rustc), so its text is checked against the header: the same set of
    functions with the same number of parameters, and the same struct fields in the same order with matching types."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rust = open(os.path.join(root, "rust", "selfplay-b200-sys", "src", "lib.rs")).read()
    # functions
    c_fns = {}
    for m in re.finditer(r"\b(?:int32_t|uint16_t|const char\*)\s+(spb_[a-z_0-9]+)\s*\(([^;]*?)\)\s*;", HEADER, re.S):
        args = re.sub(r"/\*.*?\*/", "", m.group(2), flags=re.S).strip()
        c_fns[m.group(1)] = 0 if args in ("", "void") else args.count(",") + 1
    r_fns = {}
    for m in re.finditer(r"pub fn (spb_[a-z_0-9]+)\(([^)]*)\)", rust):
        args = m.group(2).strip()
        r_fns[m.group(1)] = 0 if not args else args.count(",") + 1
    assert set(c_fns) == set(declared_symbols())
    assert c_fns == r_fns, {k: (c_fns.get(k), r_fns.get(k)) for k in set(c_fns) | set(r_fns) if c_fns.get(k) != r_fns.get(k)}
    # structs
    ctype = {"uint64_t": "u64", "uint32_t": "u32", "uint16_t": "u16", "uint8_t": "u8", "int8_t": "i8", "int32_t": "i32", "float": "f32"}
    size = {"u64": 8, "u32": 4, "u16": 2, "u8": 1, "i8": 1, "i32": 4, "f32": 4}
    defs = {m.group(1): int(m.group(2).rstrip("u"), 0) for m in re.finditer(r"#define\s+(SPB_[A-Z0-9_]+)\s+(-?\d+u?)\b", HEADER)}
    want_size = {"spb_state": 24, "spb_config": 64, "spb_counters": 96, "spb_position": 56, "spb_chess_state": 80}
    for name in want_size:
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), HEADER, re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        c_fields = []
        for m in re.finditer(r"(\w+)\s+(\w+)(?:\[(\w+)\])?;", body):
            n = m.group(3)
            c_fields.append((m.group(2), ctype[m.group(1)], None if n is None else (int(n) if n.isdigit() else defs[n])))
        rbody = re.search(r"pub struct %s \{(.*?)\n\}" % name, rust, re.S).group(1)
        r_fields = []
        for m in re.finditer(r"pub (\w+): (?:\[(\w+); (\w+)\]|(\w+)),", rbody):
            if m.group(2):
                n = m.group(3)
                r_fields.append((m.group(1), m.group(2), int(n) if n.isdigit() else defs[n]))
            else:
                r_fields.append((m.group(1), m.group(4), None))
        assert c_fields == r_fields, (name, c_fields, r_fields)
        # natural alignment, no padding inside: the sum of the field sizes is the struct size both sides assume
        assert sum(size[t] * (n or 1) for _, t, n in c_fields) == want_size[name], name
    assert re.search(r"#\[repr\(C\)\]\s*(?:#\[derive[^\]]*\]\s*)?pub struct spb_chess_state", rust)


def test_positions_to_training_matches_the_oracle_encodings():
    """spb_positions_to_training (host only): the learner's tensors (learner_concurrent.rs:126-146) from compact records —
    encodings equal the oracle's get_encoding of the recorded state, policies are counts / sum in f32, values the outcome."""
    from helpers import random_states
    from oracle import pyoracle as O
    rng = np.random.default_rng(5)
    for game in (S.GAME_C4, S.GAME_TTT):
        A = S.NUM_ACTIONS[game]
        states = random_states(game, 200, seed=3, include_terminal=False)
        pos = np.zeros(len(states), dtype=S.POSITION_DTYPE)
        for i, s in enumerate(states):
            pos[i]["stones"] = (s.stones[0], s.stones[1])
            pos[i]["current_player"] = s.current_player
            pos[i]["ply"] = s.num_actions_played
            legal = O.valid_actions(game, s)
            counts = np.zeros(9, np.uint32)
            counts[legal] = rng.integers(0, 800, len(legal))
            counts[legal[0]] += 1                                     # at least one visit
            pos[i]["visit_counts"] = counts
            pos[i]["outcome"] = int(rng.integers(-1, 2))
        enc, pol, val = S.positions_to_training(game, pos)
        assert enc.shape == (len(states), 3) + S.engine.BOARD[game] and pol.shape == (len(states), A) and val.shape == (len(states), 1)
        for i, s in enumerate(states):
            assert np.array_equal(enc[i], O.encode(game, s))
            c = pos[i]["visit_counts"][:A].astype(np.float32)
            assert np.array_equal(pol[i], c / np.float32(c.sum(dtype=np.float32)))
            assert val[i, 0] == float(pos[i]["outcome"])
    assert S.load_library().spb_positions_to_training(7, None, 0, None, None, None) == -1
