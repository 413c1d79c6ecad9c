"""Chess self-play on the device: spb_chess_selfplay_step, spb_chess_drain_trajectories, spb_chess_positions_to_training.

CPU: the spb_chess_position record agrees between the header, ctypes and the Rust -sys crate; the training tensors of records
built from oracle positions equal the oracle's encodings and counts / their f32 sum.
GPU: the device ply against the reference loop (learner_concurrent.rs:169-242) driven over the oracle's search, record for
record; against the host loop (root_children_all + last-max pick + advance) on the same engine; temperature sampling,
parking on a full buffer, the history cap, restarts and the network pipelines.
"""
import os
import re

import numpy as np
import pytest

import selfplay_b200 as S
from oracle import pychess as P
from test_chess import export_all, play
from test_chess_search import MIDGAME, py_policy_index, tree_table_device

CH = S.chess
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "selfplay_b200.h")).read()
FORCED_MATE = "4rkr1/4p1p1/8/8/8/8/6PP/4Rr1K w - - 0 1"          # the only legal move, e1f1, mates
FIFTY_99 = "4k3/8/8/8/8/8/8/R3K3 w - - 99 70"                       # no capture or pawn move: any move ends the game
NEAR_THREEFOLD = "g1f3 g8f6 f3g1 f6g8 g1f3 g8f6 f3g1"


# ---- CPU ---------------------------------------------------------------------------------------------------------

def test_chess_position_layout_agrees_across_header_ctypes_and_rust():
    ctype = {"uint32_t": "<u4", "uint16_t": "<u2", "uint8_t": "u1", "int8_t": "i1", "spb_chess_state": CH.CHESS_STATE_DTYPE}
    defs = {m.group(1): int(m.group(2).rstrip("u"), 0) for m in re.finditer(r"#define\s+(SPB_[A-Z0-9_]+)\s+(-?\d+u?)\b", HEADER)}
    body = re.search(r"typedef struct spb_chess_position \{(.*?)\} spb_chess_position;", HEADER, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    c_fields = []
    for m in re.finditer(r"(\w+)\s+(\w+)(?:\[(\w+)\])?;", body):
        n = m.group(3)
        c_fields.append((m.group(2), m.group(1), None if n is None else (int(n) if n.isdigit() else defs[n])))
    # ctypes mirror: same names, order, element types and counts
    py = [(name, CH.CHESS_POSITION_DTYPE.fields[name][0]) for name in CH.CHESS_POSITION_DTYPE.names]
    assert [f[0] for f in c_fields] == [p[0] for p in py]
    for (name, ct, n), (_, dt) in zip(c_fields, py):
        want = np.dtype(ctype[ct]) if n is None else np.dtype((ctype[ct], (n,)))
        assert dt == want, name
    # natural alignment, no padding: offsets are the running sum of the sizes
    off = 0
    for name in CH.CHESS_POSITION_DTYPE.names:
        assert CH.CHESS_POSITION_DTYPE.fields[name][1] == off, name
        off += CH.CHESS_POSITION_DTYPE.fields[name][0].itemsize
    assert off == CH.CHESS_POSITION_DTYPE.itemsize == 1624
    # Rust -sys crate: the same fields in the same order with the same types
    rust = open(os.path.join(ROOT, "rust", "selfplay-b200-sys", "src", "lib.rs")).read()
    assert re.search(r"#\[repr\(C\)\]\s*(?:#\[derive[^\]]*\]\s*)?pub struct spb_chess_position", rust)
    rbody = re.search(r"pub struct spb_chess_position \{(.*?)\n\}", rust, re.S).group(1)
    rtype = {"uint32_t": "u32", "uint16_t": "u16", "uint8_t": "u8", "int8_t": "i8", "spb_chess_state": "spb_chess_state"}
    r_fields = []
    for m in re.finditer(r"pub (\w+): (?:\[(\w+); (\w+)\]|(\w+)),", rbody):
        if m.group(2):
            n = m.group(3)
            r_fields.append((m.group(1), m.group(2), int(n) if n.isdigit() else defs[n]))
        else:
            r_fields.append((m.group(1), m.group(4), None))
    assert r_fields == [(name, rtype[ct], n) for name, ct, n in c_fields]
    assert defs["SPB_CHESS_POS_ADJUDICATED"] == CH.POS_ADJUDICATED
    assert re.search(r"pub const SPB_CHESS_POS_ADJUDICATED: u8 = %d;" % CH.POS_ADJUDICATED, rust)


def test_chess_selfplay_symbols_are_exported():
    L = S.load_library()
    for name in ("spb_chess_selfplay_step", "spb_chess_drain_trajectories", "spb_chess_positions_to_training"):
        assert hasattr(L, name) and name in S.engine.ABI, name


def record_of(g, rng, ply=0, outcome=0):
    """A record of the oracle position g with random visit counts over its legal moves (child order)."""
    s, _ = g.export()
    moves = g.legal_moves()
    r = np.zeros(1, CH.CHESS_POSITION_DTYPE)[0]
    r["state"] = np.frombuffer(bytes(s), CH.CHESS_STATE_DTYPE)[0]
    r["moves"][:] = CH.MOVE_NONE
    r["moves"][:len(moves)] = moves
    cnt = rng.integers(0, 500, len(moves)).astype(np.uint32)
    cnt[0] += 1
    r["visit_counts"][:len(moves)] = cnt
    r["n_moves"], r["ply"], r["repetitions"], r["outcome"] = len(moves), ply, g.repetitions(), outcome
    return r


def test_positions_to_training_matches_the_oracle():
    from test_chess import random_games
    rng = np.random.default_rng(11)
    games = [g for g in random_games(6, seed=5, max_plies=80) if g.status() == S.ONGOING][::3]
    games += [play("g1f3 g8f6 f3g1 f6g8"), play(NEAR_THREEFOLD), P.Game(FIFTY_99), P.Game(FORCED_MATE), P.Game(MIDGAME)]
    assert any(g.repetitions() == 3 - 1 for g in games)              # a history-driven repetition count in plane 16
    recs = np.array([record_of(g, rng, i, int(rng.integers(-1, 2))) for i, g in enumerate(games)], CH.CHESS_POSITION_DTYPE)
    enc, pol, val = CH.positions_to_training(recs)
    assert enc.shape == (len(games), 19, 8, 8) and pol.shape == (len(games), 4672) and val.shape == (len(games), 1)
    for i, g in enumerate(games):
        assert np.array_equal(enc[i], g.encode()), i
        n = int(recs[i]["n_moves"])
        cnt = recs[i]["visit_counts"][:n]
        want = np.zeros(4672, np.float32)
        total = np.float32(0)
        for c in cnt:
            total = np.float32(total + np.float32(c))
        for m, c in zip(recs[i]["moves"][:n], cnt):
            want[py_policy_index(g.side(), int(m))] = np.float32(c) / total
        assert np.array_equal(pol[i], want), i
        assert val[i, 0] == float(recs[i]["outcome"])
    # each output may be NULL
    L = S.load_library()
    assert L.spb_chess_positions_to_training(recs.ctypes.data, len(recs), None, None, None) == 0
    # malformed records and arguments
    for field, value in (("n_moves", 0), ("n_moves", 257)):
        bad = recs.copy()
        bad[0][field] = value
        assert L.spb_chess_positions_to_training(bad.ctypes.data, len(bad), None, None, None) == -1, (field, value)
    bad = recs.copy()
    bad[1]["state"]["side"] = 2
    assert L.spb_chess_positions_to_training(bad.ctypes.data, len(bad), None, None, None) == -1
    bad = recs.copy()
    bad[2]["moves"][0] = 7 | (0 << 6) | (3 << 12)                      # h1-a1 as a rook promotion: off the policy
    assert L.spb_chess_positions_to_training(bad.ctypes.data, len(bad), None, None, None) == -1
    assert L.spb_chess_positions_to_training(None, 3, None, None, None) == -1
    with pytest.raises(S.EngineError):
        CH.positions_to_training(bad)


# ---- GPU ---------------------------------------------------------------------------------------------------------

def oracle_selfplay(games, sims, evaluator, steps):
    """The reference loop (learner_concurrent.rs:179-238, greedy pick of main.rs:108-112) over the oracle's search: per step
    search, last-max pick, record the root, terminal child -> outcomes (chess.rs:172 value, sign by side), else use_subtree.
    -> (records of finished games as dicts ordered by (game id, ply), games finished per step, how each game ended)."""
    f = P.Forest(len(games))
    for i, g in enumerate(games):
        f.reset(i, g)
    live, hist, out, per_step, ends = [True] * len(games), [[] for _ in games], [], [], {}
    for _ in range(steps):
        f.search(sims, evaluator)
        fin = 0
        for i in range(len(games)):
            if not live[i]:
                continue
            mvs, cnt, ids = f.root_children(i)
            best = max(range(len(cnt)), key=lambda k: (cnt[k], k))
            root = f.state(i, 0)
            s, _ = root.export()
            hist[i].append(dict(state=bytes(s), moves=mvs, counts=cnt, repetitions=root.repetitions(), ply=len(hist[i]), side=root.side()))
            child = f.state(i, ids[best])
            if child.status() != S.ONGOING:
                v, ts = int(child.value()), child.side()
                for r in hist[i]:
                    out.append(dict(r, outcome=v if r["side"] == ts else -v, game_id=i))
                ends[i] = "mate" if child.status() == S.WON else ("repetition" if child.repetitions() >= 3 else "fifty")
                live[i] = False
                fin += 1
            else:
                f.use_subtree(i, ids[best])
        per_step.append(fin)
    out.sort(key=lambda r: (r["game_id"], r["ply"]))
    return out, per_step, ends


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, S.FLAG_FORCE_SPLIT])
@pytest.mark.parametrize("evaluator", [S.EVAL_DET, S.EVAL_UNIFORM])
def test_greedy_selfplay_matches_the_oracle_reference_loop(evaluator, flags):
    games = [P.Game(), P.Game(MIDGAME), play(NEAR_THREEFOLD), P.Game(FIFTY_99), P.Game(FORCED_MATE)]
    sims, steps = 48, 8
    want, want_fin, ends = oracle_selfplay(games, sims, evaluator, steps)
    assert {"mate", "repetition", "fifty"} <= set(ends.values()), ends
    st, hist = export_all(games)
    with CH.ChessEngine(num_games=len(games), evaluator=evaluator, flags=flags) as e:
        e.reset_games(st, hist)
        got_fin = []
        for _ in range(steps):
            e.search(sims)
            got_fin.append(e.selfplay_step(S.MOVE_GREEDY_LAST_MAX))
        pos, ids = e.drain_trajectories()
    assert got_fin == want_fin
    assert len(pos) == len(want)
    for r, i, w in zip(pos, ids, want):
        n = int(r["n_moves"])
        assert int(i) == w["game_id"] and int(r["ply"]) == w["ply"], (i, w["game_id"])
        assert r["state"].tobytes() == w["state"]
        assert r["moves"][:n].tolist() == w["moves"] and r["visit_counts"][:n].tolist() == w["counts"]
        assert (r["moves"][n:] == CH.MOVE_NONE).all() and (r["visit_counts"][n:] == 0).all()
        assert int(r["repetitions"]) == w["repetitions"] and int(r["outcome"]) == w["outcome"] and int(r["flags"]) == 0


def host_loop_step(e):
    """One ply of the caller's own loop: root_children_all, last-max pick on the host, advance."""
    mv, cnt, ids, n = e.root_children_all()
    picks = []
    for i in range(e.G):
        k = int(n[i])
        c = cnt[i, :k].tolist()
        picks.append(ids[i, max(range(k), key=lambda j: (c[j], j))])
    e.advance(picks)


@pytest.mark.gpu
def test_device_step_equals_the_host_loop_on_the_same_engine():
    games = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE)]
    st, hist = export_all(games)
    tables = []
    with CH.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e:
        for device_step in (True, False):
            e.reset_games(st, hist)
            run = []
            for _ in range(5):
                e.search(40)
                if device_step:
                    assert e.selfplay_step(S.MOVE_GREEDY_LAST_MAX) == 0
                else:
                    host_loop_step(e)
                run.append([tree_table_device(e, i) for i in range(len(games))] + [e.get_state(i, 0).tobytes() for i in range(len(games))])
            tables.append(run)
    assert tables[0] == tables[1]


def capped_roots(games, hist_len, seed=3):
    """The oracle positions with their real history followed by distinct random hashes up to hist_len plies: the history cap
    ends every game after SPB_CHESS_MAX_HISTORY - hist_len + 1 records."""
    st, hist = export_all(games)
    rng = np.random.default_rng(seed)
    for i in range(len(games)):
        h0 = int(st[i]["hist_len"])
        hist[i, h0:hist_len] = rng.integers(1 << 40, 1 << 62, hist_len - h0, dtype=np.uint64)
        st[i]["hist_len"] = hist_len
    return st, hist


@pytest.mark.gpu
def test_policy_target_equals_root_policy_read_before_the_step():
    games = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE), play("e2e4 e7e5 g1f3")]
    st, hist = capped_roots(games, 509)
    seen = {}
    with CH.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e:
        e.reset_games(st, hist)
        for ply in range(4):
            e.search(50)
            for i in range(len(games)):
                seen[(i, ply)] = e.root_policy(i)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
        pos, ids = e.drain_trajectories()
    assert len(pos) == 4 * len(games)
    _, pol, _ = CH.positions_to_training(pos)
    for r, i, p in zip(pos, ids, pol):
        assert np.array_equal(p, seen[(int(i), int(r["ply"]))]), (i, r["ply"])


@pytest.mark.gpu
def test_history_cap_ends_the_game_as_an_adjudicated_tie():
    st, hist = capped_roots([P.Game()], 510)
    assert len(set(hist[0, :510].tolist())) == 510
    with CH.ChessEngine(num_games=1, evaluator=S.EVAL_DET) as e:
        e.reset_games(st, hist)
        fin = []
        for _ in range(3):
            e.search(30)
            fin.append(e.selfplay_step(S.MOVE_GREEDY_LAST_MAX))
        pos, ids = e.drain_trajectories()
        assert e.drain_trajectories()[0].size == 0                     # drained once
    assert fin == [0, 0, 1]
    assert pos["ply"].tolist() == [0, 1, 2] and pos["state"]["hist_len"].tolist() == [510, 511, 512]
    assert (pos["flags"] == CH.POS_ADJUDICATED).all() and (pos["outcome"] == 0).all() and (ids == 0).all()


@pytest.mark.gpu
def test_temperature_sampling_follows_counts_to_the_power_t():
    from scipy import stats
    G, t = 1024, 1.0
    st, hist = export_all([P.Game()] * G)
    with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET, trajectory_capacity=4096) as e:
        e.reset_games(st, hist)
        e.search(120)
        mv, cnt, _ = e.root_children(0)
        _, cnt_all, _, n_all = e.root_children_all()
        assert (cnt_all[:, :len(cnt)] == np.array(cnt, np.uint32)).all() and (n_all == len(cnt)).all()
        e.selfplay_step(S.MOVE_TEMPERATURE, temperature=t, seed=1234)
        chosen = [e.node_stats(i, 0)["move"] for i in range(G)]
    w = np.array(cnt, np.float64) ** t
    expected = G * w / w.sum()
    observed = np.array([chosen.count(m) for m in mv], np.float64)
    assert observed.sum() == G
    big = expected >= 5                                                # pool the children expected fewer than 5 times
    obs = np.append(observed[big], observed[~big].sum())
    exp = np.append(expected[big], expected[~big].sum())
    if exp[-1] == 0:
        obs, exp = obs[:-1], exp[:-1]
    assert stats.chisquare(obs, exp).pvalue > 1e-3, (obs, exp)


@pytest.mark.gpu
def test_temperature_trajectories_depend_on_the_seed_only():
    games = [P.Game(), P.Game(MIDGAME)] * 32
    st, hist = capped_roots(games, 510)
    runs = []
    for seed in (7, 7, 8):
        with CH.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e:
            e.reset_games(st, hist)
            for _ in range(3):
                e.search(40)
                e.selfplay_step(S.MOVE_TEMPERATURE, temperature=1.0, seed=seed)
            pos, ids = e.drain_trajectories()
            assert len(pos) == 3 * len(games)
            runs.append(pos.tobytes() + ids.tobytes())
    assert runs[0] == runs[1] and runs[0] != runs[2]


@pytest.mark.gpu
def test_full_trajectory_buffer_parks_games_and_loses_nothing():
    G = 256                                                            # 256 games x 3 records > 512 records of buffer
    games = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE), play("e2e4 e7e5 g1f3")] * (G // 4)
    st, hist = capped_roots(games, 510)

    def run(capacity):
        parts, raised = [], 0
        with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET, trajectory_capacity=capacity) as e:
            e.reset_games(st, hist)
            for _ in range(3):
                e.search(30)
                try:
                    e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
                except S.EngineError as err:
                    assert err.code == -6
                    raised += 1
            parts.append(e.drain_trajectories())
            assert e.selfplay_step(S.MOVE_GREEDY_LAST_MAX) == (G - len(parts[0][0]) // 3)   # the parked games, emitted now
            parts.append(e.drain_trajectories())
        pos = np.concatenate([p for p, _ in parts])
        ids = np.concatenate([i for _, i in parts])
        order = np.lexsort((pos["ply"], ids))
        return pos[order], ids[order], raised, len(parts[0][0])

    small = run(512)
    big = run(0)
    assert small[2] == 1 and small[3] <= 512 and big[2] == 0 and big[3] == 3 * G
    assert small[0].tobytes() == big[0].tobytes() and (small[1] == big[1]).all()


@pytest.mark.gpu
def test_restart_roots_start_the_next_game_with_the_next_game_id():
    games = [P.Game(), P.Game(MIDGAME), play(NEAR_THREEFOLD), P.Game(P.KIWIPETE)]
    st, hist = capped_roots(games, 510)
    with CH.ChessEngine(num_games=4, evaluator=S.EVAL_DET, game_id_base=100, game_id_stride=10) as e:
        e.reset_games(st, hist)
        for _ in range(6):
            e.search(30)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist)
        pos, ids = e.drain_trajectories()
    first = {int(i): None for i in ids}
    for r, i in zip(pos, ids):
        if r["ply"] == 0:
            first[int(i)] = r["state"].tobytes()
    # every slot finished at least two games; the next game of slot s has id 100 + s + 10k and starts from the restart root
    for s in range(4):
        mine = sorted(i for i in first if (i - 100) % 10 == s)
        assert mine[:2] == [100 + s, 110 + s], (s, mine)
        for i in mine:
            assert first[i] == st[s].tobytes(), (s, i)
    assert (np.diff(ids.astype(np.int64)) >= 0).all()


@pytest.mark.gpu
def test_network_two_half_loops_and_lockstep_give_identical_trajectories():
    from selfplay_b200.synth import synthetic_chess_roots_device
    from selfplay_b200.weights_init import random_chess_checkpoint
    G = 256
    blob = random_chess_checkpoint(seed=2)
    out = []
    for flags in (0, S.FLAG_LOCKSTEP):
        with CH.ChessEngine(num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(blob)
            st, hist = synthetic_chess_roots_device(e, G)
            rng = np.random.default_rng(9)                              # history to 500 plies: every game ends within 13 plies
            for i in range(G):
                h0 = int(st[i]["hist_len"])
                hist[i, h0:500] = rng.integers(1 << 40, 1 << 62, 500 - h0, dtype=np.uint64)
                st[i]["hist_len"] = 500
            e.reset_games(st, hist)
            fin = []
            for _ in range(20):
                e.search(50)
                fin.append(e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist))
            pos, ids = e.drain_trajectories()
            out.append((pos.tobytes(), ids.tobytes(), fin))
    assert sum(out[0][2]) >= G and len(out[0][0]) >= G * 1624
    assert out[0] == out[1]
