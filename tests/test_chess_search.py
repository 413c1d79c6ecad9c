"""MCTS over chess (BASELINE config 5): `Mcts::search` / `Tree::use_subtree` (src/mcts.rs) on chess states.

CPU: the oracle's C++ restatement (oracle/chess_oracle.cc) against a second, independent restatement of the SEARCH
(tests/pyref.py's Tree, written from mcts.rs, driven here with chess states) and against the committed known answers
(tests/golden/chess_kats.json, made by tools/gen_chess_golden.py from the Python restatement).
GPU: the device search (csrc/chess_tree.cuh, chess_engine.cu) against the oracle node for node under the deterministic
evaluators — visit counts, value sums, priors, arena layout — and the network path against torch fp32.
PARITY UNPINNED BY THE REFERENCE (no rustc; the child order comes from the un-vendored chess crate), see DESIGN.md §2.
"""
import json
import os

import numpy as np
import pytest

import selfplay_b200 as S
from oracle import pychess as P
import pyref
from test_chess import export_all, play, random_games

F = np.float32
M64 = (1 << 64) - 1
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "chess_kats.json")
MIDGAME = "r1bq1rk1/pp2bppp/2n1pn2/2pp4/3P1B2/2PBPN2/PP1N1PPP/R2QK2R w KQ - 0 8"
MATE_IN_ONE = "7k/8/5K2/8/8/8/8/6Q1 w - - 0 1"


# ---- second restatement: pyref.Tree over chess states ------------------------------------------------------------

def mix64(x):
    return pyref.splitmix64(x)


def py_det_hash(g):
    s, _ = g.export()
    h = 0
    for x in list(s.piece) + list(s.color) + [s.side | (s.castle << 8) | (s.ep << 16)]:
        h = mix64(h ^ int(x))
    return h


def py_policy_index(side, m):
    f = m & 63
    row = 7 - (f >> 3) if side else (f >> 3)
    return P.channel(side, m) * 64 + row * 8 + (f & 7)


class PyState:
    """`State` of chess.rs for pyref.Tree: the rules come from the oracle's Game, the search does not."""

    def __init__(self, g):
        self.g = g

    def valid_actions(self):
        return self.g.legal_moves()

    def next_state(self, a):
        h = self.g.clone()
        assert h.make_move(a) == 0
        return PyState(h)

    @property
    def status(self):
        return self.g.status()


def py_search(tree, num_searches, evaluator):
    """mcts.rs:214-284 for one tree, chess.rs:168-174 for the terminal value (Won = +1.0)."""
    for _ in range(num_searches):
        nid = 0
        while tree.arena[nid]["children"]:
            nid = tree.select(nid)
        st = tree.arena[nid]["state"]
        status = st.status
        if status == S.WON:
            tree.backprop(nid, F(1))
        elif status == S.TIED:
            tree.backprop(nid, F(0))
        else:
            side = st.g.side()
            moves = st.valid_actions()
            if evaluator == S.EVAL_DET:
                h = py_det_hash(st.g)
                raw = {m: F(1 + (mix64(h ^ (0x100000000 + py_policy_index(side, m))) & 7)) * F(1.0 / 64.0) for m in moves}
                v = F(F((h >> 40) & 0xFF) - F(128)) * F(1.0 / 128.0)
            else:
                raw = {m: F(1) for m in moves}
                v = F(0)
            # mask_invalid_actions (chess.rs:251-271): the masked 4,672-cell array summed in ndarray's order
            cells = [F(0)] * P.POLICY_SIZE
            for m in moves:
                cells[py_policy_index(side, m)] = raw[m]
            total = pyref.ndarray_sum(cells)
            tree.expand(nid, {m: F(raw[m] / total) for m in moves})
            tree.backprop(nid, v)


def py_tree(g):
    return pyref.Tree(PyState(g))


def tree_table_py(tree):
    return [(n["N"], float(n["W"]), float(n["prior"]) if n["prior"] is not None else 0.0, n["children"][0] if n["children"] else 0,
             len(n["children"]), n["action"] if n["action"] is not None else 0xFFFF) for n in tree.arena]


def tree_table_oracle(f, slot):
    out = []
    for i in range(f.arena_len(slot)):
        d = f.node(slot, i)
        out.append((d["visit_count"], d["value_sum"], d["prior"], d["first_child"], d["n_children"], d["move"]))
    return out


def tree_table_device(e, slot):
    out = []
    for i in range(e.arena_len(slot)):
        d = e.node_stats(slot, i)
        out.append((d["visit_count"], d["value_sum"], d["prior"], d["first_child"], d["n_children"], d["move"]))
    return out


# ---- CPU ---------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("evaluator", [S.EVAL_DET, S.EVAL_UNIFORM])
@pytest.mark.parametrize("fen,sims", [(None, 60), (P.KIWIPETE, 40), (MATE_IN_ONE, 80)])
def test_oracle_search_equals_python_restatement_node_for_node(evaluator, fen, sims):
    g = P.Game(fen)
    f = P.Forest(1)
    f.reset(0, g)
    f.search(sims, evaluator)
    t = py_tree(g)
    py_search(t, sims, evaluator)
    assert tree_table_oracle(f, 0) == tree_table_py(t)


def test_oracle_use_subtree_equals_python_restatement():
    g = P.Game(MIDGAME)
    f = P.Forest(1)
    f.reset(0, g)
    t = py_tree(g)
    for _ in range(3):
        f.search(50, S.EVAL_DET)
        py_search(t, 50, S.EVAL_DET)
        _, cnt, ids = f.root_children(0)
        best = max(range(len(cnt)), key=lambda i: (cnt[i], i))          # last maximum, main.rs:108-112
        f.use_subtree(0, ids[best])
        t.use_subtree(ids[best])
        assert tree_table_oracle(f, 0) == tree_table_py(t)


def test_golden_known_answers():
    kats = json.load(open(GOLDEN))
    assert len(kats["cases"]) >= 6
    for case in kats["cases"]:
        g = play(case["moves"], case["fen"])
        f = P.Forest(1)
        f.reset(0, g)
        f.search(case["sims"], case["evaluator"])
        mvs, cnt, ids = f.root_children(0)
        assert mvs == case["root_moves"] and cnt == case["root_counts"], case["name"]
        assert f.arena_len(0) == case["arena_len"] and f.node(0, 0)["value_sum"] == case["root_value_sum"], case["name"]
        assert P.det_hash(g) == int(case["det_hash"], 16), case["name"]


def test_checkmate_counts_plus_one_for_the_mated_side():
    # chess.rs:172 gives Won = +1.0 to the node whose side to move is checkmated — the opposite sign of the other games —
    # so the search is steered AWAY from mating moves; reproduced, not repaired
    g = P.Game(MATE_IN_ONE)
    f = P.Forest(1)
    f.reset(0, g)
    f.search(300, S.EVAL_UNIFORM)
    mvs, cnt, ids = f.root_children(0)
    mates = []
    for m, c, i in zip(mvs, cnt, ids):
        h = g.clone()
        h.make_move(m)
        if h.status() == S.WON:
            mates.append((m, c, i))
    assert mates
    for m, c, i in mates:
        assert c >= 1 and f.node(0, i)["value_sum"] == float(c) and f.node(0, i)["n_children"] == 0
    assert max(c for _, c, _ in mates) < max(cnt)


# ---- GPU ---------------------------------------------------------------------------------------------------------

def oracle_forest(games, sims, evaluator, c=2.0):
    f = P.Forest(len(games), c)
    for i, g in enumerate(games):
        f.reset(i, g)
    f.search(sims, evaluator)
    return f


def search_roots():
    games = [P.Game(), P.Game(P.KIWIPETE), P.Game(MIDGAME), P.Game(MATE_IN_ONE), play("g1f3 g8f6 f3g1 f6g8 g1f3 g8f6"),
             P.Game("8/P6k/8/8/8/8/6Kp/8 w - - 0 1"), P.Game("4k3/8/8/8/8/8/8/R3K3 w - - 96 70")]
    games += random_games(2, seed=23, max_plies=60)[-2:]
    return [g for g in games if g.status() == S.ONGOING]


@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [S.EVAL_DET, S.EVAL_UNIFORM])
def test_device_search_matches_oracle_node_for_node(evaluator):
    games = search_roots()
    st, hist = export_all(games)
    f = oracle_forest(games, 200, evaluator)
    with S.ChessEngine(num_games=len(games), evaluator=evaluator) as e:
        e.reset_games(st, hist)
        e.search(120)
        e.search(80)                                              # accumulating searches on the same trees
        mv_all, cnt_all, ids_all, n_all = e.root_children_all()
        for i in range(len(games)):
            want = f.root_children(i)
            assert e.root_children(i) == want, i
            k = int(n_all[i])
            assert (mv_all[i, :k].tolist(), cnt_all[i, :k].tolist(), ids_all[i, :k].tolist()) == want, i
            assert e.arena_len(i) == f.arena_len(i), i
        for i in (0, 3, 4, len(games) - 1):
            assert tree_table_device(e, i) == tree_table_oracle(f, i), i
        c = e.counters()
        want = f.counters()
        for k in want:
            assert c[k] == want[k], k
        # the Policy half of the result (mcts.rs:315-328)
        mvs, cnt, _ = f.root_children(0)
        pol = e.root_policy(0)
        assert pol.sum() == pytest.approx(1.0, abs=1e-6)
        for m, cc in zip(mvs, cnt):
            assert pol[py_policy_index(games[0].side(), m)] == np.float32(cc) / np.float32(sum(cnt))


@pytest.mark.gpu
def test_device_use_subtree_and_greedy_play_match_oracle():
    games = [P.Game(), P.Game(MIDGAME), play("g1f3 g8f6 f3g1 f6g8")]
    st, hist = export_all(games)
    f = P.Forest(len(games))
    for i, g in enumerate(games):
        f.reset(i, g)
    with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e:
        e.reset_games(st, hist)
        for ply in range(6):
            f.search(100, S.EVAL_DET)
            e.search(100)
            picks = []
            for i in range(len(games)):
                mvs, cnt, ids = f.root_children(i)
                assert e.root_children(i) == (mvs, cnt, ids), (ply, i)
                best = max(range(len(cnt)), key=lambda k: (cnt[k], k))
                picks.append(ids[best])
            new_states = e.advance(picks)
            for i in range(len(games)):
                f.use_subtree(i, picks[i])
                root = f.state(i, 0)
                ws, wh = root.export()
                assert new_states[i].tobytes() == bytes(ws), (ply, i)
                assert e.get_state(i, 0).tobytes() == bytes(ws)
                assert tree_table_device(e, i) == tree_table_oracle(f, i), (ply, i)
                # a node deep in the tree: its state equals the oracle's (moves replayed from the root)
                deep = f.arena_len(i) - 1
                got = e.get_state(i, deep)
                want, _ = f.state(i, deep).export()
                want.hist_len = ws.hist_len
                assert got.tobytes() == bytes(want), (ply, i)
        # a call with one bad entry, or a slot listed twice, moves no tree
        def snapshot():
            return [(e.arena_len(i), tree_table_device(e, i), e.get_state(i, 0).tobytes()) for i in range(len(games))]
        before = snapshot()
        child = e.root_children(1)[2][0]
        for call in (lambda: e.advance([0, 1, 1]),              # node 0 is not a child of the root
                     lambda: e.advance([child, child], slots=[1, 1]),
                     lambda: e.reset_games(st[:2], hist[:2], slots=[2, 2])):
            with pytest.raises(S.EngineError) as ei:
                call()
            assert ei.value.code == -1
            assert snapshot() == before


@pytest.mark.gpu
def test_device_search_finds_repetition_draws_inside_the_tree():
    # two occurrences of the start list are already in the history: the third is found INSIDE the search (path + history)
    g = play("g1f3 g8f6 f3g1 f6g8 g1f3 g8f6 f3g1")
    assert g.status() == S.ONGOING
    st, hist = export_all([g])
    f = oracle_forest([g], 400, S.EVAL_UNIFORM)
    assert f.counters()["terminal_leaves"] > 0
    with S.ChessEngine(num_games=1, evaluator=S.EVAL_UNIFORM) as e:
        e.reset_games(st, hist)
        e.search(400)
        assert tree_table_device(e, 0) == tree_table_oracle(f, 0)
        assert e.counters()["terminal_leaves"] == f.counters()["terminal_leaves"]


@pytest.mark.gpu
def test_device_pool_overflow_is_reported():
    with S.ChessEngine(num_games=2, evaluator=S.EVAL_UNIFORM, max_nodes_per_tree=512) as e:
        e.reset_games()
        with pytest.raises(S.EngineError) as ei:
            e.search(400)
        assert ei.value.code == -3


@pytest.mark.gpu
def test_device_many_trees_agree_with_each_other():
    # 512 trees at the same root must all be identical (one warp per tree, no cross-talk)
    g = P.Game(MIDGAME)
    st, hist = export_all([g] * 512)
    f = oracle_forest([g], 200, S.EVAL_DET)
    with S.ChessEngine(num_games=512, evaluator=S.EVAL_DET) as e:
        e.reset_games(st, hist)
        e.search(200)
        mv_all, cnt_all, ids_all, n_all = e.root_children_all()
        want = f.root_children(0)
        k = len(want[0])
        assert (n_all == k).all()
        assert (cnt_all[:, :k] == np.array(want[1], np.uint32)).all() and (mv_all[:, :k] == np.array(want[0], np.uint16)).all()


# ---- GPU: the 10 x 256 network (src/model/chess.rs) ----------------------------------------------------------------
RTOL = 1e-2          # north_star: "within 1e-2 relative on policy logits and value"


@pytest.fixture(scope="module")
def chess_net():
    from oracle import torch_net
    return torch_net.make_chess_net(seed=0)


def net_positions():
    games = random_games(3, seed=31, max_plies=90)
    games = [g for g in games if g.status() == S.ONGOING][::7][:20]
    games += [P.Game(), P.Game(P.KIWIPETE), P.Game(MIDGAME), play("g1f3 g8f6 f3g1 f6g8 g1f3"), P.Game("4k3/8/8/8/8/8/8/R3K3 w - - 96 70")]
    return games


def test_chess_checkpoint_parser_accepts_both_naming_schemes(chess_net):
    from oracle import torch_net
    for blob in (torch_net.chess_to_safetensors_tch(chess_net), torch_net.chess_to_safetensors_explicit(chess_net),
                 torch_net.chess_to_safetensors_tch(chess_net, shuffle_seed=3)):
        rc, msg = S.chess.check_weights(blob)
        assert rc == 0, msg
    rc, msg = S.chess.check_weights(torch_net.to_safetensors_tch(torch_net.make_net(S.GAME_C4, seed=1)))
    assert rc == -5 and "census" in msg
    assert S.chess.check_weights(b"\x00" * 16)[0] == -5


@pytest.mark.gpu
def test_chess_network_matches_torch_fp32(chess_net):
    from oracle import torch_net
    games = net_positions()
    st, hist = export_all(games)
    enc = np.stack([g.encode() for g in games])
    probs_ref, v_ref, logit_ref = torch_net.chess_forward(chess_net, enc)
    with S.ChessEngine(num_games=64, evaluator=S.EVAL_NET) as e:
        e.load_weights(torch_net.chess_to_safetensors_tch(chess_net))
        pol, v, lg = e.predict(st, hist, want_logits=True)
        scale = float(np.abs(logit_ref).max())
        err = float(np.abs(lg - logit_ref).max())
        assert np.allclose(lg, logit_ref, rtol=RTOL, atol=RTOL * scale), (err, scale)
        assert np.allclose(v, v_ref, rtol=RTOL, atol=RTOL), float(np.abs(v - v_ref).max())
        # Model::predict's tail: softmax, mask to the legal moves, renormalise (chess.rs:251-271)
        for i, g in enumerate(games):
            idx = [py_policy_index(g.side(), m) for m in g.legal_moves()]
            want = np.zeros(P.POLICY_SIZE, np.float32)
            want[idx] = probs_ref[i, idx] / probs_ref[i, idx].sum()
            assert np.allclose(pol[i], want, rtol=5 * RTOL, atol=1e-4), i
            assert abs(float(pol[i].sum()) - 1.0) < 1e-4 and np.count_nonzero(pol[i]) == len(idx)
        # a batch that is not a multiple of the tile: the same positions one by one give the same numbers
        pol1, v1, lg1 = e.predict(st[3:4], hist[3:4], want_logits=True)
        assert np.array_equal(lg1[0], lg[3]) and v1[0] == v[3]


@pytest.mark.gpu
def test_chess_network_search_matches_oracle_with_torch_evaluator(chess_net):
    from oracle import torch_net
    games = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE), play("e2e4 e7e5 g1f3")]
    st, hist = export_all(games)
    sims = 48

    def net_fn(enc):
        p, v, _ = torch_net.chess_forward(chess_net, enc)
        return p, v

    f = P.Forest(len(games))
    for i, g in enumerate(games):
        f.reset(i, g)
    f.search(sims, S.EVAL_NET, net_fn)
    with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_NET) as e:
        e.load_weights(torch_net.chess_to_safetensors_explicit(chess_net))
        e.reset_games(st, hist)
        e.search(sims)
        c = e.counters()
        assert c["simulations"] == sims * len(games) and c["evaluations"] + c["terminal_leaves"] == c["simulations"]
        for i in range(len(games)):
            mvs, cnt, _ = f.root_children(i)
            gm, gc, _ = e.root_children(i)
            assert gm == mvs and sum(gc) == sum(cnt) == sims - 1
            # evaluators differ by ~1e-3 (bf16 operands), so counts are compared as distributions
            tv = 0.5 * sum(abs(a - b) for a, b in zip(gc, cnt)) / (sims - 1)
            assert tv < 0.15, (i, tv, gc, cnt)
            # root priors: softmax masked to the legal moves
            fc = f.node(i, 0)["first_child"]
            pri_ref = np.array([f.node(i, fc + k)["prior"] for k in range(len(mvs))])
            pri = np.array([e.node_stats(i, fc + k)["prior"] for k in range(len(mvs))])
            assert np.allclose(pri, pri_ref, rtol=5 * RTOL, atol=1e-4), i


@pytest.mark.gpu
def test_chess_network_pipeline_two_half_loops_equal_one_loop(chess_net):
    """From 256 trees on, the network pipeline runs the two halves of the trees as two lock-step loops on two streams (tree
    kernels of one half under the convolutions of the other).  Trees never interact, so every tree must come out exactly as
    from one loop over all trees (SPB_FLAG_LOCKSTEP); 301 trees: an odd split, a ragged last tile."""
    from oracle import torch_net
    from selfplay_b200.synth import synthetic_chess_roots_device
    blob = torch_net.chess_to_safetensors_explicit(chess_net)
    out = []
    for flags in (0, S.FLAG_LOCKSTEP):
        with S.ChessEngine(num_games=301, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(blob)
            st, hist = synthetic_chess_roots_device(e, 301)
            e.reset_games(st, hist)
            e.search(20)
            mv, cnt, ids, n = e.root_children_all()
            out.append((mv.copy(), cnt.copy(), ids.copy(), n.copy(), e.counters()))
    for a, b in zip(out[0][:4], out[1][:4]):
        assert (a == b).all()
    for k in ("simulations", "evaluations", "terminal_leaves"):
        assert out[0][4][k] == out[1][4][k], k
    assert (out[0][1].sum(axis=1)[out[0][3] > 0] == 19).all()   # 19 visits below every non-terminal root


# ---- GPU: the kernels of the network pipeline under the deterministic evaluators, and the full size of configs[4] --------

@pytest.mark.gpu
@pytest.mark.parametrize("evaluator", [S.EVAL_DET, S.EVAL_UNIFORM])
def test_device_lockstep_pipeline_matches_oracle_node_for_node(evaluator):
    """SPB_FLAG_FORCE_SPLIT: select -> evaluate -> expand + backup as three kernels per simulation step (the pipeline the
    network uses) instead of the fused kernel; results must not change by a bit."""
    games = search_roots()
    st, hist = export_all(games)
    f = oracle_forest(games, 150, evaluator)
    with S.ChessEngine(num_games=len(games), evaluator=evaluator, flags=S.FLAG_FORCE_SPLIT) as e:
        e.reset_games(st, hist)
        e.search(150)
        for i in range(len(games)):
            assert e.root_children(i) == f.root_children(i), i
        for i in (0, 2, 4, len(games) - 1):
            assert tree_table_device(e, i) == tree_table_oracle(f, i), i
        c, want = e.counters(), f.counters()
        for k in want:
            assert c[k] == want[k], k


def synthetic_chess_root(g, max_ply=41):
    """The oracle-side twin of selfplay_b200.synth.synthetic_chess_roots_device (bench.py --game chess)."""
    from helpers import splitmix64
    while True:
        r = splitmix64(0xC4E55000 + g)
        plies = r % max_ply
        game = P.Game()
        ok = True
        for _ in range(plies):
            if game.status() != 0:
                ok = False
                break
            lm = game.legal_moves()
            r = splitmix64(r)
            game.make_move(lm[r % len(lm)])
        if ok and game.status() == 0:
            return game
        g += 1 << 32


@pytest.mark.gpu
def test_full_size_chess_4096_games_x_200_sims():
    """configs[4] at full size under DetEval: the bench's synthetic roots come out of the device rules exactly as the oracle
    builds them; 4,096 trees x 200 simulations; 12 trees spread over the batch replayed by the oracle node for node; every
    tree conserves its budget; fused and lock-step pipelines agree on every root (SHA-256)."""
    import hashlib
    from selfplay_b200.synth import synthetic_chess_roots_device
    G, sims = 4096, 200
    digests = []
    for flags in (0, S.FLAG_FORCE_SPLIT):
        with S.ChessEngine(num_games=G, evaluator=S.EVAL_DET, flags=flags, max_nodes_per_tree=14336) as e:
            st, hist = synthetic_chess_roots_device(e, G)
            sample = list(range(0, G, 372))
            if flags == 0:
                for i in sample:
                    ws, wh = synthetic_chess_root(i).export()
                    assert st[i].tobytes() == bytes(ws) and (hist[i] == wh).all(), i
            e.reset_games(st, hist)
            e.search(sims)
            mv, cnt, ids, n = e.root_children_all()
            assert (cnt.sum(1) == sims - 1).all() and (n > 0).all()
            c = e.counters()
            assert c["simulations"] == G * sims and c["evaluations"] + c["terminal_leaves"] == G * sims
            digests.append(hashlib.sha256(mv.tobytes() + cnt.tobytes() + ids.tobytes() + n.tobytes()).hexdigest())
            if flags == 0:
                games = [synthetic_chess_root(i) for i in sample]
                f = oracle_forest(games, sims, S.EVAL_DET)
                for k, i in enumerate(sample):
                    assert e.root_children(i) == f.root_children(k), i
                    assert e.arena_len(i) == f.arena_len(k), i
    assert digests[0] == digests[1]
