"""Dirichlet noise at the search root (DESIGN.md §4.6): P' = (1 - eps) P + eps eta at the root's children only, eta ~ Dir(alpha)
drawn on the device from (seed, game id, root ply, number of root children).

CPU: the Python restatement of the mixing (tests/noise_ref.py, on pyref's tree) against the oracle and by hand.  GPU: argument checks, the default path unchanged bit for bit in every pipeline,
the properties and the distribution of eta, exact parity with the oracle given the device's eta, the pipelines agreeing with
each other, and self-play with noise."""
import hashlib

import numpy as np
import pytest

import noise_ref as NR
import pyref
import selfplay_b200 as S
from helpers import synthetic_roots
from oracle import pychess as P
from oracle import pyoracle as O

ERR_ARG, ERR_STATE = -1, -6          # SPB_ERR_ARG, SPB_ERR_STATE


def _legal_count(game, st):
    """Legal moves of a position (oracle State or a row of the engine's state array)."""
    if not isinstance(st, O.State):
        st = _to_oracle_state(st)
    return len(O.valid_actions(game, st)) if st.status == O.ONGOING else 0


def _to_oracle_state(row):
    s = O.State()
    s.stones[0], s.stones[1] = int(row["stones"][0]), int(row["stones"][1])
    s.current_player, s.num_actions_played, s.status = int(row["current_player"]), int(row["num_actions_played"]), int(row["status"])
    return s


def _oracle_tree(f, slot):
    return [f.node_stats(slot, i) for i in range(f.arena_len(slot))]


def _device_tree(e, slot):
    return [e.node_stats(slot, i) for i in range(e.arena_len(slot))]


def _assert_same_tree(e, t, slot):
    """Device tree `slot` == the restatement's tree t: root children, visit counts, value sums, priors, arena layout."""
    assert e.arena_len(slot) == len(t.arena), slot
    assert e.root_children(slot) == NR.root_children(t), slot
    assert _device_tree(e, slot) == NR.table(t), slot


# ---- CPU: the restatement --------------------------------------------------------------------------------------------

@pytest.mark.parametrize("game", [O.GAME_C4, O.GAME_TTT])
def test_restated_roots_are_the_oracles(game):
    mp = 11 if game == O.GAME_C4 else 4
    for g in range(40):
        s, p = NR.synthetic_root(game, g, mp)
        assert s.key() == synthetic_roots(game, 1, start=g, max_ply=mp)[0].key()
        x, o = p.stones()
        assert (x, o, p.player, p.n, p.status) == s.key()


@pytest.mark.parametrize("game", [O.GAME_C4, O.GAME_TTT])
@pytest.mark.parametrize("k", [1, 4, 16])
def test_restatement_at_epsilon_zero_is_the_oracle_search(game, k):
    """With eps = 0 and any eta the restatement is the plain search: node for node equal to the oracle (search and, for K > 1,
    search_vl)."""
    G, sims = 4, 120
    pairs = [NR.synthetic_root(game, 7 + g, 9 if game == O.GAME_C4 else 3) for g in range(G)]
    f = O.Forest(game, G, leaves_per_tree=k)
    f.reset([s for s, _ in pairs])
    f.search(sims)
    rng = np.random.default_rng(0)
    trees = []
    for s, p in pairs:
        t = NR.NoisyTree(p)
        t.set_root_noise(rng.dirichlet([0.3] * _legal_count(game, s)).astype(np.float32), 0.0)
        trees.append(t)
    if k == 1:
        pyref.search(trees, sims, pyref.det_eval)
    else:
        NR.search_vl(trees, sims, k, pyref.det_eval)
    for g, t in enumerate(trees):
        assert NR.table(t) == _oracle_tree(f, g), g


def test_restatement_tictactoe_one_hot_eta_known_answer():
    """Uniform evaluator, eps = 1, eta = e_j: after the first simulation expands the root, every child but j scores exactly 0
    (q = 0 unvisited, u = c * 0 * ...), child j scores q + u > 0, so all the other 49 simulations go below child j."""
    for j in (0, 4, 8):
        t = NR.NoisyTree(pyref.TTT())
        eta = np.zeros(9, np.float32)
        eta[j] = 1.0
        t.set_root_noise(eta, 1.0)
        pyref.search([t], 50, pyref.uniform_eval)
        assert t.root_counts() == [49 if i == j else 0 for i in range(9)], (j, t.root_counts())
        assert t.arena[1 + j]["prior"] == np.float32(1.0 / 9.0)            # the stored prior is the evaluator's
    t = NR.NoisyTree(pyref.TTT())
    pyref.search([t], 50, pyref.uniform_eval)
    assert max(t.root_counts()) < 49                                        # without noise the visits spread


@pytest.mark.parametrize("k", [1, 4])
def test_restatement_use_subtree_drops_the_noise(k):
    rng = np.random.default_rng(1)

    def run(ts, n):
        if k == 1:
            pyref.search(ts, n, pyref.det_eval)
        else:
            NR.search_vl(ts, n, k, pyref.det_eval)

    for g in range(4):
        s, p = NR.synthetic_root(O.GAME_C4, 3 + g, 8)
        a, b = NR.NoisyTree(p), NR.NoisyTree(p)
        eta = rng.dirichlet([0.5] * _legal_count(O.GAME_C4, s)).astype(np.float32)
        for t in (a, b):
            t.set_root_noise(eta, 0.25)
        run([a, b], 60)
        cnt = a.root_counts()
        pick = a.arena[0]["children"][int(np.argmax(cnt))]
        a.use_subtree(pick)
        b.use_subtree(pick)
        b.set_root_noise([], 0.0)                                           # explicit "off" equals what use_subtree left
        run([a, b], 60)
        assert NR.table(a) == NR.table(b)
        assert a.eta is None


# ---- GPU -------------------------------------------------------------------------------------------------------------

def _sha_trees(e, slots):
    h = hashlib.sha256()
    for s in slots:
        for d in _device_tree(e, s):
            h.update(repr(sorted(d.items())).encode())
    return h.hexdigest()


def _c4_net_blob(game):
    from oracle import torch_net
    return torch_net.to_safetensors_tch(torch_net.make_net(1 if game == S.GAME_C4 else 0, seed=0))


@pytest.mark.gpu
def test_setters_reject_bad_arguments_and_root_noise_needs_noise_on():
    with S.Engine(game=S.GAME_C4, num_games=4, evaluator=S.EVAL_DET) as e, S.ChessEngine(num_games=2, evaluator=S.EVAL_DET) as c:
        e.reset_games()
        c.reset_games()
        for eng in (e, c):
            for alpha, eps in [(0.0, 0.25), (-1.0, 0.25), (float("nan"), 0.25), (float("inf"), 0.25), (0.3, -0.1), (0.3, 1.5),
                               (0.3, float("nan"))]:
                with pytest.raises(S.EngineError) as ex:
                    eng.set_root_noise(alpha, eps, 1)
                assert ex.value.code == ERR_ARG, (alpha, eps)
            with pytest.raises(S.EngineError) as ex:
                eng.root_noise(0)
            assert ex.value.code == ERR_STATE
            eng.set_root_noise(0.3, 1.0, 1)
            assert len(eng.root_noise(0)) > 0
            eng.set_root_noise(0.3, 0.0, 1)
            with pytest.raises(S.EngineError) as ex:
                eng.root_noise(0)
            assert ex.value.code == ERR_STATE


C4_PIPELINES = {"fused": dict(flags=0), "async": dict(flags=S.FLAG_FORCE_SPLIT), "lockstep": dict(flags=S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP),
                "k16": dict(flags=S.FLAG_FORCE_SPLIT, leaves_per_tree=16)}


@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
@pytest.mark.parametrize("pipe", list(C4_PIPELINES) + ["net-async", "net-lockstep"])
def test_epsilon_zero_leaves_every_pipeline_bit_identical(game, pipe):
    G = 24
    roots = synthetic_roots(game, G, start=40, max_ply=15 if game == S.GAME_C4 else 4)
    if pipe.startswith("net"):
        kw = dict(evaluator=S.EVAL_NET, flags=S.FLAG_LOCKSTEP if pipe == "net-lockstep" else 0)
    else:
        kw = dict(evaluator=S.EVAL_DET, **C4_PIPELINES[pipe])
    shas = []
    for mode in ("never", "zero", "on-then-off"):
        with S.Engine(game=game, num_games=G, **kw) as e:
            if pipe.startswith("net"):
                e.load_weights(_c4_net_blob(game))
            e.reset_games(roots)
            if mode == "on-then-off":
                e.set_root_noise(0.3, 0.25, 5)
                e.search(8)                                    # captures a step graph with the noise on
                e.reset_games(roots)
            if mode != "never":
                e.set_root_noise(0.3, 0.0, 5)
            e.search(48)
            e.search(16)
            shas.append(_sha_trees(e, range(G)))
    assert shas[0] == shas[1] == shas[2]


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, S.FLAG_FORCE_SPLIT], ids=["fused", "lockstep"])
def test_chess_epsilon_zero_leaves_the_search_bit_identical(flags):
    from test_chess_search import search_roots, tree_table_device
    from test_chess import export_all
    games = search_roots()
    st, hist = export_all(games)
    tables = []
    for mode in ("never", "zero"):
        with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET, flags=flags) as e:
            if mode == "zero":
                e.set_root_noise(0.3, 0.0, 9)
            e.reset_games(st, hist)
            e.search(120)
            tables.append([tree_table_device(e, i) for i in range(len(games))])
    assert tables[0] == tables[1]


@pytest.mark.gpu
def test_chess_epsilon_zero_two_half_network_pipeline_unchanged():
    from oracle import torch_net
    from selfplay_b200.synth import synthetic_chess_roots_device
    blob = torch_net.chess_to_safetensors_explicit(torch_net.make_chess_net(seed=0))
    out = []
    for mode in ("never", "zero"):
        with S.ChessEngine(num_games=260, evaluator=S.EVAL_NET) as e:
            e.load_weights(blob)
            if mode == "zero":
                e.set_root_noise(0.3, 0.0, 9)
            st, hist = synthetic_chess_roots_device(e, 260)
            e.reset_games(st, hist)
            e.search(8)
            out.append([a.copy() for a in e.root_children_all()])
    for a, b in zip(*out):
        assert (a == b).all()


@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
def test_eta_properties(game):
    G = 32
    roots = synthetic_roots(game, G, start=11, max_ply=12 if game == S.GAME_C4 else 4)
    roots = [r for r in roots if r.status == O.ONGOING][:16]
    G = len(roots)

    def etas(seed, base=0, searched=0):
        with S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET, game_id_base=base) as e:
            e.reset_games(roots)
            e.set_root_noise(0.3, 0.25, seed)
            out = [e.root_noise(s) for s in range(G)]         # unexpanded roots
            if searched:
                e.search(searched)
                again = [e.root_noise(s) for s in range(G)]   # the same root: the same eta
                assert all((a == b).all() for a, b in zip(out, again))
            return out

    a = etas(7, searched=30)
    for s, r in enumerate(roots):
        assert len(a[s]) == _legal_count(game, r)
        assert (a[s] >= 0).all() and abs(float(a[s].astype(np.float64).sum()) - 1.0) <= 1e-5
    b = etas(7)
    assert all((x == y).all() for x, y in zip(a, b))                   # across engines
    c = etas(8)
    d = etas(7, base=1000)
    assert sum((x == y).all() for x, y in zip(a, c)) == 0               # the seed changes every eta
    assert sum((x == y).all() for x, y in zip(a, d)) == 0               # so does the game id
    # the ply: advancing to a child gives a fresh eta; the stored priors equal those of a run without noise
    with S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET) as e, S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET) as q:
        for eng in (e, q):
            eng.reset_games(roots)
        e.set_root_noise(0.3, 0.25, 7)
        e.search(40)
        q.search(40)
        for s in range(G):
            nc = e.node_stats(s, 0)["n_children"]
            fc = e.node_stats(s, 0)["first_child"]
            assert [e.node_stats(s, fc + i)["prior"] for i in range(nc)] == [q.node_stats(s, q.node_stats(s, 0)["first_child"] + i)["prior"] for i in range(nc)]
        ids = [e.root_children(s)[2][0] for s in range(G)]
        new = e.advance(ids)
        for s in range(G):
            eta = e.root_noise(s)
            assert len(eta) == _legal_count(game, new[s])
            if len(eta) == len(a[s]) and len(eta) > 1:
                assert not (eta == a[s]).all()
        # a restarted slot: a fresh root, the eta of (game id, ply 0)
        e.reset_games(roots[:1], slots=[0])
        assert (e.root_noise(0) == a[0]).all()


@pytest.mark.gpu
def test_chess_eta_properties():
    from test_chess import export_all
    from test_chess_search import search_roots
    games = search_roots()
    st, hist = export_all(games)
    with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e, S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as q:
        for eng in (e, q):
            eng.reset_games(st, hist)
        e.set_root_noise(0.3, 0.25, 3)
        first = [e.root_noise(i) for i in range(len(games))]
        for i, g in enumerate(games):
            assert len(first[i]) == len(g.legal_moves())
            assert (first[i] >= 0).all() and abs(float(first[i].astype(np.float64).sum()) - 1.0) <= 1e-5
        e.search(60)
        q.search(60)
        for i in range(len(games)):
            assert (e.root_noise(i) == first[i]).all()
            nc, fc = e.node_stats(i, 0)["n_children"], e.node_stats(i, 0)["first_child"]
            qfc = q.node_stats(i, 0)["first_child"]
            assert [e.node_stats(i, fc + k)["prior"] for k in range(nc)] == [q.node_stats(i, qfc + k)["prior"] for k in range(nc)]
    with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET, game_id_base=50) as e:
        e.reset_games(st, hist)
        e.set_root_noise(0.3, 0.25, 3)
        assert all(not (e.root_noise(i) == first[i]).all() for i in range(len(games)))


# ---- GPU: the distribution -------------------------------------------------------------------------------------------

def _ks_and_corr(etas, n, alpha):
    """p-value of eta[:, 0] against Beta(alpha, (n - 1) alpha), and the correlation of eta[:, 0] and eta[:, 1].  Below the
    smallest normal f32 t, eta is stored as 0 or a denormal (for alpha = 0.03 that is ~4 % of the mass): the share at or below
    t is checked against F(t) by a binomial test, the rest by a KS test against the Beta conditioned on X > t."""
    from scipy import stats
    x = etas[:, 0]
    t = float(np.finfo(np.float32).tiny)
    d = stats.beta(alpha, (n - 1) * alpha)
    ft = float(d.cdf(t))
    p_atom = stats.binomtest(int((x <= t).sum()), len(x), ft).pvalue if ft > 0 else 1.0
    p_ks = stats.kstest(x[x > t].astype(np.float64), lambda v: (d.cdf(v) - ft) / (1.0 - ft)).pvalue
    r = np.corrcoef(etas[:, 0], etas[:, 1])[0, 1]
    return min(p_atom, p_ks), r


@pytest.mark.gpu
@pytest.mark.parametrize("alpha", [0.03, 0.3, 1.0, 10.0])
def test_eta_marginals_are_beta_and_pairs_anticorrelated(alpha):
    G = 4096
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        e.reset_games()
        e.set_root_noise(alpha, 0.25, 11)
        etas = np.stack([e.root_noise(s) for s in range(G)])
    assert etas.shape == (G, 7)
    for i in (0, 3, 6):
        p, _ = _ks_and_corr(etas[:, [i, (i + 1) % 7]], 7, alpha)
        assert p > 1e-3, (alpha, i, p)
    _, r = _ks_and_corr(etas, 7, alpha)
    assert abs(r - (-1.0 / 6.0)) < 0.06, r
    with S.ChessEngine(num_games=G, evaluator=S.EVAL_DET, max_nodes_per_tree=512) as c:
        c.reset_games()
        c.set_root_noise(alpha, 0.25, 11)
        etas = np.stack([c.root_noise(s) for s in range(G)])
    assert etas.shape == (G, 20)
    for i in (0, 19):
        p, _ = _ks_and_corr(etas[:, [i, (i + 1) % 20]], 20, alpha)
        assert p > 1e-3, (alpha, i, p)
    _, r = _ks_and_corr(etas, 20, alpha)
    assert abs(r - (-1.0 / 19.0)) < 0.06, r


# ---- GPU: exact parity with the restatement given the device's eta ---------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
@pytest.mark.parametrize("pipe", ["fused", "async", "lockstep", "k4", "k16"])
def test_noisy_search_matches_the_restatement_over_a_greedy_game(game, pipe):
    G, sims, eps = 8, 64, 0.25
    k = {"k4": 4, "k16": 16}.get(pipe, 1)
    flags = {"fused": 0, "async": S.FLAG_FORCE_SPLIT, "lockstep": S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP}.get(pipe, S.FLAG_FORCE_SPLIT)
    pairs = [NR.synthetic_root(game, 200 + g, 10 if game == S.GAME_C4 else 2) for g in range(G)]
    trees = [NR.NoisyTree(p) for _, p in pairs]
    with S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET, flags=flags, leaves_per_tree=k) as e:
        e.reset_games([s for s, _ in pairs])
        e.set_root_noise(0.3, eps, 21)
        live = list(range(G))
        for ply in range(12 if game == S.GAME_C4 else 9):
            for g in live:
                trees[g].set_root_noise(e.root_noise(g), eps)    # redrawn for every new root
            e.search(sims)
            if k == 1:
                pyref.search(trees, sims, pyref.det_eval)
            else:
                NR.search_vl(trees, sims, k, pyref.det_eval)
            for g in range(G):
                _assert_same_tree(e, trees[g], g)
            picks = {}
            for g in live:
                ch, cnt = trees[g].arena[0]["children"], trees[g].root_counts()
                if cnt:
                    picks[g] = ch[max(range(len(cnt)), key=lambda i: (cnt[i], i))]
            live = [g for g in picks if trees[g].arena[picks[g]]["state"].status == 0]
            if not live:
                break
            e.advance([picks[g] for g in live], slots=live)
            for g in live:
                trees[g].use_subtree(picks[g])


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, S.FLAG_FORCE_SPLIT], ids=["fused", "lockstep"])
def test_chess_noisy_search_matches_the_restatement_with_use_subtree(flags):
    from test_chess import export_all, play
    from test_chess_search import MIDGAME, PyState, py_search, tree_table_device, tree_table_py
    games = [P.Game(), P.Game(MIDGAME), play("g1f3 g8f6 f3g1 f6g8")]
    st, hist = export_all(games)
    trees = [NR.NoisyTree(PyState(g)) for g in games]
    eps = 0.25
    with S.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET, flags=flags) as e:
        e.reset_games(st, hist)
        e.set_root_noise(0.3, eps, 4)
        for ply in range(4):
            for i, t in enumerate(trees):
                t.set_root_noise(e.root_noise(i), eps)
                py_search(t, 50, S.EVAL_DET)
            e.search(30)
            e.search(20)                                        # accumulating searches of one root: the same eta
            picks = []
            for i, t in enumerate(trees):
                assert tree_table_device(e, i) == tree_table_py(t), (ply, i)
                ch, cnt = t.arena[0]["children"], t.root_counts()
                picks.append(ch[max(range(len(cnt)), key=lambda k: (cnt[k], k))])
            e.advance(picks)
            for i, t in enumerate(trees):
                t.use_subtree(picks[i])


# ---- GPU: pipelines agree with the noise on ----------------------------------------------------------------------------

@pytest.mark.gpu
def test_noisy_network_async_equals_lockstep():
    G = 4096
    roots = synthetic_roots(S.GAME_C4, G, start=0, max_ply=21)
    out = []
    for flags in (0, S.FLAG_LOCKSTEP):
        with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(_c4_net_blob(S.GAME_C4))
            e.reset_games(roots)
            e.set_root_noise(0.3, 0.25, 99)
            e.search(64)
            h = hashlib.sha256()
            for a in e.root_children_all():
                h.update(np.ascontiguousarray(a).tobytes())
            out.append(h.hexdigest())
    assert out[0] == out[1]


@pytest.mark.gpu
def test_noisy_chess_two_half_equals_one_loop():
    from oracle import torch_net
    from selfplay_b200.synth import synthetic_chess_roots_device
    blob = torch_net.chess_to_safetensors_explicit(torch_net.make_chess_net(seed=0))
    out = []
    for flags in (0, S.FLAG_LOCKSTEP):
        with S.ChessEngine(num_games=301, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(blob)
            st, hist = synthetic_chess_roots_device(e, 301)
            e.reset_games(st, hist)
            e.set_root_noise(0.3, 0.25, 99)
            e.search(12)
            out.append([a.copy() for a in e.root_children_all()])
    for a, b in zip(*out):
        assert (a == b).all()


# ---- GPU: self-play with noise -----------------------------------------------------------------------------------------

def _play(G, noise_seed, eps, temp_seed=0, rule=S.MOVE_GREEDY_LAST_MAX, sims=32):
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        e.reset_games()
        e.set_root_noise(0.3, eps, noise_seed)
        for _ in range(42):
            e.search(sims)
            e.selfplay_step(rule=rule, temperature=1.0, seed=temp_seed)
        pos, ids = e.drain_trajectories()
        return pos, ids


@pytest.mark.gpu
def test_selfplay_with_noise_is_reproducible_and_depends_on_the_seeds():
    G = 16
    a = _play(G, 1, 0.25, temp_seed=5, rule=S.MOVE_TEMPERATURE)
    b = _play(G, 1, 0.25, temp_seed=5, rule=S.MOVE_TEMPERATURE)
    assert len(a[0]) > 0 and a[0].tobytes() == b[0].tobytes() and (a[1] == b[1]).all()
    g1, g2 = _play(G, 1, 0.25), _play(G, 2, 0.25)
    assert g1[0].tobytes() != g2[0].tobytes()                    # greedy games from one start differ across noise seeds
    games = {bytes(g1[0][g1[1] == i].tobytes()) for i in np.unique(g1[1])}
    assert len(games) > 1                                        # ... and across the game ids of one seed
    z1, z2 = _play(G, 1, 0.0), _play(G, 2, 0.0)
    assert z1[0].tobytes() == z2[0].tobytes()                    # eps = 0: the seed plays no part
    assert len({bytes(z1[0][z1[1] == i].tobytes()) for i in np.unique(z1[1])}) == 1


@pytest.mark.gpu
def test_noise_conserves_the_simulation_budget():
    G, sims = 64, 100
    roots = synthetic_roots(S.GAME_C4, G, start=5, max_ply=8)
    for flags in (0, S.FLAG_FORCE_SPLIT, S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP):
        with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET, flags=flags) as e:
            e.reset_games(roots)
            e.set_root_noise(1.0, 0.5, 3)
            e.search(sims)
            assert e.counters()["simulations"] == G * sims
            for s in range(G):
                assert e.node_stats(s, 0)["visit_count"] == sims
