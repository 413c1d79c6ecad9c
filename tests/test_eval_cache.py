"""Evaluation cache of the asynchronous pipeline (async.cuh, DESIGN.md §4.2a): a leaf whose position its tree has already
sent to the evaluator in the same search is expanded with that record instead of being evaluated again.  The evaluator is
a pure function of the position, so nothing a caller sees may change; what changes is the number of positions the
evaluator receives (async_stats()["boards"]) against the leaves the reference evaluates (counters()["evaluations"])."""
import numpy as np
import pytest

import pyref
import selfplay_b200 as S
from helpers import splitmix64, synthetic_roots
from oracle import torch_net

pytestmark = pytest.mark.gpu


def _pyref_root(game, g, max_ply):
    """helpers.synthetic_root, replayed with the pure-Python rules."""
    while True:
        r = splitmix64(0x5EED0000 + g)
        s = pyref.C4() if game == S.GAME_C4 else pyref.TTT()
        ok = True
        for _ in range(r % max_ply):
            va = s.valid_actions()
            r = splitmix64(r)
            s = s.next_state(va[r % len(va)])
            if s.status != 0:
                ok = False
                break
        if ok:
            return s
        g += 1 << 32


M64 = (1 << 64) - 1
MAX_SLOTS, WINDOW = 4096, 32                                      # tree.cuh: EVAL_CACHE_MAX_SLOTS, EVAL_CACHE_WINDOW


def _table_slots(sims):
    """Slots per tree of the engine's table after a first search of `sims` simulations (engine.cu: ensure_eval_cache)."""
    n = WINDOW
    while n < 2 * sims and n < MAX_SLOTS:
        n <<= 1
    return n


def _pyref_search(root, sims):
    """One tree searched by the restatement under DetEval -> (root visit counts, evaluations, evaluations of a position
    this tree had already evaluated in the search, positions the engine's table sends to the evaluator).  The last one
    models the table: probe windows of WINDOW slots from splitmix64 of the 16-byte position, first empty or equal slot,
    no insert when the window is full."""
    t = pyref.Tree(root)
    slots = _table_slots(sims)
    table = [None] * slots
    seen, n = set(), [0, 0, 0]

    def evaluator(st):
        x, o = st.stones()
        key = (x, o | (st.n << 48) | (st.player << 60))            # games.cuh: ps_make of an ongoing position
        n[0] += 1
        n[1] += key in seen
        seen.add(key)
        h = pyref.splitmix64(key[0] ^ pyref.splitmix64(key[1])) & 0xFFFFFFFF
        for i in range(WINDOW):
            s = (h + i) & (slots - 1)
            if table[s] is None or table[s] == key:
                if table[s] is None:
                    table[s] = key
                    n[2] += 1
                break
        else:
            n[2] += 1
        return pyref.det_eval(st)

    pyref.search([t], sims, evaluator)
    return t.root_counts(), n[0], n[1], n[2]


def _async_search(game, G, sims, roots, flags=S.FLAG_FORCE_SPLIT):
    with S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET, flags=flags) as e:
        e.reset_games(roots)
        e.reset_counters()
        e.search(sims)
        return e.root_children_all(), e.counters(), e.async_stats()


@pytest.mark.parametrize("game,G,sims,max_ply", [(S.GAME_C4, 32, 200, 21), (S.GAME_TTT, 32, 60, 4)])
def test_hits_are_the_repeated_leaves_of_each_tree(game, G, sims, max_ply):
    """Under DetEval the asynchronous pipeline equals the restatement node for node, so the leaves served from the cache
    (evaluations - boards) are exactly the leaves that repeat an earlier leaf position of the same tree and search."""
    start = 100
    (_, counts, _, n), ctr, stats = _async_search(game, G, sims, synthetic_roots(game, G, start=start, max_ply=max_ply))
    evals = repeats = boards = 0
    for g in range(G):
        rc, ev, rep, nb = _pyref_search(_pyref_root(game, start + g, max_ply), sims)
        assert list(counts[g][:n[g]]) == rc, g
        evals += ev
        repeats += rep
        boards += nb
    assert ctr["evaluations"] == evals
    assert repeats > 0 and boards == evals - repeats              # no window is full at these sizes
    assert ctr["evaluations"] - stats["boards"] == repeats


def test_weights_swapped_between_searches_are_never_served_stale():
    """Entries live for one search (its epoch): after new weights the same roots search as on a fresh engine and as the
    lock-step pipeline (no cache).  The first search is short, so the second one also grows the table."""
    G, sims = 48, 40
    roots = synthetic_roots(S.GAME_C4, G, start=3)
    blob_a = torch_net.to_safetensors_tch(torch_net.make_net(S.GAME_C4, seed=11))
    blob_b = torch_net.to_safetensors_tch(torch_net.make_net(S.GAME_C4, seed=12))
    results = []
    for flags, first in ((0, blob_a), (0, None), (S.FLAG_LOCKSTEP, None)):
        with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
            if first is not None:
                e.load_weights(first)
                e.reset_games(roots)
                e.search(8)
            e.load_weights(blob_b)
            e.reset_games(roots)
            e.reset_counters()
            e.search(sims)
            got = [x.copy() for x in e.root_children_all()]
            e.search(9)                                           # a second search on the same trees: the next epoch
            got += [x.copy() for x in e.root_children_all()]
            c = e.counters()
            results.append((got, c, e.async_stats()["boards"] if flags == 0 else None))
    for got, c, _ in results[1:]:
        for u, v in zip(results[0][0], got):
            assert np.array_equal(u, v)
        for k in ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "nodes_live"):
            assert c[k] == results[0][1][k], k
    assert results[0][2] == results[1][2]                         # the same evaluations were served from the cache


def test_full_probe_windows_still_equal_lockstep():
    """Tic-tac-toe from the empty board at 20,000 simulations evaluates more distinct positions than fit at a low load into
    the largest table, so some probe windows are full and those positions are evaluated again; results stay those of the
    lock-step pipeline."""
    G, sims = 4, 20000
    got, ctr, stats = _async_search(S.GAME_TTT, G, sims, None)
    want, want_ctr, _ = _async_search(S.GAME_TTT, G, sims, None, flags=S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP)
    for u, v in zip(got, want):
        assert np.array_equal(u, v)
    for k in ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "nodes_live"):
        assert ctr[k] == want_ctr[k], k
    _, evals, repeats, boards = _pyref_search(pyref.TTT(), sims)
    assert boards > evals - repeats                               # the model: some positions found their window full
    assert ctr["evaluations"] == G * evals
    assert stats["boards"] == G * boards


def test_hit_fraction_at_the_bench_shape():
    """bench.py's default workload: 4,096 Connect4 trees x 800 simulations with its weights and roots.  The fraction of
    leaves served from the cache is reported (the CPU estimate from the restatement was 0.19)."""
    from selfplay_b200.synth import synthetic_roots_device
    from selfplay_b200.weights_init import random_checkpoint

    G, sims = 4096, 800
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, max_nodes_per_tree=8192) as e:
        e.load_weights(random_checkpoint(1, 0))
        e.reset_games(synthetic_roots_device(e, G, start=0, max_ply=21))
        e.reset_counters()
        e.search(sims)
        ctr, stats = e.counters(), e.async_stats()
    frac = 1.0 - stats["boards"] / ctr["evaluations"]
    print("evaluations %d boards %d hit fraction %.4f" % (ctr["evaluations"], stats["boards"], frac))
    assert ctr["simulations"] == G * sims
    assert 0.0 < frac < 1.0
