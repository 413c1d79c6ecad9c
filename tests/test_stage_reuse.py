"""Reuse of the engine's grow-only stage (HostEngine::ensure_stage): the chess entry points that take their device arrays
from it give, on an engine whose stage still holds the bytes of earlier calls, larger and smaller, exactly what they give
on a fresh engine."""
import numpy as np
import pytest

import selfplay_b200 as S
from selfplay_b200.weights_init import random_chess_checkpoint
from test_chess import export_all, random_games

G = 128          # the large batches fill the engine (spb_chess_predict takes at most num_games states)


def phase_inputs(seed, n):
    """n ongoing positions with their histories, and one legal move of each."""
    rng = np.random.default_rng(seed)
    games = [g for g in random_games(max(n, 8), seed, max_plies=160) if g.status() == S.ONGOING]
    games = [games[i] for i in rng.choice(len(games), n, replace=False)]
    moves = [g.legal_moves() for g in games]
    st, hist = export_all(games)
    return st, hist, np.array([m[rng.integers(len(m))] for m in moves], np.uint16)


def run_phase(e, st, hist, moves):
    """next_states (its history round trip feeds every later call), the rules, predict, reset with history, advance."""
    n = len(st)
    slots = np.arange(n, dtype=np.uint32)[::-1].copy()
    st2, hist2, err = e.next_states(st, hist, moves)
    out = [st2, hist2, err, *e.legal_moves(st2, hist2), e.encode(st2, hist2), *e.predict(st2, hist2, want_logits=True)]
    e.reset_games(st2, hist2, slots=slots)
    e.search(8)
    live = [int(s) for s in slots if e.root_children(int(s))[0]]     # a terminal root has no child to advance to
    out.append(e.advance([e.root_children(s)[2][0] for s in live], slots=live))
    out += [e.get_state(s, 0) for s in live]
    return [np.asarray(x).tobytes() for x in out]


@pytest.mark.gpu
def test_chess_calls_on_a_reused_stage_equal_a_fresh_engine():
    blob = random_chess_checkpoint(seed=0)
    phases = [phase_inputs(1, G), phase_inputs(2, 5), phase_inputs(3, G)]   # large -> small -> large

    def engine():
        e = S.ChessEngine(num_games=G, evaluator=S.EVAL_DET, max_nodes_per_tree=4096)
        e.load_weights(blob)
        return e

    with engine() as e:
        reused = [run_phase(e, *p) for p in phases]
    for i, p in enumerate(phases):
        with engine() as f:
            fresh = run_phase(f, *p)
        assert len(reused[i]) == len(fresh), i
        for k, (a, b) in enumerate(zip(reused[i], fresh)):
            assert a == b, (i, k)
