"""GPU parity: select / expand / backup / re-root kernels vs the oracle under the deterministic
evaluators — visit counts, value sums, priors and arena layout bit-exact."""
import json
import os

import numpy as np
import pytest

import selfplay_b200 as S
from helpers import synthetic_roots
from oracle import pyoracle as O

pytestmark = pytest.mark.gpu
KAT = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "survey_kats.json")))


def _assert_same_tree(e, f, slot, full=True):
    n = f.arena_len(slot)
    assert e.arena_len(slot) == n
    assert e.root_children(slot) == f.root_children(slot)
    ids = range(n) if full else list(range(min(n, 40))) + list(range(max(0, n - 40), n))
    for i in ids:
        assert e.node_stats(slot, i) == f.node_stats(slot, i), (slot, i)


PIPELINES = {"fused": 0, "async": S.FLAG_FORCE_SPLIT, "lockstep-graph": S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP,
             "lockstep": S.FLAG_FORCE_SPLIT | S.FLAG_LOCKSTEP | S.FLAG_NO_GRAPH}


@pytest.mark.parametrize("flags", list(PIPELINES.values()), ids=list(PIPELINES))
def test_survey_kats_on_device(flags):
    for S_, ev, key in [(800, S.EVAL_DET, "c4_det"), (100, S.EVAL_DET, "c4_det"), (800, S.EVAL_UNIFORM, "c4_uniform"), (9, S.EVAL_UNIFORM, "c4_uniform")]:
        with S.Engine(game=S.GAME_C4, num_games=3, evaluator=ev, flags=flags) as e:
            e.reset_games()
            e.search(S_)
            for slot in range(3):
                assert e.root_children(slot)[1] == KAT[key][str(S_)]
            if ev == S.EVAL_DET:
                assert e.node_stats(0, 0)["value_sum"] == KAT["c4_det_root_w"][str(S_)]
                assert e.arena_len(0) == KAT["c4_det_arena"][str(S_)]
            c = e.counters()
            assert c["simulations"] == 3 * S_ and c["evaluations"] + c["terminal_leaves"] == 3 * S_
            if S_ == 800 and ev == S.EVAL_DET:
                assert c["path_length_sum"] == 3 * KAT["c4_det_800_path_sum"] and c["terminal_leaves"] == 3
    for S_ in ("10", "11", "600"):
        with S.Engine(game=S.GAME_TTT, num_games=2, evaluator=S.EVAL_UNIFORM, flags=flags) as e:
            e.reset_games()
            e.search(int(S_))
            assert e.root_children(1)[1] == KAT["ttt_uniform"][S_]


@pytest.mark.parametrize("game,ev", [(S.GAME_C4, S.EVAL_DET), (S.GAME_C4, S.EVAL_UNIFORM), (S.GAME_TTT, S.EVAL_DET)])
@pytest.mark.parametrize("flags", list(PIPELINES.values())[:3], ids=list(PIPELINES)[:3])
def test_search_matches_oracle_node_for_node(game, ev, flags):
    G = 48
    roots = synthetic_roots(game, G, start=100, max_ply=21 if game == S.GAME_C4 else 5)
    f = O.Forest(game, G)
    f.reset(roots)
    with S.Engine(game=game, num_games=G, evaluator=ev, flags=flags) as e:
        e.reset_games(roots)
        for rnd, sims in enumerate([1, 37, 200]):             # statistics accumulate across calls
            e.search(sims)
            f.search(sims, ev)
            for slot in range(G):
                _assert_same_tree(e, f, slot, full=(slot < 4))
        ce, cf = e.counters(), f.counters()
        for k in ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "nodes_live"):
            assert ce[k] == cf[k], k
        a, c, i, n = e.root_children_all()
        for slot in range(G):
            fa, fc, fi = f.root_children(slot)
            assert list(a[slot, :n[slot]]) == fa and list(c[slot, :n[slot]]) == fc and list(i[slot, :n[slot]]) == fi
            assert np.array_equal(e.root_policy(slot), f.root_policy(slot))


@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
def test_use_subtree_and_greedy_games_match_oracle(game):
    """Full greedy games (main.rs:108-112 rule) with subtree reuse, compared after every move."""
    G = 12
    roots = synthetic_roots(game, G, start=7, max_ply=8 if game == S.GAME_C4 else 3)
    sims = 150
    f = O.Forest(game, G)
    f.reset(roots)
    with S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET) as e:
        e.reset_games(roots)
        live = list(range(G))
        for move in range(45):
            e.search(sims)
            f.search(sims, O.EVAL_DET)
            picks = []
            for slot in live:
                _assert_same_tree(e, f, slot, full=(move < 2 and slot < 3))
                acts, counts, ids = f.root_children(slot)
                best = max(range(len(ids)), key=lambda j: (counts[j], j))   # last max
                picks.append(ids[best])
            new_states = e.advance(picks, slots=live)
            nxt = []
            for k, slot in enumerate(live):
                f.use_subtree(slot, picks[k])
                want = f.get_state(slot, 0)
                assert O.state_from_record(new_states[k]).key() == want.key()
                assert e.get_state(slot, 0).key() == want.key()
                _assert_same_tree(e, f, slot, full=(move < 2 and slot < 3))
                last = f.arena_len(slot) - 1
                assert e.get_state(slot, last).key() == f.get_state(slot, last).key()
                if want.status == O.ONGOING:
                    nxt.append(slot)
            # finished trees are restarted so that every slot keeps searching (engine searches all live slots)
            done = [s for s in live if s not in nxt]
            if done:
                e.reset_games([roots[s] for s in done], slots=done)
                f.reset([roots[s] for s in done], slots=done)
            if move > 12 and not nxt:
                break
        # a slot listed twice is refused before any tree is touched
        e.search(sims)

        def snapshot(s):
            n = e.arena_len(s)
            return n, [e.node_stats(s, i) for i in range(n)], [e.get_state(s, i).key() for i in range(n)]
        before = snapshot(0)
        child = e.root_children(0)[2][0]
        for call in (lambda: e.advance([child, child], slots=[0, 0]), lambda: e.reset_games([roots[1], roots[2]], slots=[0, 0])):
            with pytest.raises(S.EngineError) as ei:
                call()
            assert ei.value.code == -1
            assert snapshot(0) == before


def test_survey_greedy_game_800():
    k = KAT["c4_det_greedy_800"]
    with S.Engine(game=S.GAME_C4, num_games=1, evaluator=S.EVAL_DET) as e:
        e.reset_games()
        actions, sizes = [], []
        for _ in range(7):
            e.search(800)
            sizes.append(e.arena_len(0))
            acts, counts, ids = e.root_children(0)
            best = max(range(len(ids)), key=lambda j: (counts[j], j))
            last_counts = counts
            st = e.advance([ids[best]])
            actions.append(acts[best])
        assert actions == k["actions"] and sizes == k["arena_sizes"] and last_counts == k["last_counts"]
        assert st[0]["status"] == S.WON


def test_selfplay_step_trajectories_match_oracle():
    """The on-device self-play ply (greedy rule) reproduces learner_concurrent.rs:179-238 driven by the oracle."""
    G, sims = 24, 60
    roots = synthetic_roots(S.GAME_C4, G, start=900, max_ply=30)
    f = O.Forest(O.GAME_C4, G)
    f.reset(roots)
    want = {}      # game id -> list of (stones, counts by action, player, outcome)
    hist = {s: [] for s in range(G)}
    live = set(range(G))
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        e.reset_games(roots)
        finished_total = 0
        while live:
            e.search(sims)
            f.search(sims, O.EVAL_DET)
            fin = e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
            n_fin = 0
            for slot in sorted(live):
                acts, counts, ids = f.root_children(slot)
                root = f.get_state(slot, 0)
                by_action = [0] * 9
                for a, c in zip(acts, counts):
                    by_action[a] = c
                hist[slot].append((root.stones[0], root.stones[1], by_action, root.current_player))
                best = max(range(len(ids)), key=lambda j: (counts[j], j))
                child = f.get_state(slot, ids[best])
                if child.status != O.ONGOING:
                    value = -1 if child.status == O.WON else 0
                    want[slot] = [(x, o, ba, p, value if p == child.current_player else -value) for (x, o, ba, p) in hist[slot]]
                    live.discard(slot)
                    n_fin += 1
                else:
                    f.use_subtree(slot, ids[best])
            assert fin == n_fin
            finished_total += n_fin
            # oracle forest keeps searching finished trees; harmless (they are never read again)
        pos, gids = e.drain_trajectories()
    assert sorted(set(int(g) for g in gids)) == sorted(want)
    k = 0
    for g in sorted(want):
        for ply, (x, o, ba, p, outcome) in enumerate(want[g]):
            r = pos[k]
            assert int(gids[k]) == g and int(r["ply"]) == ply
            assert (int(r["stones"][0]), int(r["stones"][1]), int(r["current_player"]), int(r["outcome"])) == (x, o, p, outcome)
            assert list(r["visit_counts"]) == ba
            k += 1
    assert k == len(pos)


def test_fixed_pool_exhaustion_is_an_error_not_ub():
    with S.Engine(game=S.GAME_C4, num_games=2, evaluator=S.EVAL_DET, max_nodes_per_tree=64, flags=S.FLAG_FIXED_POOL) as e:
        e.reset_games()
        with pytest.raises(S.EngineError) as ei:
            e.search(200)
        assert ei.value.code == -3
        e.reset_games()
        e.search(5)                                  # engine stays usable
        assert sum(e.root_children(0)[1]) == 4


@pytest.mark.parametrize("flags", list(PIPELINES.values())[:3], ids=list(PIPELINES)[:3])
def test_pools_grow_like_the_reference_arena(flags):
    """mcts.rs:19 — the reference's arena is an unbounded Vec.  Starting from 16 nodes per tree, the pools are widened
    before each search that could outgrow them and the trees stay bit-identical to the oracle, re-roots included."""
    G = 6
    roots = synthetic_roots(S.GAME_C4, G, start=40, max_ply=6)
    f = O.Forest(O.GAME_C4, G)
    f.reset(roots)
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET, max_nodes_per_tree=16, flags=flags) as e:
        e.reset_games(roots)
        for sims in (40, 300, 150, 700):
            e.search(sims)
            f.search(sims, O.EVAL_DET)
            picks = []
            for slot in range(G):
                _assert_same_tree(e, f, slot, full=False)
                acts, counts, ids = f.root_children(slot)
                assert ids, "roots this shallow cannot finish within four moves"
                best = max(range(len(ids)), key=lambda j: (counts[j], j))
                picks.append(ids[best])
            e.advance(picks)
            for slot in range(G):
                f.use_subtree(slot, picks[slot])
                _assert_same_tree(e, f, slot, full=False)
        assert max(e.arena_len(s) for s in range(G)) > 2048


def test_reference_shaped_host_api():
    """Mcts / Tree mirror of mcts.rs:196 — result i belongs to trees[i]."""
    with S.Engine(game=S.GAME_C4, num_games=3, evaluator=S.EVAL_DET) as e:
        trees = [S.Tree(e, i) for i in range(3)]
        mcts = S.Mcts(S.Args(num_searches=100), e)
        res = mcts.search(trees)
        for policy, pairs in res:
            assert [int(c) for _, c in pairs] == KAT["c4_det"]["100"]
            assert abs(float(policy.sum()) - 1.0) < 1e-6
        best = max(res[0][1], key=lambda p: (p[1], p[0]))[0]
        trees[0].use_subtree(best)
        assert trees[0].node_state(0).num_actions_played == 1


def test_selfplay_step_temperature_sampling_distribution():
    """learner_concurrent.rs:189-194: the move is sampled in proportion to visit_count^temperature.  The reference
    uses the unseedable thread_rng, so only the distribution can be checked (counter-based RNG on the device)."""
    G, sims, temp = 1024, 200, 1.25
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        e.reset_games()
        e.search(sims)
        acts, counts, ids = e.root_children(0)
        e.selfplay_step(S.MOVE_TEMPERATURE, temperature=temp, seed=12345)
        chosen = np.zeros(7)
        for slot in range(G):
            st = e.get_state(slot, 0)
            col = [c for c in range(7) if (st.stones[0] >> (c * 7)) & 1][0]
            chosen[col] += 1
        w = np.array([float(c) ** temp for c in counts])
        p = np.zeros(7)
        p[acts] = w / w.sum()
        expected = p * G
        assert chosen.sum() == G
        chi2 = float((((chosen - expected) ** 2) / np.maximum(expected, 1e-9))[expected > 0].sum())
        assert chi2 < 40, (chi2, chosen, expected)            # 6 degrees of freedom; 40 is far in the tail
        assert np.all(chosen[expected == 0] == 0)
        # a different seed gives a different sample; the same seed the same one
        e.reset_games(); e.search(sims); e.selfplay_step(S.MOVE_TEMPERATURE, temperature=temp, seed=12345)
        again = [e.get_state(s, 0).key() for s in range(64)]
        e.reset_games(); e.search(sims); e.selfplay_step(S.MOVE_TEMPERATURE, temperature=temp, seed=12345)
        assert again == [e.get_state(s, 0).key() for s in range(64)]


def test_one_process_can_drive_engines_on_several_gpus():
    """main.rs:169 runs one Mcts per worker thread; a host that owns several GPUs creates one engine per device in the
    same process.  Each engine (tree kernels + tcgen05 evaluator) must work on its own device."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from selfplay_b200.weights_init import random_checkpoint
    blob = random_checkpoint(1, 0)
    res = []
    for dev in (0, 1):
        with S.Engine(game=S.GAME_C4, num_games=40, evaluator=S.EVAL_NET, device=dev) as e:
            e.load_weights(blob)
            e.reset_games()
            e.search(60)
            res.append([e.root_children(s) for s in range(40)])
    assert res[0] == res[1]
    assert sum(res[0][0][1]) == 59


def test_trajectory_buffer_overflow_parks_games_and_loses_nothing():
    """A finished game whose trajectory does not fit the output buffer is parked, the call reports SPB_ERR_STATE, and
    after a drain the next ply emits it: every record that is drained is complete, no game is lost, and the union of all
    drains equals the trajectories of an engine with a large buffer."""
    G, sims = 64, 30

    def play(capacity):
        out = []
        with S.Engine(game=S.GAME_TTT, num_games=G, evaluator=S.EVAL_DET, trajectory_capacity=capacity) as e:
            e.reset_games()
            errors = 0
            for _ in range(40):
                e.search(sims)
                try:
                    e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
                except S.EngineError as err:
                    assert err.code == -6 and "trajectory buffer full" in str(err)
                    errors += 1
                pos, ids = e.drain_trajectories()
                assert len(pos) <= max(capacity, 9) or capacity == 0
                out += [(int(i), p.tobytes()) for p, i in zip(pos, ids)]
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)               # emits what is still parked
            pos, ids = e.drain_trajectories()
            out += [(int(i), p.tobytes()) for p, i in zip(pos, ids)]
        return sorted(out), errors

    want, e0 = play(0)
    got, e1 = play(20)                                            # room for two or three games per ply
    assert e0 == 0 and e1 > 0
    assert len(want) > G * 5 and got == want


def _play_generation(e, roots, plies, sims):
    e.reset_games(roots)
    for _ in range(plies):
        e.search(sims)
        e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)


def test_gather_over_the_c_abi_with_one_rank_equals_drain():
    """spb_gather_trajectories on a one-rank NCCL communicator returns exactly what spb_drain_trajectories returns
    (ordered by game id, then ply), the size query keeps the records staged, and the learner hand-off tensors follow."""
    G, plies, sims = 48, 14, 40
    roots = synthetic_roots(S.GAME_C4, G, start=0)
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        _play_generation(e, roots, plies, sims)
        want_pos, want_ids = e.drain_trajectories()
    assert len(want_pos) > 50
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as e:
        e.comm_init(S.comm_unique_id(), 0, 1)
        _play_generation(e, roots, plies, sims)
        pos, ids = e.gather_trajectories(0)
        assert pos.tobytes() == want_pos.tobytes() and ids.tobytes() == want_ids.tobytes()
        again, _ = e.gather_trajectories(0)                      # handed over: nothing left, the local buffer is empty too
        assert len(again) == 0 and len(e.drain_trajectories()[0]) == 0
        e.comm_destroy()
    enc, pol, val = S.positions_to_training(S.GAME_C4, pos)
    assert enc.shape == (len(pos), 3, 6, 7) and np.allclose(pol.sum(1), 1.0) and set(np.unique(val)) <= {-1.0, 0.0, 1.0}
    assert np.array_equal(enc[:, 2], 1.0 - enc[:, 0] - enc[:, 1])


@pytest.mark.gpu
def test_root_children_all_writes_into_caller_buffers():
    """bench.py's end-to-end steps hand page-locked arrays to root_children_all(out=...): same numbers as a fresh call,
    into pageable and page-locked arrays.  Each row equals the per-slot call's, which writes whole rows (no move, count 0
    and id 0 past n) and takes a NULL n_children.  For both engines; the odd slots hold no tree."""
    import torch
    keep = []

    def pinned(x):
        t = torch.empty(max(1, x.nbytes), dtype=torch.uint8, pin_memory=True)
        keep.append(t)
        out = t.numpy()[:x.nbytes].view(x.dtype).reshape(x.shape)
        out[...] = 0xFF
        return out
    for make in (lambda: S.Engine(game=S.GAME_C4, num_games=16, evaluator=S.EVAL_DET),
                 lambda: S.Engine(game=S.GAME_TTT, num_games=16, evaluator=S.EVAL_DET),
                 lambda: S.ChessEngine(num_games=16, evaluator=S.EVAL_DET)):
        with make() as e:
            e.reset_games(slots=list(range(0, 16, 2)))
            e.search(50)
            fresh = e.root_children_all()
            for bufs in (tuple(np.full_like(x, 0xFF) for x in fresh), tuple(pinned(x) for x in fresh)):
                got = e.root_children_all(bufs)
                assert all(g is b for g, b in zip(got, bufs))
                for g, f in zip(got, fresh):
                    assert (g == f).all()
            mv, cnt, ids, n = fresh
            assert n[0] > 0 and n[1] == 0
            for slot in range(16):
                row = [np.full_like(x[slot], 0xAB) for x in (mv, cnt, ids)]
                e._chk(e._fn("root_children")(e._h, slot, *map(np.ctypeslib.as_ctypes, row), None))
                assert all((r == x[slot]).all() for r, x in zip(row, (mv, cnt, ids)))
                k = int(n[slot])
                assert (row[0][k:] == np.iinfo(mv.dtype).max).all() and not row[1][k:].any() and not row[2][k:].any()
