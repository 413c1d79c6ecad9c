"""Chess records across GPUs and on the device: spb_chess_comm_init / spb_chess_gather_trajectories and
spb_chess_positions_to_training_device.

CPU: chess records go through distributed.gather_records over gloo (world size 2) byte-identical to a one-rank merge; the new
entry points reject a NULL engine.
GPU: the gather on a one-rank NCCL communicator equals the drain of the same generation; the device builder equals the host
builder bit for bit (oracle records, real self-play records, sizes, duplicated moves, unaligned and NULL outputs, indices);
malformed rows are rejected with nothing written; with two GPUs, two ranks equal one rank playing all the games.
"""
import ctypes as C
import hashlib
import os
import socket

import numpy as np
import pytest

import selfplay_b200 as S
from oracle import pychess as P
from selfplay_b200.distributed import merge_trajectories
from test_chess import play, random_games
from test_chess_search import MIDGAME
from test_chess_selfplay import FIFTY_99, FORCED_MATE, NEAR_THREEFOLD, capped_roots, record_of

CH = S.chess
REC = CH.CHESS_POSITION_DTYPE


# ---- CPU ---------------------------------------------------------------------------------------------------------

def fake_chess_game(game_id: int):
    """Deterministic fake chess trajectory: 2 + game_id % 4 records whose bytes depend on (game id, ply)."""
    n = 2 + game_id % 4
    pos = np.zeros(n, REC)
    rng = np.random.default_rng(game_id)
    for ply in range(n):
        pos[ply]["state"]["piece"] = rng.integers(0, 1 << 62, 6, dtype=np.uint64)
        pos[ply]["visit_counts"][:20] = rng.integers(0, 1000, 20, dtype=np.uint32)
        pos[ply]["moves"][:] = CH.MOVE_NONE
        pos[ply]["moves"][:20] = rng.integers(0, 4096, 20, dtype=np.uint16)
        pos[ply]["n_moves"], pos[ply]["ply"], pos[ply]["outcome"] = 20, ply, game_id % 3 - 1
    return pos


def chess_rank_records(lo, hi, shuffle_seed):
    games = list(range(lo, hi))
    np.random.default_rng(shuffle_seed).shuffle(games)
    parts = [fake_chess_game(g) for g in games]
    pos = np.concatenate(parts) if parts else np.zeros(0, REC)
    ids = np.concatenate([np.full(len(p), g, np.uint64) for p, g in zip(parts, games)]) if parts else np.zeros(0, np.uint64)
    return pos, ids


def _gloo_worker(rank, world, port, total_games, out_path):
    import torch.distributed as dist
    from selfplay_b200.distributed import gather_records, shard_range
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lo, hi = shard_range(total_games, rank, world)
    pos, ids = chess_rank_records(lo, hi, 100 + rank)
    mpos, mids = gather_records(pos, ids, dst=0)
    if rank == 0:
        np.savez(out_path, pos=mpos.view(np.uint8), ids=mids, dtype_ok=mpos.dtype == REC)
    else:
        assert len(mpos) == 0 and mpos.dtype == REC
    dist.barrier()
    dist.destroy_process_group()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_chess_records_gather_over_gloo_like_one_rank(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "merged.npz")
    mp.spawn(_gloo_worker, args=(2, free_port(), 13, out), nprocs=2, join=True)
    got = np.load(out)
    want_pos, want_ids = merge_trajectories([chess_rank_records(0, 13, 7)])
    assert want_pos.dtype == REC and bool(got["dtype_ok"])
    assert got["pos"].tobytes() == want_pos.tobytes() and got["ids"].tobytes() == want_ids.tobytes()


def test_merge_of_nothing_keeps_the_record_type():
    pos, ids = merge_trajectories([], dtype=REC)
    assert pos.dtype == REC and len(pos) == 0 and len(ids) == 0
    assert merge_trajectories([])[0].dtype == S.POSITION_DTYPE


def test_new_entry_points_reject_a_null_engine():
    L = S.load_library()
    n = C.c_size_t(7)
    buf = (C.c_uint8 * S.COMM_ID_BYTES)()
    assert L.spb_chess_comm_init(None, C.cast(buf, C.c_void_p), 0, 1) == -1
    assert L.spb_chess_comm_destroy(None) == -1
    assert L.spb_chess_gather_trajectories(None, 0, None, 0, C.byref(n), None) == -1
    assert L.spb_chess_positions_to_training_device(None, None, 0, None, 0, None, None, None) == -1


# ---- GPU: gather -------------------------------------------------------------------------------------------------

GATHER_GAMES = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE), play("e2e4 e7e5 g1f3")] * 16


def play_generation(e, steps=8, sims=30):
    st, hist = capped_roots(GATHER_GAMES, 506)                         # every game ends after 7 records, then restarts
    e.reset_games(st, hist)
    for _ in range(steps):
        e.search(sims)
        e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist)


@pytest.mark.gpu
def test_one_rank_gather_equals_the_drain_of_the_same_generation():
    G = len(GATHER_GAMES)
    with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as e:
        play_generation(e)
        want_pos, want_ids = e.drain_trajectories()
    assert len(want_pos) >= 6 * G                                       # games end at the history cap after 7 records
    L = S.load_library()
    with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as e:
        with pytest.raises(S.EngineError) as ei:                       # no communicator yet
            e.gather_trajectories(0)
        assert ei.value.code == -6
        e.comm_init(S.comm_unique_id(), 0, 1)
        with pytest.raises(S.EngineError) as ei:
            e.gather_trajectories(1)
        assert ei.value.code == -1
        play_generation(e)
        # size query, then a buffer one record short: the records stay staged; the next call delivers them
        n = C.c_size_t()
        assert L.spb_chess_gather_trajectories(e._h, 0, None, 0, C.byref(n), None) == 0 and n.value == len(want_pos)
        short = np.zeros(n.value - 1, REC)
        assert L.spb_chess_gather_trajectories(e._h, 0, short.ctypes.data, len(short), C.byref(n), None) == 0
        assert n.value == len(want_pos) and not short.view(np.uint8).any()
        pos, ids = e.gather_trajectories(0)
        assert pos.tobytes() == want_pos.tobytes() and ids.tobytes() == want_ids.tobytes()
        again, _ = e.gather_trajectories(0)
        assert len(again) == 0 and len(e.drain_trajectories()[0]) == 0
        e.comm_destroy()


@pytest.mark.gpu
def test_engine_that_never_played_gathers_nothing_and_destroy_releases_the_communicator():
    e = CH.ChessEngine(num_games=8, evaluator=S.EVAL_DET)
    e.comm_init(S.comm_unique_id(), 0, 1)
    pos, ids = e.gather_trajectories(0)
    assert len(pos) == 0 and len(ids) == 0 and pos.dtype == REC
    assert len(e.drain_trajectories()[0]) == 0
    e.close()                                                          # communicator still live
    with CH.ChessEngine(num_games=4, evaluator=S.EVAL_DET) as e2:
        e2.comm_init(S.comm_unique_id(), 0, 1)
        assert len(e2.gather_trajectories(0)[0]) == 0
        e2.comm_destroy()
        e2.comm_destroy()                                              # no communicator: nothing to do


def _nccl_worker(rank, world, port, out_path):
    import torch
    import torch.distributed as dist
    from selfplay_b200.distributed import comm_init_over_process_group
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)       # carries only the 128-byte id
    g = len(GATHER_GAMES) // world
    st, hist = capped_roots(GATHER_GAMES, 506)
    st, hist = st[rank * g:(rank + 1) * g], hist[rank * g:(rank + 1) * g]
    with CH.ChessEngine(num_games=g, evaluator=S.EVAL_DET, device=rank, game_id_base=rank * g, game_id_stride=world * g) as e:
        comm_init_over_process_group(e, rank, world)
        e.reset_games(st, hist)
        for _ in range(8):
            e.search(30)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist)
        pos, ids = e.gather_trajectories(0)
        e.comm_destroy()
    if rank == 0:
        np.savez(out_path, sha=hashlib.sha256(pos.tobytes() + ids.tobytes()).hexdigest(), n=len(pos))
    else:
        assert len(pos) == 0
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_ranks_gather_what_one_rank_plays(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "two.npz")
    mp.spawn(_nccl_worker, args=(2, free_port(), out), nprocs=2, join=True)
    with CH.ChessEngine(num_games=len(GATHER_GAMES), evaluator=S.EVAL_DET) as e:
        play_generation(e)
        pos, ids = e.drain_trajectories()
    got = np.load(out)
    assert int(got["n"]) == len(pos) and str(got["sha"]) == hashlib.sha256(pos.tobytes() + ids.tobytes()).hexdigest()


# ---- GPU: the device training builder ----------------------------------------------------------------------------

def oracle_records():
    """The records of test_positions_to_training_matches_the_oracle: random games, repetition and fifty-move positions."""
    rng = np.random.default_rng(11)
    games = [g for g in random_games(6, seed=5, max_plies=80) if g.status() == S.ONGOING][::3]
    games += [play("g1f3 g8f6 f3g1 f6g8"), play(NEAR_THREEFOLD), P.Game(FIFTY_99), P.Game(FORCED_MATE), P.Game(MIDGAME)]
    return np.array([record_of(g, rng, i, int(rng.integers(-1, 2))) for i, g in enumerate(games)], REC)


@pytest.fixture(scope="module")
def selfplay_records():
    """Records of 1,024 real self-play games (DetEval), ended by the history cap after 4 records each."""
    games = [P.Game(), P.Game(MIDGAME), P.Game(P.KIWIPETE), play("e2e4 e7e5 g1f3")] * 256
    st, hist = capped_roots(games, 509)
    with CH.ChessEngine(num_games=len(games), evaluator=S.EVAL_DET) as e:
        e.reset_games(st, hist)
        for _ in range(4):
            e.search(40)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
        pos, _ = e.drain_trajectories()
    assert len(pos) == 4 * len(games)
    return pos


@pytest.fixture(scope="module")
def engine():
    with CH.ChessEngine(num_games=1, evaluator=S.EVAL_DET) as e:
        yield e


def to_numpy(tensors):
    return [t.cpu().numpy() for t in tensors]


def assert_bit_identical(got, want, nan_rows=()):
    for g, w in zip(got, want):
        assert g.shape == w.shape and g.dtype == np.float32
        ok = np.ones(len(w), bool)
        ok[list(nan_rows)] = False
        assert np.array_equal(g[ok].view(np.uint32), w[ok].view(np.uint32))
        for r in nan_rows:
            assert np.array_equal(g[r], w[r], equal_nan=True)


@pytest.mark.gpu
def test_device_builder_equals_host_builder_on_oracle_records(engine):
    recs = oracle_records()
    assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, recs)), CH.positions_to_training(recs))


@pytest.mark.gpu
def test_device_builder_equals_host_builder_on_self_play_records(engine, selfplay_records):
    import torch
    recs = selfplay_records
    want = CH.positions_to_training(recs)
    assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, recs)), want)
    # records already in device memory, as a uint8 [n, 1624] tensor
    dev = torch.from_numpy(recs.view(np.uint8).reshape(len(recs), -1)).cuda()
    assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, dev)), want)
    for n in (0, 1, 333, 4093):                                        # no multiple of any block size
        got = to_numpy(CH.positions_to_training_device(engine, recs[:n]))
        assert got[0].shape == (n, 19, 8, 8) and got[1].shape == (n, 4672) and got[2].shape == (n, 1)
        assert_bit_identical(got, [w[:n] for w in want])


@pytest.mark.gpu
def test_duplicated_move_and_zero_counts_match_the_host(engine, selfplay_records):
    recs = selfplay_records[:8].copy()
    r = recs[1]
    r["moves"][1] = r["moves"][0]                                      # the later child wins on both sides
    r["visit_counts"][:2] = (7, 11)
    recs[2]["moves"][3:6] = recs[2]["moves"][2]
    recs[3]["visit_counts"][:] = 0                                     # 0 / 0: NaN on both sides
    want = CH.positions_to_training(recs)
    assert want[1][1, CH.policy_index(int(r["state"]["side"]), int(r["moves"][0]))] == np.float32(11) / np.float32(r["visit_counts"].sum(dtype=np.uint64))
    assert np.isnan(want[1][3]).any()
    assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, recs)), want, nan_rows=(3,))


def raw_outputs(n, offset_floats=0, fill=np.float32(-7.5)):
    import torch
    bufs = [torch.full((n * k + offset_floats,), float(fill), dtype=torch.float32, device="cuda") for k in (19 * 64, 4672, 1)]
    ptrs = [b.data_ptr() + 4 * offset_floats for b in bufs]
    return bufs, ptrs


def raw_call(e, pos_t, n_positions, idx_ptr, n, ptrs):
    import torch
    torch.cuda.synchronize()
    return e._L.spb_chess_positions_to_training_device(e._h, pos_t.data_ptr(), n_positions, idx_ptr, n, *ptrs)


@pytest.mark.gpu
def test_unaligned_and_null_outputs(engine, selfplay_records):
    import torch
    recs = selfplay_records[:301]
    want = CH.positions_to_training(recs)
    pos_t = torch.from_numpy(recs.view(np.uint8).reshape(len(recs), -1)).cuda()
    n = len(recs)
    bufs, ptrs = raw_outputs(n, offset_floats=1)                       # 4-byte aligned only: the scalar path
    assert raw_call(engine, pos_t, n, None, n, ptrs) == 0
    got = [b.cpu().numpy()[1:].reshape(w.shape) for b, w in zip(bufs, want)]
    assert_bit_identical(got, want)
    for k in range(3):                                                 # each output NULL in turn, the others written
        bufs, ptrs = raw_outputs(n)
        ptrs[k] = None
        assert raw_call(engine, pos_t, n, None, n, ptrs) == 0
        for j in range(3):
            host = bufs[j].cpu().numpy()
            if j == k:
                assert (host == np.float32(-7.5)).all()
            else:
                assert np.array_equal(host.view(np.uint32), want[j].reshape(-1).view(np.uint32)), (k, j)
    assert raw_call(engine, pos_t, n, None, n, [None, None, None]) == 0


@pytest.mark.gpu
def test_indices_pick_rows_of_a_device_resident_buffer(engine, selfplay_records):
    import torch
    recs = selfplay_records
    rng = np.random.default_rng(4)
    idx = rng.integers(0, len(recs), 777)
    idx[:10] = idx[10]                                                 # repeats
    want = CH.positions_to_training(recs[idx])
    dev = torch.from_numpy(recs.view(np.uint8).reshape(len(recs), -1)).cuda()
    for ix in (idx, torch.from_numpy(idx.astype(np.int64)).cuda(), torch.from_numpy(idx.astype(np.uint64)).cuda()):
        assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, dev, ix)), want)
    # with indices, n may exceed n_positions
    small = recs[:5]
    ix = rng.integers(0, 5, 64)
    assert_bit_identical(to_numpy(CH.positions_to_training_device(engine, small, ix)), CH.positions_to_training(small[ix]))


@pytest.mark.gpu
def test_malformed_rows_are_rejected_and_nothing_is_written(engine, selfplay_records):
    import torch
    recs = selfplay_records[:40].copy()
    L = S.load_library()
    cases = []
    for field, value in (("n_moves", 0), ("n_moves", 257)):
        bad = recs.copy()
        bad[6][field] = value
        bad[9][field] = value
        cases.append((bad, None))
    bad = recs.copy()
    bad[6]["state"]["side"] = 2
    cases.append((bad, None))
    bad = recs.copy()
    bad[6]["moves"][0] = 7 | (0 << 6) | (3 << 12)                      # h1-a1 as a rook promotion: off the policy
    cases.append((bad, None))
    idx = np.arange(40, dtype=np.int64)
    idx[6] = 40                                                        # index >= n_positions
    cases.append((recs, idx))
    for bad, ix in cases:
        pos_t = torch.from_numpy(bad.view(np.uint8).reshape(len(bad), -1)).cuda()
        idx_t = None if ix is None else torch.from_numpy(ix).cuda()
        bufs, ptrs = raw_outputs(40)
        rc = raw_call(engine, pos_t, 40, None if idx_t is None else idx_t.data_ptr(), 40, ptrs)
        assert rc == -1
        assert "row 6" in L.spb_chess_last_error(engine._h).decode()
        for b in bufs:
            assert (b.cpu().numpy() == np.float32(-7.5)).all()
        with pytest.raises(S.EngineError) as ei:
            CH.positions_to_training_device(engine, bad, ix)
        assert ei.value.code == -1
    # a host pointer, and n > n_positions without indices
    bufs, ptrs = raw_outputs(40)
    assert engine._L.spb_chess_positions_to_training_device(engine._h, recs.ctypes.data, 40, None, 40, *ptrs) == -1
    pos_t = torch.from_numpy(recs.view(np.uint8).reshape(40, -1)).cuda()
    assert raw_call(engine, pos_t, 40, None, 41, ptrs) == -1
    for b in bufs:
        assert (b.cpu().numpy() == np.float32(-7.5)).all()
