"""The learner hand-off in device memory: spb_drain_trajectories_device / spb_chess_drain_trajectories_device,
spb_gather_trajectories_device / spb_chess_gather_trajectories_device and spb_positions_to_training_device.

CPU: the Python wrappers reject CPU tensors, wrong dtypes and wrong widths before they reach the library.
GPU: every device form equals its host form byte for byte (records, ids, training tensors) for Connect4, tic-tac-toe and
chess; size queries, short and host buffers, offset slices, parking, staging across calls and the form rules of a pending
gather; with two GPUs, a two-rank device gather equals one rank playing all the games.
"""
import ctypes as C
import hashlib
import os

import numpy as np
import pytest

import selfplay_b200 as S
from helpers import synthetic_roots
from test_chess_gather import GATHER_GAMES, assert_bit_identical, free_port, play_generation

CH = S.chess
W_C4, W_CHESS = S.POSITION_DTYPE.itemsize, CH.CHESS_POSITION_DTYPE.itemsize


# ---- CPU -------------------------------------------------------------------------------------------------------------

def fake(cls, **attrs):
    """An engine object with no library handle: what the wrappers check before any call."""
    e = object.__new__(cls)
    e._h, e._L, e.device = None, S.load_library(), 0
    for k, v in attrs.items():
        setattr(e, k, v)
    return e


def test_wrappers_reject_cpu_tensors_wrong_dtypes_and_widths():
    import torch
    c4, chess = fake(S.Engine, game=S.GAME_C4), fake(CH.ChessEngine)
    for drain, width in ((c4.drain_trajectories_device, W_C4), (chess.drain_trajectories_device, W_CHESS),
                         (c4.gather_trajectories_device, W_C4), (chess.gather_trajectories_device, W_CHESS)):
        with pytest.raises(TypeError, match="CUDA"):
            drain(out=torch.zeros((4, width), dtype=torch.uint8))
        with pytest.raises(TypeError, match="CUDA"):
            drain(out=np.zeros((4, width), np.uint8))
        with pytest.raises(TypeError, match="torch.uint8"):
            drain(out=torch.zeros((4, width), dtype=torch.int32))
        with pytest.raises(ValueError, match="n, %d" % width):
            drain(out=torch.zeros((4, width + 8), dtype=torch.uint8))
        with pytest.raises(ValueError):
            drain(out=torch.zeros(4 * width, dtype=torch.uint8))
        with pytest.raises(TypeError, match="torch.int64"):
            drain(ids_out=torch.zeros(4, dtype=torch.float64))
        with pytest.raises(TypeError, match="CUDA"):
            drain(ids_out=torch.zeros(4, dtype=torch.int64))
    with pytest.raises(TypeError, match="CUDA"):
        S.positions_to_training_device(c4, torch.zeros((4, W_C4), dtype=torch.uint8))
    with pytest.raises(ValueError, match="n, 56"):
        S.positions_to_training_device(c4, torch.zeros((4, W_CHESS), dtype=torch.uint8))
    with pytest.raises(TypeError, match="torch.uint8"):
        S.positions_to_training_device(c4, torch.zeros((4, W_C4), dtype=torch.float32))
    with pytest.raises(TypeError, match="indices"):
        S.positions_to_training_device(c4, np.zeros(4, S.POSITION_DTYPE), torch.zeros(4, dtype=torch.float32))


# ---- GPU: helpers ----------------------------------------------------------------------------------------------------

def records(t):
    """CUDA uint8 [n, w] -> host bytes."""
    return t.cpu().numpy().tobytes()


def ids_bytes(t):
    return t.cpu().numpy().astype(np.uint64).tobytes()


def play_c4(e, G, plies, sims, seed, game=S.GAME_C4):
    """EVAL_DET search, seeded temperature moves, restarts: games of many lengths finish out of order."""
    roots = synthetic_roots(game, G, start=0, max_ply=9 if game == S.GAME_TTT else 21)
    e.reset_games(roots)
    for p in range(plies):
        e.search(sims)
        e.selfplay_step(S.MOVE_TEMPERATURE, temperature=1.0, seed=seed + p, restart_roots=roots)


def c4_pair(game, G, plies, sims, seed=7, **kw):
    """Two identically configured engines that have played the same plies."""
    es = [S.Engine(game=game, num_games=G, evaluator=S.EVAL_DET, **kw) for _ in range(2)]
    for e in es:
        play_c4(e, G, plies, sims, seed, game)
    return es


def cuda_full(shape, value, dtype):
    import torch
    return torch.full(shape, value, dtype=dtype, device="cuda")


# ---- GPU: drain ------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("game,G,plies,sims", [(S.GAME_C4, 48, 30, 24), (S.GAME_TTT, 64, 20, 24), (S.GAME_C4, 4096, 30, 8)])
def test_device_drain_equals_host_drain(game, G, plies, sims):
    a, b = c4_pair(game, G, plies, sims)
    with a, b:
        want_pos, want_ids = a.drain_trajectories()
        pos, ids = b.drain_trajectories_device()
        assert pos.is_cuda and ids.is_cuda and pos.shape == (len(want_pos), W_C4)
        assert len(want_pos) > G and records(pos) == want_pos.tobytes() and ids_bytes(ids) == want_ids.tobytes()
        assert len(b.drain_trajectories()[0]) == 0 and len(b.drain_trajectories_device()[0]) == 0


@pytest.mark.gpu
def test_chess_device_drain_equals_host_drain():
    G = len(GATHER_GAMES)
    with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as a, CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as b:
        play_generation(a)
        play_generation(b)
        want_pos, want_ids = a.drain_trajectories()
        pos, ids = b.drain_trajectories_device()
        assert len(want_pos) >= 6 * G and pos.shape == (len(want_pos), W_CHESS)
        assert records(pos) == want_pos.tobytes() and ids_bytes(ids) == want_ids.tobytes()
        assert len(b.drain_trajectories_device()[0]) == 0


@pytest.mark.gpu
def test_parked_games_drain_to_the_device_and_nothing_is_lost():
    """The pattern of test_trajectory_buffer_overflow_parks_games_and_loses_nothing: with a small buffer the union of the
    device drains equals the union of the host drains."""
    G, sims = 64, 30

    def play(device):
        out = []
        with S.Engine(game=S.GAME_TTT, num_games=G, evaluator=S.EVAL_DET, trajectory_capacity=20) as e:
            e.reset_games()
            errors = 0
            for _ in range(41):
                e.search(sims)
                try:
                    e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
                except S.EngineError as err:
                    assert err.code == -6
                    errors += 1
                if device:
                    pos, ids = e.drain_trajectories_device()
                    pos, ids = pos.cpu().numpy(), ids.cpu().numpy().astype(np.uint64)
                    out += [(int(i), p.tobytes()) for p, i in zip(pos, ids)]
                else:
                    pos, ids = e.drain_trajectories()
                    out += [(int(i), p.tobytes()) for p, i in zip(pos, ids)]
        return sorted(out), errors

    want, e0 = play(False)
    got, e1 = play(True)
    assert e0 > 0 and e1 == e0 and len(want) > G * 5 and got == want


@pytest.mark.gpu
def test_drain_edge_cases():
    import torch
    L = S.load_library()
    a, b = c4_pair(S.GAME_C4, 32, 24, 24)
    with a, b:
        want_pos, want_ids = a.drain_trajectories()
        N = len(want_pos)
        assert N > 32
        n = C.c_size_t(0)
        # size query: the records stay
        for _ in range(2):
            assert L.spb_drain_trajectories_device(b._h, None, 0, C.byref(n), None) == 0 and n.value == N
        # short capacity: SPB_ERR_ARG, the buffer untouched, the records still there
        short = cuda_full((N - 1, W_C4), 0xAB, torch.uint8)
        torch.cuda.synchronize()
        assert L.spb_drain_trajectories_device(b._h, short.data_ptr(), N - 1, C.byref(n), None) == -1
        assert "too small" in L.spb_last_error(b._h).decode()
        assert bool((short == 0xAB).all())
        # host memory: rejected by name, nothing drained
        host = np.zeros((N, W_C4), np.uint8)
        assert L.spb_drain_trajectories_device(b._h, host.ctypes.data, N, C.byref(n), None) == -1
        assert "buf_dev" in L.spb_last_error(b._h).decode()
        ids_host = np.zeros(N, np.uint64)
        big = cuda_full((N, W_C4), 0, torch.uint8)
        assert L.spb_drain_trajectories_device(b._h, big.data_ptr(), N, C.byref(n), ids_host.ctypes.data) == -1
        assert "game_ids_dev" in L.spb_last_error(b._h).decode() and not ids_host.any()
        assert L.spb_drain_trajectories_device(b._h, None, 0, C.byref(n), None) == 0 and n.value == N
        # a device buffer that is not 8-byte aligned: rejected by name, nothing drained
        odd = cuda_full((N * W_C4 + 8,), 0xEE, torch.uint8)
        torch.cuda.synchronize()
        assert L.spb_drain_trajectories_device(b._h, odd.data_ptr() + 1, N, C.byref(n), None) == -1
        assert "buf_dev is not 8-byte aligned" in L.spb_last_error(b._h).decode() and bool((odd == 0xEE).all())
        assert L.spb_drain_trajectories_device(b._h, big.data_ptr(), N, C.byref(n), odd.data_ptr() + 4) == -1
        assert "game_ids_dev is not 8-byte aligned" in L.spb_last_error(b._h).decode()
        assert L.spb_drain_trajectories_device(b._h, None, 0, C.byref(n), None) == 0 and n.value == N
        # an offset slice of a larger sentinel-filled buffer: only [off, off + n) is written
        off = 5
        ring = cuda_full((N + 11, W_C4), 0xCD, torch.uint8)
        ring_ids = cuda_full((N + 11,), -3, torch.int64)
        pos, ids = b.drain_trajectories_device(out=ring[off:], ids_out=ring_ids[off:])
        assert pos.data_ptr() == ring[off:].data_ptr() and len(pos) == N
        host_ring, host_ids = ring.cpu().numpy(), ring_ids.cpu().numpy()
        assert (host_ring[:off] == 0xCD).all() and (host_ring[off + N:] == 0xCD).all()
        assert (host_ids[:off] == -3).all() and (host_ids[off + N:] == -3).all()
        assert host_ring[off:off + N].tobytes() == want_pos.tobytes() and host_ids[off:off + N].astype(np.uint64).tobytes() == want_ids.tobytes()
        assert L.spb_drain_trajectories_device(b._h, None, 0, C.byref(n), None) == 0 and n.value == 0
    # a chess engine that never played holds 0 records (and allocates nothing)
    with CH.ChessEngine(num_games=4, evaluator=S.EVAL_DET) as e:
        n.value = 9
        assert L.spb_chess_drain_trajectories_device(e._h, None, 0, C.byref(n), None) == 0 and n.value == 0
        pos, ids = e.drain_trajectories_device()
        assert pos.shape == (0, W_CHESS) and len(ids) == 0
        assert L.spb_chess_drain_trajectories_device(e._h, None, 0, None, None) == -1


# ---- GPU: gather -----------------------------------------------------------------------------------------------------

def check_one_rank_gather(a, b, play, width, prefix):
    """a: no communicator (host drain = the reference); b: one-rank communicator, the device gather."""
    import torch
    L = S.load_library()
    gather_dev = getattr(L, prefix + "gather_trajectories_device")
    gather_host = getattr(L, prefix + "gather_trajectories")
    play(a)
    want_pos, want_ids = a.drain_trajectories()
    N = len(want_pos)
    assert N > 0
    b.comm_init(S.comm_unique_id(), 0, 1)
    play(b)
    n = C.c_size_t()
    # size query, then a buffer one record short: the records stay staged on the device
    assert gather_dev(b._h, 0, None, 0, C.byref(n), None) == 0 and n.value == N
    short = cuda_full((N - 1, width), 0x5A, torch.uint8)
    torch.cuda.synchronize()
    assert gather_dev(b._h, 0, short.data_ptr(), N - 1, C.byref(n), None) == 0 and n.value == N
    assert bool((short == 0x5A).all())
    # a host buffer is rejected at delivery, after the collective; the records stay staged
    host = np.zeros((N, width), np.uint8)
    assert gather_dev(b._h, 0, host.ctypes.data, N, C.byref(n), None) == -1 and not host.any()
    # the host form cannot claim it; the records stay
    last_error = L.spb_chess_last_error if prefix == "spb_chess_" else L.spb_last_error
    assert gather_host(b._h, 0, None, 0, C.byref(n), None) == -6
    assert last_error(b._h).decode().endswith("call " + prefix + "gather_trajectories_device")
    pos, ids = b.gather_trajectories_device(0)
    assert records(pos) == want_pos.tobytes() and ids_bytes(ids) == want_ids.tobytes()
    again, _ = b.gather_trajectories_device(0)
    assert len(again) == 0 and len(b.gather_trajectories(0)[0]) == 0 and len(b.drain_trajectories()[0]) == 0
    # a gather staged by the host form cannot be claimed by the device form
    play(a)
    want_pos, want_ids = a.drain_trajectories()
    play(b)
    assert gather_host(b._h, 0, None, 0, C.byref(n), None) == 0 and n.value == len(want_pos) > 0
    assert gather_dev(b._h, 0, None, 0, C.byref(n), None) == -6
    assert last_error(b._h).decode().endswith("call " + prefix + "gather_trajectories")
    pos, ids = b.gather_trajectories(0)
    assert pos.tobytes() == want_pos.tobytes() and ids.tobytes() == want_ids.tobytes()
    assert len(b.gather_trajectories_device(0)[0]) == 0
    b.comm_destroy()


@pytest.mark.gpu
def test_one_rank_device_gather_connect4():
    G = 48
    with S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as a, S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) as b:
        check_one_rank_gather(a, b, lambda e: play_c4(e, G, 24, 24, 3), W_C4, "spb_")


@pytest.mark.gpu
def test_one_rank_device_gather_chess():
    G = len(GATHER_GAMES)
    with CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as a, CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) as b:
        check_one_rank_gather(a, b, play_generation, W_CHESS, "spb_chess_")


def _nccl_device_worker(rank, world, port, out_path):
    import torch
    import torch.distributed as dist
    from selfplay_b200.distributed import comm_init_over_process_group
    from test_chess_selfplay import capped_roots
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
        pos, ids = e.gather_trajectories_device(0)
        pos, ids = pos.cpu().numpy(), ids.cpu().numpy().astype(np.uint64)
        e.comm_destroy()
    if rank == 0:
        np.savez(out_path, sha=hashlib.sha256(pos.tobytes() + ids.tobytes()).hexdigest(), n=len(pos))
    else:
        assert len(pos) == 0
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_ranks_device_gather_what_one_rank_plays(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "two.npz")
    mp.spawn(_nccl_device_worker, args=(2, free_port(), out), nprocs=2, join=True)
    with CH.ChessEngine(num_games=len(GATHER_GAMES), evaluator=S.EVAL_DET) as e:
        play_generation(e)
        pos, ids = e.drain_trajectories()
    got = np.load(out)
    assert int(got["n"]) == len(pos) and str(got["sha"]) == hashlib.sha256(pos.tobytes() + ids.tobytes()).hexdigest()


# ---- GPU: the Connect4 / tic-tac-toe training builder ------------------------------------------------------------------

def random_records(game, n, seed):
    rng = np.random.default_rng(seed)
    pos = np.zeros(n, S.POSITION_DTYPE)
    pos["stones"] = rng.integers(0, 1 << 63, (n, 2), dtype=np.uint64) | rng.integers(0, 2, (n, 2), dtype=np.uint64) << np.uint64(63)
    pos["visit_counts"] = rng.integers(0, 1 << 23, (n, 9), dtype=np.uint32)   # sums past 2^24 round: same order
    pos["visit_counts"][:, 0] += 1
    pos["current_player"] = rng.integers(0, 256, n)                    # high bits set: the host reads & 1
    pos["ply"] = rng.integers(0, 256, n)
    pos["outcome"] = rng.integers(-1, 2, n)
    return pos


def shapes(game, n):
    R, Cc = S.engine.BOARD[game]
    return (n, 3, R, Cc), (n, S.NUM_ACTIONS[game]), (n, 1)


def to_numpy(ts):
    return [t.cpu().numpy() for t in ts]


@pytest.fixture(scope="module")
def engines():
    es = {g: S.Engine(game=g, num_games=1, evaluator=S.EVAL_DET) for g in (S.GAME_C4, S.GAME_TTT)}
    yield es
    for e in es.values():
        e.close()


@pytest.fixture(scope="module")
def selfplay_c4():
    with S.Engine(game=S.GAME_C4, num_games=256, evaluator=S.EVAL_DET) as e:
        play_c4(e, 256, 30, 24, 11)
        pos, _ = e.drain_trajectories()
    assert len(pos) > 1000
    return pos


@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
def test_device_builder_equals_host_builder_on_random_records(engines, game):
    import torch
    e = engines[game]
    recs = random_records(game, 3001, seed=game)
    want = S.positions_to_training(game, recs)
    assert_bit_identical(to_numpy(S.positions_to_training_device(e, recs)), want)
    dev = torch.from_numpy(recs.view(np.uint8).reshape(len(recs), -1)).cuda()
    for n in (0, 1, 2, 3, 5, 333, 1027):
        got = to_numpy(S.positions_to_training_device(e, dev[:n]))
        assert [g.shape for g in got] == list(shapes(game, n))
        assert_bit_identical(got, [w[:n] for w in want])
    rng = np.random.default_rng(2)
    idx = rng.integers(0, len(recs), 4099)
    idx[:17] = idx[17]                                                 # repeats
    for ix in (idx, torch.from_numpy(idx.astype(np.int64)).cuda(), torch.from_numpy(idx.astype(np.uint64)).cuda()):
        assert_bit_identical(to_numpy(S.positions_to_training_device(e, dev, ix)), S.positions_to_training(game, recs[idx]))
    small = rng.integers(0, 5, 77)                                     # with indices n may exceed n_positions
    assert_bit_identical(to_numpy(S.positions_to_training_device(e, recs[:5], small)), S.positions_to_training(game, recs[:5][small]))


@pytest.mark.gpu
def test_device_builder_equals_host_builder_on_self_play_records(engines, selfplay_c4):
    want = S.positions_to_training(S.GAME_C4, selfplay_c4)
    assert_bit_identical(to_numpy(S.positions_to_training_device(engines[S.GAME_C4], selfplay_c4)), want)


def raw_outputs(game, n, offset_floats=0, fill=-7.5):
    import torch
    widths = [int(np.prod(s[1:])) for s in shapes(game, 1)]
    bufs = [torch.full((n * k + offset_floats,), fill, dtype=torch.float32, device="cuda") for k in widths]
    return bufs, [b.data_ptr() + 4 * offset_floats for b in bufs]


def raw_call(e, pos_t, n_positions, idx_ptr, n, ptrs):
    import torch
    torch.cuda.synchronize()
    return e._L.spb_positions_to_training_device(e._h, pos_t.data_ptr(), n_positions, idx_ptr, n, *ptrs)


@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_C4, S.GAME_TTT])
def test_unaligned_null_outputs_and_zero_count_rows(engines, game):
    import torch
    e = engines[game]
    recs = random_records(game, 301, seed=5)
    recs["visit_counts"][[3, 200]] = 0                                  # 0 / 0: NaN on both sides
    want = S.positions_to_training(game, recs)
    assert np.isnan(want[1][3]).all() and np.isnan(want[1][200]).all()
    pos_t = torch.from_numpy(recs.view(np.uint8).reshape(len(recs), -1)).cuda()
    n = len(recs)
    for off in (1, 2, 3):                                              # 4-byte aligned only: scalar head, float4 body, tail
        bufs, ptrs = raw_outputs(game, n, offset_floats=off)
        assert raw_call(e, pos_t, n, None, n, ptrs) == 0
        got = [b.cpu().numpy()[off:].reshape(w.shape) for b, w in zip(bufs, want)]
        assert all((b.cpu().numpy()[:off] == np.float32(-7.5)).all() for b in bufs)
        assert_bit_identical(got, want, nan_rows=(3, 200))
    for k in range(3):                                                 # each output NULL in turn
        bufs, ptrs = raw_outputs(game, n)
        ptrs[k] = None
        assert raw_call(e, pos_t, n, None, n, ptrs) == 0
        for j in range(3):
            host = bufs[j].cpu().numpy()
            if j == k:
                assert (host == np.float32(-7.5)).all()
            else:
                assert_bit_identical([host.reshape(want[j].shape)], [want[j]], nan_rows=(3, 200) if j == 1 else ())
    assert raw_call(e, pos_t, n, None, n, [None, None, None]) == 0


@pytest.mark.gpu
def test_bad_index_and_host_pointers_write_nothing(engines):
    import torch
    e = engines[S.GAME_C4]
    L = S.load_library()
    recs = random_records(S.GAME_C4, 40, seed=9)
    pos_t = torch.from_numpy(recs.view(np.uint8).reshape(40, -1)).cuda()
    idx = np.arange(40, dtype=np.int64)
    idx[[6, 30]] = 40                                                  # index >= n_positions
    idx_t = torch.from_numpy(idx).cuda()
    bufs, ptrs = raw_outputs(S.GAME_C4, 40)
    assert raw_call(e, pos_t, 40, idx_t.data_ptr(), 40, ptrs) == -1
    assert "row 6" in L.spb_last_error(e._h).decode()
    with pytest.raises(S.EngineError) as ei:
        S.positions_to_training_device(e, recs, idx)
    assert ei.value.code == -1
    assert raw_call(e, pos_t, 40, None, 41, ptrs) == -1                # n > n_positions without indices
    host_out = np.zeros(40 * 126, np.float32)
    assert L.spb_positions_to_training_device(e._h, recs.ctypes.data, 40, None, 40, *ptrs) == -1
    assert "positions" in L.spb_last_error(e._h).decode()
    assert raw_call(e, pos_t, 40, None, 40, [host_out.ctypes.data, ptrs[1], ptrs[2]]) == -1
    assert "encodings" in L.spb_last_error(e._h).decode()
    assert raw_call(e, pos_t, 40, idx.ctypes.data, 40, ptrs) == -1
    assert "indices" in L.spb_last_error(e._h).decode()
    assert not host_out.any()
    # misaligned records, indices or outputs: rejected by name, not a fault on the device
    raw = torch.zeros(40 * 56 + 8, dtype=torch.uint8, device="cuda")
    raw[1:1 + 40 * 56] = pos_t.reshape(-1)
    torch.cuda.synchronize()
    assert e._L.spb_positions_to_training_device(e._h, raw.data_ptr() + 1, 40, None, 40, *ptrs) == -1
    assert "positions is not 8-byte aligned" in L.spb_last_error(e._h).decode()
    idx_raw = torch.zeros(41, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    assert raw_call(e, pos_t, 40, idx_raw.data_ptr() + 4, 40, ptrs) == -1
    assert "indices is not 8-byte aligned" in L.spb_last_error(e._h).decode()
    assert raw_call(e, pos_t, 40, None, 40, [ptrs[0], ptrs[1] + 2, ptrs[2]]) == -1
    assert "policies is not 4-byte aligned" in L.spb_last_error(e._h).decode()
    for b in bufs:
        assert (b.cpu().numpy() == np.float32(-7.5)).all()


@pytest.mark.gpu
def test_chess_builder_rejects_misaligned_pointers():
    import torch
    L = S.load_library()
    with CH.ChessEngine(num_games=1, evaluator=S.EVAL_DET) as e:
        raw = torch.zeros(4 * W_CHESS + 8, dtype=torch.uint8, device="cuda")
        out = torch.full((4 * 19 * 64 + 1,), -7.5, dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        assert L.spb_chess_positions_to_training_device(e._h, raw.data_ptr() + 4, 4, None, 4, None, None, None) == -1
        assert "positions is not 8-byte aligned" in L.spb_chess_last_error(e._h).decode()
        assert L.spb_chess_positions_to_training_device(e._h, raw.data_ptr(), 4, None, 4, out.data_ptr() + 1, None, None) == -1
        assert "encodings is not 4-byte aligned" in L.spb_chess_last_error(e._h).decode()
        assert bool((out == -7.5).all())


@pytest.mark.gpu
def test_device_drain_then_device_builder_equals_host_drain_then_host_builder():
    a, b = c4_pair(S.GAME_C4, 128, 30, 16)
    with a, b:
        pos_h, _ = a.drain_trajectories()
        pos_d, _ = b.drain_trajectories_device()
        want = S.positions_to_training(S.GAME_C4, pos_h)
        got = to_numpy(S.positions_to_training_device(b, pos_d))
    assert len(pos_h) > 128
    assert_bit_identical(got, want)
