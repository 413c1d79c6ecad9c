"""spb_load_weights_device / spb_chess_load_weights_device and spb_broadcast_weights (csrc/weights_device.cu, gather.cu).

The device path folds BatchNorm and packs the weight image on the GPU from a learner's device tensors.  It must write the
bytes the safetensors path writes, so every comparison here is bit for bit against an engine loaded from a checkpoint of
the same tensors: predict at 4,096 positions (also through the SIMT kernel, the only reader of the SIMT section), and the
roots of a network search.  The sensitivity test shows such a comparison sees one weight changed by one part in 128.
"""
import ctypes as C
import os
import re
import socket

import numpy as np
import pytest
import torch

import selfplay_b200 as S
from helpers import random_states
from oracle import torch_net
from weight_tables import (CHESS_SCHEMES, SCHEMES, chess_named_explicit, chess_named_tch, named_explicit, named_tch, on_device,
                           write_safetensors)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = open(os.path.join(ROOT, "include", "selfplay_b200.h")).read()
N = 4096


# ---- CPU -----------------------------------------------------------------------------------------------------------

def test_named_lists_write_the_oracle_checkpoints():
    """The (name, tensor) lists are the tensors, names and order of torch_net's writers: the same bytes."""
    for game in (S.GAME_TTT, S.GAME_C4):
        net = torch_net.make_net(game, seed=3)
        assert write_safetensors(named_explicit(net)) == torch_net.to_safetensors_explicit(net)
        assert write_safetensors(named_tch(net)) == torch_net.to_safetensors_tch(net)
        assert write_safetensors(named_tch(net, shuffle_seed=5)) == torch_net.to_safetensors_tch(net, shuffle_seed=5)
        order = ("running_mean", "running_var", "weight", "bias")
        assert write_safetensors(named_tch(net, bn_order=order)) == torch_net.to_safetensors_tch(net, bn_order=order)
    net = torch_net.make_chess_net(seed=0, blocks=1)
    assert write_safetensors(chess_named_explicit(net)) == torch_net.chess_to_safetensors_explicit(net)
    assert write_safetensors(chess_named_tch(net, shuffle_seed=3)) == torch_net.chess_to_safetensors_tch(net, shuffle_seed=3)


def test_spb_tensor_layout_and_dtype_constants_agree_across_header_ctypes_and_rust():
    body = re.sub(r"/\*.*?\*/", "", re.search(r"typedef struct spb_tensor \{(.*?)\} spb_tensor;", HEADER, re.S).group(1), flags=re.S)
    c_fields = re.findall(r"(\w+\*?)\s+(\w+)(?:\[(\d+)\])?;", body)
    assert [f[1] for f in c_fields] == ["name", "data", "dtype", "ndim", "shape"]
    assert [f for f, _ in S.Tensor._fields_] == ["name", "data", "dtype", "ndim", "shape"]
    assert C.sizeof(S.Tensor) == 56 and S.Tensor.shape.offset == 24 and S.Tensor.dtype.offset == 16
    rust = open(os.path.join(ROOT, "rust", "selfplay-b200-sys", "src", "lib.rs")).read()
    rbody = re.search(r"pub struct spb_tensor \{(.*?)\n\}", rust, re.S).group(1)
    assert re.findall(r"pub (\w+):", rbody) == ["name", "data", "dtype", "ndim", "shape"]
    assert "pub shape: [i64; 4]," in rbody and "pub dtype: i32," in rbody and "pub ndim: i32," in rbody
    defs = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(SPB_DTYPE_[A-Z0-9]+)\s+(\d+)", HEADER)}
    assert defs == {"SPB_DTYPE_F32": S.DTYPE_F32, "SPB_DTYPE_BF16": S.DTYPE_BF16, "SPB_DTYPE_F64": S.DTYPE_F64, "SPB_DTYPE_F16": S.DTYPE_F16}
    for name, v in defs.items():
        assert re.search(r"pub const %s: i32 = %d;" % (name, v), rust), name


def test_new_entry_points_reject_a_null_engine():
    L = S.load_library()
    assert L.spb_load_weights_device(None, None, 0) == -1 and L.spb_chess_load_weights_device(None, None, 0) == -1
    assert L.spb_broadcast_weights(None, 0) == -1 and L.spb_chess_broadcast_weights(None, 0) == -1


# ---- GPU: Connect4 / tic-tac-toe -----------------------------------------------------------------------------------

NETS = {"fresh": dict(seed=3), "trained": dict(seed=4, trained_like=True)}


def small_predict(e, states):
    pol, val, lg = e.predict(states, want_logits=True)
    return pol, val, lg


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def small_engines():
    """Per game: (blob engine, device engine) for the tcgen05 kernel and for the SIMT kernel, and 4,096 positions."""
    out = {}
    for game in (S.GAME_TTT, S.GAME_C4):
        out[game] = dict(states=random_states(game, N, seed=11, include_terminal=False),
                         engines=[(S.Engine(game=game, num_games=64, flags=f), S.Engine(game=game, num_games=64, flags=f))
                                  for f in (0, S.FLAG_EVAL_SIMT)])
    yield out
    for v in out.values():
        for a, b in v["engines"]:
            a.close()
            b.close()


@pytest.mark.gpu
@pytest.mark.parametrize("game", [S.GAME_TTT, S.GAME_C4], ids=["ttt", "c4"])
@pytest.mark.parametrize("kind", list(NETS))
@pytest.mark.parametrize("scheme", list(SCHEMES))
def test_device_load_predicts_bit_identically_to_the_blob(small_engines, game, kind, scheme):
    net = torch_net.make_net(game, **NETS[kind])
    named = SCHEMES[scheme](net)
    for blob_e, dev_e in small_engines[game]["engines"]:
        blob_e.load_weights(write_safetensors(named))
        dev_e.load_weights_device(on_device(named))
        states = small_engines[game]["states"]
        assert same(small_predict(blob_e, states), small_predict(dev_e, states))


def search_roots(e, roots, sims):
    e.reset_games(roots)
    e.search(sims)
    return e.root_children_all()


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [S.FLAG_FORCE_SPLIT, S.FLAG_LOCKSTEP], ids=["async", "lockstep"])
@pytest.mark.parametrize("kind", list(NETS))
def test_device_load_searches_like_the_blob_connect4(flags, kind):
    net = torch_net.make_net(S.GAME_C4, **NETS[kind])
    roots = random_states(S.GAME_C4, 256, seed=2, include_terminal=False)
    with S.Engine(game=S.GAME_C4, num_games=256, flags=flags) as a, S.Engine(game=S.GAME_C4, num_games=256, flags=flags) as b:
        a.load_weights(write_safetensors(named_tch(net)))
        b.load_weights_device(on_device(named_tch(net)))
        assert same(search_roots(a, roots, 96), search_roots(b, roots, 96))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float64], ids=["bf16", "f64"])
def test_bf16_and_f64_sources_equal_the_blob_of_that_dtype(small_engines, dtype):
    net = torch_net.make_net(S.GAME_C4, trained_like=True, seed=4)
    named = named_explicit(net)
    blob_e, dev_e = small_engines[S.GAME_C4]["engines"][0]
    blob_e.load_weights(write_safetensors(named, dtype))
    dev_e.load_weights_device(on_device(named, dtype=dtype))
    states = small_engines[S.GAME_C4]["states"]
    want = small_predict(blob_e, states)
    assert same(want, small_predict(dev_e, states))
    if dtype == torch.bfloat16:                                            # the dtype reached the image (f64 holds the f32 values)
        blob_e.load_weights(write_safetensors(named))
        assert not same(want, small_predict(blob_e, states))


@pytest.mark.gpu
def test_one_weight_changed_in_the_table_changes_the_outputs(small_engines):
    net = torch_net.make_net(S.GAME_C4, trained_like=True, seed=4)
    named = on_device(named_explicit(net))
    blob_e, dev_e = small_engines[S.GAME_C4]["engines"][0]
    blob_e.load_weights(write_safetensors(named))
    w = dict(named)["conv4.weight"]                                        # block 2, first conv
    w[5, 7, 1, 1] *= 1 + 2 ** -7
    dev_e.load_weights_device(named)
    states = small_engines[S.GAME_C4]["states"]
    assert not same(small_predict(blob_e, states), small_predict(dev_e, states))


@pytest.mark.gpu
def test_hot_swap_and_sources_are_not_read_after_the_call():
    a_net, b_net = torch_net.make_net(S.GAME_C4, seed=3), torch_net.make_net(S.GAME_C4, seed=8, trained_like=True)
    roots = random_states(S.GAME_C4, 128, seed=4, include_terminal=False)
    states = random_states(S.GAME_C4, N, seed=12, include_terminal=False)
    with S.Engine(game=S.GAME_C4, num_games=128) as e, S.Engine(game=S.GAME_C4, num_games=128) as fresh:
        e.load_weights_device(on_device(named_tch(a_net)))
        search_roots(e, roots, 64)
        b = on_device(named_tch(b_net))
        e.load_weights_device(b)
        fresh.load_weights(write_safetensors(named_tch(b_net)))
        want = small_predict(fresh, states)
        assert same(want, small_predict(e, states))
        assert same(search_roots(fresh, roots, 64), search_roots(e, roots, 64))
        for _, t in b:
            t.normal_()
        torch.cuda.synchronize()
        assert same(want, small_predict(e, states))


def raw_table(named):
    table, n, names = S.tensor_table(named, 0)
    return table, n, names


@pytest.mark.gpu
def test_bad_tables_return_their_code_and_keep_the_loaded_net():
    net = torch_net.make_net(S.GAME_C4, seed=3)
    states = random_states(S.GAME_C4, 512, seed=13, include_terminal=False)
    L = S.load_library()
    with S.Engine(game=S.GAME_C4, num_games=64) as e:
        good = on_device(named_explicit(net))
        e.load_weights_device(good)
        want = small_predict(e, states)

        def expect(rc_want, table, n, blob=None):
            rc = L.spb_load_weights_device(e._h, table, n)
            msg = L.spb_last_error(e._h).decode()
            assert rc == rc_want, msg
            if blob is not None:                                          # the checkpoint of the same tensors is refused alike
                rc_b, msg_b = S.check_weights(S.GAME_C4, blob)
                assert rc_b == -5 and msg.endswith(msg_b), (msg, msg_b)
            assert same(want, small_predict(e, states))
            return msg

        missing = [x for x in good if x[0] != "bn3.running_var"]
        expect(-5, *raw_table(missing)[:2], blob=write_safetensors(missing))
        wrong = [(n, t.reshape(-1) if n == "conv2.weight" else t) for n, t in good]
        expect(-5, *raw_table(wrong)[:2], blob=write_safetensors(wrong))
        tch = on_device(named_tch(net))
        extra = tch + [("weight__999", torch.zeros(4, 4, 3, 3, device="cuda"))]
        assert "census" in expect(-5, *raw_table(extra)[:2], blob=write_safetensors(extra))
        half = [(n, t.half() if n == "conv1.bias" else t) for n, t in good]
        assert expect(-5, *raw_table(half)[:2]).endswith("unsupported dtype F16 for conv1.bias (expected F32)")
        table, n, keep = raw_table(good)
        table[3].ndim = 5
        expect(-1, table, n)
        table, n, keep = raw_table(good)
        table[7].name = None
        expect(-1, table, n)
        expect(-1, None, 0)
        host = torch.zeros(64, 64, 3, 3)
        table, n, keep = raw_table(good)
        i = [k for k in range(n) if table[k].name == b"conv1.weight"][0]
        table[i].data = host.data_ptr()
        assert "not device memory" in expect(-1, table, n)
        table, n, keep = raw_table(good)
        table[i].data = table[i].data + 2
        assert "aligned" in expect(-1, table, n)
        if torch.cuda.device_count() > 1:
            other = torch.zeros(64, 64, 3, 3, device="cuda:1")
            table, n, keep = raw_table(good)
            table[i].data = other.data_ptr()
            expect(-1, table, n)
        with pytest.raises(ValueError):
            e.load_weights_device([(n_, t.t() if t.dim() == 2 else t) for n_, t in good])   # not contiguous


# ---- GPU: chess ----------------------------------------------------------------------------------------------------

CHESS_NETS = {"seed0": dict(seed=0), "calibrated": dict(seed=0, calibrated=True)}


@pytest.fixture(scope="module")
def chess_engines():
    from test_net_numerics import distinct_positions
    a, b = S.ChessEngine(num_games=N), S.ChessEngine(num_games=N)
    st, hist = distinct_positions(a, N)
    yield a, b, st, hist
    a.close()
    b.close()


def chess_predict(e, st, hist):
    _, v, lg = e.predict(st, hist, want_logits=True)
    return v, lg


@pytest.mark.gpu
@pytest.mark.parametrize("kind", list(CHESS_NETS))
@pytest.mark.parametrize("scheme", list(CHESS_SCHEMES))
def test_chess_device_load_predicts_bit_identically_to_the_blob(chess_engines, kind, scheme):
    a, b, st, hist = chess_engines
    named = CHESS_SCHEMES[scheme](torch_net.make_chess_net(**CHESS_NETS[kind]))
    a.load_weights(write_safetensors(named))
    b.load_weights_device(on_device(named))
    assert same(chess_predict(a, st, hist), chess_predict(b, st, hist))


@pytest.mark.gpu
def test_chess_device_load_searches_like_the_blob(chess_engines):
    _, _, st, hist = chess_engines
    named = chess_named_tch(torch_net.make_chess_net(seed=0, calibrated=True))
    out = []
    for load in (lambda e: e.load_weights(write_safetensors(named)), lambda e: e.load_weights_device(on_device(named))):
        with S.ChessEngine(num_games=256) as e:                            # two-half pipeline
            load(e)
            e.reset_games(st[:256], hist[:256])
            e.search(16)
            out.append(e.root_children_all() + tuple(e.node_stats(i, 0)["value_sum"] for i in range(0, 256, 5)))
    assert all(np.array_equal(x, y) for x, y in zip(*out))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float64], ids=["bf16", "f64"])
def test_chess_bf16_and_f64_sources_equal_the_blob_of_that_dtype(chess_engines, dtype):
    a, b, st, hist = chess_engines
    named = chess_named_explicit(torch_net.make_chess_net(seed=0, calibrated=True))
    a.load_weights(write_safetensors(named, dtype))
    b.load_weights_device(on_device(named, dtype=dtype))
    assert same(chess_predict(a, st[:1024], hist[:1024]), chess_predict(b, st[:1024], hist[:1024]))


@pytest.mark.gpu
def test_chess_one_weight_changed_in_the_table_changes_the_outputs(chess_engines):
    a, b, st, hist = chess_engines
    named = on_device(chess_named_explicit(torch_net.make_chess_net(seed=0, calibrated=True)))
    a.load_weights(write_safetensors(named))
    dict(named)["conv10.weight"][17, 200, 1, 1] *= 1 + 2 ** -7             # block 5, second conv
    b.load_weights_device(named)
    assert not same(chess_predict(a, st, hist), chess_predict(b, st, hist))


@pytest.mark.gpu
def test_chess_bad_tables_keep_the_loaded_net(chess_engines):
    _, b, st, hist = chess_engines
    L = S.load_library()
    good = on_device(chess_named_explicit(torch_net.make_chess_net(seed=0)))
    b.load_weights_device(good)
    want = chess_predict(b, st[:256], hist[:256])
    missing = [x for x in good if x[0] != "value_fc2.bias"]
    table, n, keep = S.tensor_table(missing, 0)
    assert L.spb_chess_load_weights_device(b._h, table, n) == -5
    assert L.spb_chess_last_error(b._h).decode().endswith(S.chess.check_weights(write_safetensors(missing))[1])
    table, n, keep = S.tensor_table(good, 0)
    table[0].data = table[0].data + 2
    assert L.spb_chess_load_weights_device(b._h, table, n) == -1
    assert same(want, chess_predict(b, st[:256], hist[:256]))


# ---- GPU: broadcast ------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_one_rank_broadcast_keeps_outputs_and_checks_its_arguments(small_engines, chess_engines):
    net = torch_net.make_net(S.GAME_C4, seed=3)
    states = small_engines[S.GAME_C4]["states"]
    with S.Engine(game=S.GAME_C4, num_games=64) as e:
        with pytest.raises(S.EngineError) as ei:
            e.broadcast_weights(0)
        assert ei.value.code == -6                                         # no communicator
        e.comm_init(S.comm_unique_id(), 0, 1)
        with pytest.raises(S.EngineError) as ei:
            e.broadcast_weights(0)
        assert ei.value.code == -6 and "no weights" in str(ei.value)       # the root has none
        e.load_weights_device(on_device(named_tch(net)))
        want = small_predict(e, states)
        e.broadcast_weights(0)
        assert same(want, small_predict(e, states))
        with pytest.raises(S.EngineError) as ei:
            e.broadcast_weights(1)
        assert ei.value.code == -1
        e.comm_destroy()
    _, b, st, hist = chess_engines
    b.load_weights_device(on_device(chess_named_tch(torch_net.make_chess_net(seed=0, calibrated=True))))
    want = chess_predict(b, st, hist)
    with pytest.raises(S.EngineError) as ei:
        b.broadcast_weights(0)
    assert ei.value.code == -6
    b.comm_init(S.comm_unique_id(), 0, 1)
    b.broadcast_weights(0)
    assert same(want, chess_predict(b, st, hist))
    with pytest.raises(S.EngineError) as ei:
        b.broadcast_weights(-1)
    assert ei.value.code == -1
    b.comm_destroy()


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _broadcast_worker(rank, world, port, out_path):
    import torch.distributed as dist
    from selfplay_b200.distributed import comm_init_over_process_group
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)       # carries only the 128-byte id
    states = random_states(S.GAME_C4, 1024, seed=11, include_terminal=False)
    c4 = torch_net.make_net(S.GAME_C4, seed=4, trained_like=True)
    codes = []
    with S.Engine(game=S.GAME_C4, num_games=64, device=rank) as e:
        comm_init_over_process_group(e, rank, world)
        for _ in range(2):                                                 # a root with no weights fails on both ranks
            try:
                e.broadcast_weights(0)
                codes.append(0)
            except S.EngineError as x:
                codes.append(x.code)
            if rank == 0:
                e.load_weights_device(on_device(named_tch(c4), device=rank))
        c4_out = small_predict(e, states)
        e.comm_destroy()
    with S.Engine(game=S.GAME_C4 if rank == 0 else S.GAME_TTT, num_games=64, device=rank) as e:   # a game mix fails on both
        comm_init_over_process_group(e, rank, world)
        if rank == 0:
            e.load_weights(write_safetensors(named_tch(c4)))
        try:
            e.broadcast_weights(0)
            codes.append(0)
        except S.EngineError as x:
            codes.append(x.code)
        e.comm_destroy()
    ch = torch_net.make_chess_net(seed=0, calibrated=True)
    with S.ChessEngine(num_games=256, device=rank) as e:
        from test_net_numerics import distinct_positions
        st, hist = distinct_positions(e, 256)
        comm_init_over_process_group(e, rank, world)
        if rank == 0:
            e.load_weights_device(on_device(chess_named_tch(ch), device=rank))
        e.broadcast_weights(0)
        ch_out = chess_predict(e, st, hist)
        e.comm_destroy()
    np.savez(out_path % rank, *c4_out, *ch_out, codes=np.array(codes))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_ranks_broadcast_what_the_root_loaded(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    out = str(tmp_path / "rank%d.npz")
    mp.spawn(_broadcast_worker, args=(2, free_port(), out), nprocs=2, join=True)
    r0, r1 = np.load(out % 0), np.load(out % 1)
    assert list(r0["codes"]) == list(r1["codes"]) == [-6, 0, -1]
    for k in r0.files:
        if k != "codes":
            assert np.array_equal(r0[k], r1[k]), k
