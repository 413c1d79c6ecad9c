"""Weight hand-off: spb_load_weights from an in-memory safetensors blob (parse, fold and pack on one CPU thread, then a
synchronous copy) against spb_load_weights_device from the learner's CUDA tensors (fold and pack on the GPU), for the
Connect4 4x64 net and the chess 10x256 net; and spb_broadcast_weights when two GPUs exist.  Writes one JSON file.

Both loads are checked to give bit-identical predictions.  Times are wall clock around calls that return synchronised:
median, min and max of --reps rounds after one untimed warm-up round (the first load allocates the image and loads the
kernels).  The blob is built once, outside the timed region, as a learner that already holds the checkpoint bytes would.

usage: python tools/weight_handoff_bench.py --out profiles/r08_weight_handoff_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import selfplay_b200 as S  # noqa: E402
from oracle import torch_net  # noqa: E402
from weight_tables import chess_named_tch, named_tch, on_device, write_safetensors  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return name, power


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts), "reps": reps}


def case(name, make_engine, named, blob, predict, reps):
    a, b = make_engine(), make_engine()
    dev = on_device(named)
    host = timed(lambda: a.load_weights(blob), reps)
    device = timed(lambda: b.load_weights_device(dev), reps)
    equal = all(np.array_equal(x, y) for x, y in zip(predict(a), predict(b)))
    params = sum(t.numel() for _, t in named)
    out = {"net": name, "tensors": len(named), "f32_parameters": params, "f32_bytes_read": params * 4, "blob_bytes": len(blob),
           "spb_load_weights": host, "spb_load_weights_device": device, "speedup_median": host["median_ms"] / device["median_ms"],
           "predictions_bit_identical": equal}
    a.close()
    b.close()
    return out


def _bcast_worker(rank, world, port, reps, out_path):
    import torch.distributed as dist
    from selfplay_b200.distributed import comm_init_over_process_group
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    res = {}
    for name, eng, named in (("connect4", lambda: S.Engine(game=S.GAME_C4, num_games=4096, device=rank), named_tch(torch_net.make_net(1, seed=4))),
                             ("chess", lambda: S.ChessEngine(num_games=4096, device=rank), chess_named_tch(torch_net.make_chess_net(seed=0)))):
        e = eng()
        comm_init_over_process_group(e, rank, world)
        if rank == 0:
            e.load_weights_device(on_device(named, device=rank))
        res[name] = timed(lambda: (dist.barrier(), e.broadcast_weights(0)), reps)
        e.comm_destroy()
        e.close()
    if rank == 0:
        with open(out_path, "w") as f:
            json.dump(res, f)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    name, power = gpu_info()
    from helpers import random_states
    from test_net_numerics import distinct_positions
    c4_states = random_states(S.GAME_C4, 4096, seed=11, include_terminal=False)
    c4_named = named_tch(torch_net.make_net(S.GAME_C4, seed=4, trained_like=True))
    res = {"gpu": name, "power_limit": power, "cases": []}
    res["cases"].append(case("connect4 4x64", lambda: S.Engine(game=S.GAME_C4, num_games=4096), c4_named, write_safetensors(c4_named),
                             lambda e: e.predict(c4_states, want_logits=True), a.reps))
    ch_named = chess_named_tch(torch_net.make_chess_net(seed=0, calibrated=True))
    with S.ChessEngine(num_games=4096) as e:
        st, hist = distinct_positions(e, 4096)
    res["cases"].append(case("chess 10x256", lambda: S.ChessEngine(num_games=4096), ch_named, write_safetensors(ch_named),
                             lambda e: e.predict(st, hist, want_logits=True)[1:], a.reps))
    if torch.cuda.device_count() >= 2:
        import socket
        import tempfile
        import torch.multiprocessing as mp
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        path = os.path.join(tempfile.mkdtemp(), "bcast.json")
        mp.spawn(_bcast_worker, args=(2, port, a.reps, path), nprocs=2, join=True)
        res["broadcast_2_ranks"] = json.load(open(path))
    else:
        res["broadcast_2_ranks"] = "not measured: one GPU"
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
