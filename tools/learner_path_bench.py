"""Learner hand-off: host drain / gather + H2D copy into a CUDA tensor (the path INTEGRATION §7 documented before the device
forms) against spb_drain_trajectories_device / spb_gather_trajectories_device straight into the tensor, for Connect4 and
chess at 4,096 games; the Connect4 / tic-tac-toe device training builder against the host builder; one bench.py line per
game to show the search path is unchanged.  Runs on one B200; writes one JSON file.

Both engines of a pair play the same plies (EvalDet, 2 simulations, greedy moves, restarts), so their output buffers hold the
same records: the drain cost does not depend on the evaluator.  Every drain and gather is checked byte for byte against the
other path.  Times are wall clock around calls that return synchronised: median, min and max of --reps rounds after one untimed
warm-up round (the first device call grows the engine's stage and loads its kernels).

usage: python tools/learner_path_bench.py --out profiles/r06_learner_path_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import selfplay_b200 as S  # noqa: E402

CH = S.chess
HBM_GBPS = 6545.0          # DESIGN §4.1: the HBM rate measured on this card


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return name, power


def c4_pair(G):
    from helpers import synthetic_roots
    roots = synthetic_roots(S.GAME_C4, G, start=0)
    es = [S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_DET) for _ in range(2)]

    def play(e, plies):
        for _ in range(plies):
            e.search(2)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)
    for e in es:
        e.reset_games(roots)
    return es, play


def chess_pair(G):
    from oracle import pychess as P
    from test_chess_selfplay import capped_roots
    games = [P.Game(), P.Game(P.KIWIPETE)] * (G // 2)
    st, hist = capped_roots(games, 506)                                # every game ends after 7 records, then restarts
    es = [CH.ChessEngine(num_games=G, evaluator=S.EVAL_DET) for _ in range(2)]

    def play(e, plies):
        for _ in range(plies):
            e.search(2)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist)
    for e in es:
        e.reset_games(st, hist)
    return es, play


def timed(f):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = f()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def hand_off(name, pair, G, plies, reps, width):
    """Drain and one-rank gather, host path vs device path, on identically played engines."""
    import torch
    (a, b), play = pair(G)
    out = {"games": G, "plies_per_round": plies, "record_bytes": width}
    a.comm_init(S.comm_unique_id(), 0, 1)
    b.comm_init(S.comm_unique_id(), 0, 1)
    for form in ("drain", "gather"):
        host_s, dev_s, counts = [], [], []
        for rnd in range(reps + 1):                                    # round 0 warms up: stage growth, first launches
            play(a, plies)
            play(b, plies)
            host_fn = a.drain_trajectories if form == "drain" else a.gather_trajectories
            dev_fn = b.drain_trajectories_device if form == "drain" else b.gather_trajectories_device

            def host_path():
                pos, ids = host_fn() if form == "drain" else host_fn(0)
                k = len(pos)
                ra = torch.empty((k, width), dtype=torch.uint8, device="cuda")
                ia = torch.empty(k, dtype=torch.int64, device="cuda")
                ra.copy_(torch.from_numpy(pos.view(np.uint8).reshape(k, width)))
                ia.copy_(torch.from_numpy(ids.view(np.int64)))
                return ra, ia
            th, (ra, ia) = timed(host_path)
            k = len(ra)
            # the replay slice of the device path exists before the call, as a learner's ring does
            replay_b = torch.empty((k, width), dtype=torch.uint8, device="cuda")
            ids_b = torch.empty(k, dtype=torch.int64, device="cuda")
            td, (rb, ib) = timed(lambda: dev_fn(out=replay_b, ids_out=ids_b) if form == "drain" else dev_fn(0, out=replay_b, ids_out=ids_b))
            assert len(rb) == k and torch.equal(ra, rb) and torch.equal(ia, ib), (name, form, "bytes differ")
            if rnd == 0:
                continue
            host_s.append(th)
            dev_s.append(td)
            counts.append(k)
        n = int(statistics.median(counts))
        th, td = statistics.median(host_s), statistics.median(dev_s)
        moved = 2.0 * n * (width + 8)                                  # bytes read + written by the device ordering
        out[form] = {"records": counts, "host_ms": [x * 1e3 for x in host_s], "device_ms": [x * 1e3 for x in dev_s],
                     "host_ms_median": th * 1e3, "device_ms_median": td * 1e3, "device_ms_min": min(dev_s) * 1e3,
                     "device_ms_max": max(dev_s) * 1e3, "speedup": th / td,
                     "device_GBps": moved / td / 1e9, "device_share_of_hbm": moved / td / 1e9 / HBM_GBPS,
                     "bytes_equal": True}
        print(name, form, json.dumps(out[form]), flush=True)
    for e in (a, b):
        e.comm_destroy()
        e.close()
    return out


def builder(reps):
    import torch
    from test_device_records import random_records
    with S.Engine(game=S.GAME_C4, num_games=1, evaluator=S.EVAL_DET) as e:
        n_buf = 1 << 20
        recs = random_records(S.GAME_C4, n_buf, seed=1)
        dev = torch.from_numpy(recs.view(np.uint8).reshape(n_buf, -1)).cuda()
        row_out = (126 + 7 + 1) * 4
        res = {"buffer_records": n_buf}
        rng = np.random.default_rng(0)
        for rows, use_idx in ((4096, True), (262144, False)):
            idx = torch.from_numpy(rng.integers(0, n_buf, rows).astype(np.int64)).cuda() if use_idx else None
            src = dev if use_idx else dev[:rows]
            enc = torch.empty((rows, 3, 6, 7), dtype=torch.float32, device="cuda")
            pol = torch.empty((rows, 7), dtype=torch.float32, device="cuda")
            val = torch.empty((rows, 1), dtype=torch.float32, device="cuda")
            args = (e._h, src.data_ptr(), len(src), None if idx is None else idx.data_ptr(), rows, enc.data_ptr(), pol.data_ptr(), val.data_ptr())
            for _ in range(5):
                assert e._L.spb_positions_to_training_device(*args) == 0
            iters = 200 if rows == 4096 else 50
            times = []
            for _ in range(reps):
                t, _ = timed(lambda: [e._L.spb_positions_to_training_device(*args) for _ in range(iters)])
                times.append(t / iters)
            t = statistics.median(times)
            moved = rows * (row_out + 56 + (8 if use_idx else 0))
            res["rows_%d" % rows] = {"indices": use_idx, "call_us": [x * 1e6 for x in times], "call_us_median": t * 1e6,
                                     "rows_per_s": rows / t, "GBps": moved / t / 1e9}
        want = S.positions_to_training(S.GAME_C4, recs[:262144])
        got = [x.cpu().numpy() for x in S.positions_to_training_device(e, dev[:262144])]
        assert all(np.array_equal(g.view(np.uint32), w.view(np.uint32)) for g, w in zip(got, want))
        host = []
        for _ in range(reps):
            t0 = time.perf_counter()
            S.positions_to_training(S.GAME_C4, recs[:262144])
            host.append(time.perf_counter() - t0)
        res["host_262144"] = {"ms": [x * 1e3 for x in host], "rows_per_s": 262144 / statistics.median(host)}
        res["bit_identical_262144"] = True
        print("builder", json.dumps(res), flush=True)
        return res


def bench_line(extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "3"] + extra,
                       capture_output=True, text=True, cwd=ROOT)
    lines = [x for x in r.stdout.splitlines() if x.startswith("{")]
    return json.loads(lines[-1]) if lines else {"error": r.stderr[-2000:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--c4-plies", type=int, default=60)
    ap.add_argument("--chess-plies", type=int, default=48)
    ap.add_argument("--no-bench", action="store_true")
    a = ap.parse_args()
    name, power = gpu_info()
    res = {"tool": "tools/learner_path_bench.py", "gpu": name, "power_limit": power, "hbm_GBps_reference": HBM_GBPS}
    res["connect4"] = hand_off("connect4", c4_pair, 4096, a.c4_plies, a.reps, S.POSITION_DTYPE.itemsize)
    res["chess"] = hand_off("chess", chess_pair, 4096, a.chess_plies, a.reps, CH.CHESS_POSITION_DTYPE.itemsize)
    res["connect4_builder"] = builder(a.reps)
    if not a.no_bench:
        res["bench_c4"] = bench_line([])
        res["bench_chess"] = bench_line(["--game", "chess"])
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "power_limit")}))


if __name__ == "__main__":
    main()
