"""Cost of Dirichlet root noise (DESIGN.md §4.6) at the bench workloads, in one process (one JSON line on stdout and in
--out, default profiles/r05_root_noise_bench.json).

  * Connect4: 4,096 games x 800 simulations, network evaluator (random-init checkpoint), the bench's synthetic roots.
  * chess:    4,096 games x 200 simulations, network evaluator (random-init checkpoint), the bench's synthetic roots.
Per game, one engine with the noise off and one with it on (alpha 0.3, epsilon 0.25) search the same roots, alternating search
by search so that both see the same power state; every search starts from fresh trees (reset_games outside the timed window).
The search time is spb_last_search_timing / spb_chess_last_search_ms (CUDA events around the whole search, including the draw).
The draw alone (k_root_noise / k_chess_root_noise over all 4,096 roots) is timed with CUDA events through spb_root_noise,
which launches it once and then copies one row: the events bracket the call, so the time is an upper bound on the kernel.

usage: python tools/root_noise_bench.py [--games 4096] [--c4-sims 800] [--chess-sims 200] [--reps 5] [--draws 50]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as ex:                                           # the numbers are still printed, without the card
        return "unknown (%s)" % ex, "unknown"


def time_draw(torch, eng, n):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eng.root_noise(0)                                                 # warm-up
    torch.cuda.synchronize()
    ms = []
    for _ in range(n):
        ev0.record()
        eng.root_noise(0)
        ev1.record()
        ev1.synchronize()
        ms.append(ev0.elapsed_time(ev1))
    return float(np.median(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--c4-sims", type=int, default=800)
    ap.add_argument("--chess-sims", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--draws", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_root_noise_bench.json"))
    a = ap.parse_args()
    import torch
    import selfplay_b200 as S
    from selfplay_b200.synth import synthetic_chess_roots_device, synthetic_roots_device
    from selfplay_b200.weights_init import random_checkpoint, random_chess_checkpoint
    G = a.games
    alpha, eps = 0.3, 0.25
    res = dict(tool="root_noise_bench", games=G, alpha=alpha, epsilon=eps, reps=a.reps, evaluator="net (random init)")

    # ---- Connect4 -----------------------------------------------------------------------------------------------------
    blob = random_checkpoint(1, 0)
    engs = [S.Engine(game=S.GAME_C4, num_games=G, evaluator=S.EVAL_NET) for _ in range(2)]
    for e in engs:
        e.load_weights(blob)
    roots = synthetic_roots_device(engs[0], G, start=0, max_ply=21)
    engs[1].set_root_noise(alpha, eps, 1)
    ms = [[], []]
    for k in range(a.reps + 1):
        for i, e in enumerate(engs):
            e.reset_games(roots)
            e.search(a.c4_sims)
            if k:
                ms[i].append(e.last_search_timing()[0])
    res["c4_sims"] = a.c4_sims
    res["c4_search_ms_off"] = [round(x, 3) for x in ms[0]]
    res["c4_search_ms_on"] = [round(x, 3) for x in ms[1]]
    res["c4_sims_per_s_off"] = G * a.c4_sims / (1e-3 * float(np.median(ms[0])))
    res["c4_sims_per_s_on"] = G * a.c4_sims / (1e-3 * float(np.median(ms[1])))
    engs[1].reset_games(roots)
    res["c4_draw_ms"] = time_draw(torch, engs[1], a.draws)
    for e in engs:
        e.close()

    # ---- chess --------------------------------------------------------------------------------------------------------
    cblob = random_chess_checkpoint(seed=0)
    cap = 1024 * ((64 * a.chess_sims + 2048) // 1024)                 # the bench's pool size
    cengs = [S.ChessEngine(num_games=G, evaluator=S.EVAL_NET, max_nodes_per_tree=cap) for _ in range(2)]
    for e in cengs:
        e.load_weights(cblob)
    croots, chist = synthetic_chess_roots_device(cengs[0], G)
    cengs[1].set_root_noise(alpha, eps, 1)
    ms = [[], []]
    for k in range(a.reps + 1):
        for i, e in enumerate(cengs):
            e.reset_games(croots, chist)
            e.search(a.chess_sims)
            if k:
                ms[i].append(e.last_search_ms())
    res["chess_sims"] = a.chess_sims
    res["chess_search_ms_off"] = [round(x, 2) for x in ms[0]]
    res["chess_search_ms_on"] = [round(x, 2) for x in ms[1]]
    res["chess_sims_per_s_off"] = G * a.chess_sims / (1e-3 * float(np.median(ms[0])))
    res["chess_sims_per_s_on"] = G * a.chess_sims / (1e-3 * float(np.median(ms[1])))
    cengs[1].reset_games(croots, chist)
    res["chess_draw_ms"] = time_draw(torch, cengs[1], a.draws)
    for e in cengs:
        e.close()

    res["gpu"], res["power_limit"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
