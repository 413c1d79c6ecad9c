"""Evaluation cache of the asynchronous pipeline at bench.py's default shape (4,096 trees x 800 simulations, bench's weights
and seeded roots): leaves the reference evaluates (counters.evaluations), positions the network received (async_stats
boards), the fraction served from the cache, and the network's true tensor rate = boards x FLOPs per position / search
time (bench.py's roofline.achieved counts every evaluation, so it overstates the rate by 1 / (1 - hit fraction)).

    python tools/eval_cache_hits.py [--game c4|ttt ...] [--searches N]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import selfplay_b200 as S
from selfplay_b200.synth import synthetic_roots_device
from selfplay_b200.weights_init import random_checkpoint


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--game", nargs="+", default=["c4", "ttt"], choices=["c4", "ttt"])
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=800)
    ap.add_argument("--searches", type=int, default=3)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    for game in args.game:
        c4 = game == "c4"
        with S.Engine(game=S.GAME_C4 if c4 else S.GAME_TTT, num_games=args.games, evaluator=S.EVAL_NET,
                      max_nodes_per_tree=1024 * ((7 * args.sims + 1024) // 1024)) as e:
            e.load_weights(random_checkpoint(1 if c4 else 0, 0))
            roots = synthetic_roots_device(e, args.games, start=0, max_ply=21 if c4 else 5)
            e.reset_games(roots)
            e.search(args.sims)                                   # warm-up (allocates the table)
            for _ in range(args.searches):
                e.reset_games(roots)
                e.reset_counters()
                e.search(args.sims)
                ms = e.last_search_timing()[0]
                ctr, st = e.counters(), e.async_stats()
                _, _, flops = e.time_evaluator(iters=2)
                print(json.dumps({"game": game, "gpu": gpu, "evaluations": ctr["evaluations"], "boards": st["boards"],
                                  "hit_fraction": 1.0 - st["boards"] / ctr["evaluations"], "search_ms": ms,
                                  "sims_per_s": args.games * args.sims / (ms * 1e-3),
                                  "network_tflops": st["boards"] * flops / (ms * 1e-3) / 1e12,
                                  "tflops_counting_every_evaluation": ctr["evaluations"] * flops / (ms * 1e-3) / 1e12,
                                  "tree_warp_busy_frac": st["tree_busy_ns"] / max(1, st["tree_warps"]) / (ms * 1e6),
                                  "us_per_tree_visit": st["tree_busy_ns"] / max(1, st["tree_visits"]) / 1e3}), flush=True)


if __name__ == "__main__":
    main()
