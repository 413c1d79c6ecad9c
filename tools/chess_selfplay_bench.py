"""Chess self-play ply on the device against the caller's own host loop, in one process (one JSON line on stdout).

4,096 games x 200 simulations with the network evaluator (random-init checkpoint) from the bench's synthetic roots.  Two
engines with the same weights and roots run M moves, alternating move by move so that both see the same power state:
  (a) spb_chess_search + spb_chess_selfplay_step(greedy, restart_roots = the roots)
  (b) spb_chess_search + spb_chess_root_children_all + last-max pick on the host + spb_chess_advance
Before every step both engines' root children (moves and counts) are compared slot by slot, outside the timed windows: equal
trees mean both loops chose the same moves.  Slots whose game ended in (a) are left out from then on, since (a) restarts
them and (b) does not.  Times are host clocks around calls that end in a stream synchronisation; the self-play step alone is
also timed with CUDA events recorded before and after its (synchronous) call.

usage: python tools/chess_selfplay_bench.py [--games 4096] [--sims 200] [--moves 8] [--warmup 1]
"""
import argparse
import json
import os
import subprocess
import sys
import time

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=4096)
    ap.add_argument("--sims", type=int, default=200)
    ap.add_argument("--moves", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=1)
    a = ap.parse_args()
    import torch
    import selfplay_b200 as S
    from selfplay_b200.synth import synthetic_chess_roots_device
    from selfplay_b200.weights_init import random_chess_checkpoint
    CH = S.chess
    G, sims = a.games, a.sims
    blob = random_chess_checkpoint(seed=0)
    cap = G * (a.warmup + a.moves + 1)                                # every game of the run fits: no parking in the timed window
    ea = CH.ChessEngine(num_games=G, evaluator=S.EVAL_NET, trajectory_capacity=cap)
    eb = CH.ChessEngine(num_games=G, evaluator=S.EVAL_NET)
    for e in (ea, eb):
        e.load_weights(blob)
    roots, hist = synthetic_chess_roots_device(ea, G)
    for e in (ea, eb):
        e.reset_games(roots, hist)
    bufs = tuple(torch.empty(s, dtype=d).pin_memory().numpy() for s, d in (((G, CH.MAX_MOVES), torch.int16), ((G, CH.MAX_MOVES), torch.int32),
                                                                          ((G, CH.MAX_MOVES), torch.int32), ((G,), torch.int32)))
    bufs = (bufs[0].view(np.uint16), bufs[1].view(np.uint32), bufs[2].view(np.uint32), bufs[3].view(np.uint32))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t = dict(a_search=0.0, a_step=0.0, a_step_events=0.0, b_search=0.0, b_host=0.0)
    finished = drained = 0
    ended = np.zeros(G, bool)
    mismatch = 0
    for k in range(a.warmup + a.moves):
        timed = k >= a.warmup
        t0 = time.perf_counter()
        ea.search(sims)
        t1 = time.perf_counter()
        eb.search(sims)
        t2 = time.perf_counter()
        mv_a, cnt_a, _, n_a = (x.copy() for x in ea.root_children_all())
        mv_b, cnt_b, _, n_b = (x.copy() for x in eb.root_children_all())
        same = (mv_a == mv_b).all(1) & (cnt_a == cnt_b).all(1) & (n_a == n_b)
        mismatch += int((~same & ~ended).sum())
        t3 = time.perf_counter()
        ev0.record()
        fin = ea.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots, restart_history=hist)
        ev1.record()
        t4 = time.perf_counter()
        mv, cnt, ids, n = eb.root_children_all(out=bufs)
        c = np.where(np.arange(CH.MAX_MOVES)[None, :] < n[:, None], cnt.astype(np.int64), -1)
        last = CH.MAX_MOVES - 1 - np.argmax(c[:, ::-1], axis=1)         # last maximum, main.rs:108-112
        live = np.flatnonzero(n > 0)                                    # a game that ended in (b) stays at its terminal root
        eb.advance(ids[live, last[live]], slots=live)
        t5 = time.perf_counter()
        torch.cuda.synchronize()
        if fin:
            pos, gid = ea.drain_trajectories()
            drained += len(pos)
            ended[(gid % G).astype(np.int64)] = True
        if timed:
            finished += fin
            t["a_search"] += t1 - t0
            t["b_search"] += t2 - t1
            t["a_step"] += t4 - t3
            t["a_step_events"] += ev0.elapsed_time(ev1) / 1e3
            t["b_host"] += t5 - t4
    drained += len(ea.drain_trajectories()[0])
    name, limit = card()
    M = a.moves
    loop_a = t["a_search"] + t["a_step"]
    loop_b = t["b_search"] + t["b_host"]
    out = dict(
        tool="chess_selfplay_bench", games=G, sims_per_move=sims, moves=M, warmup=a.warmup, evaluator="net (random init)",
        loop_a_sims_per_s=G * sims * M / loop_a, loop_a_positions_per_s=G * M / loop_a,
        loop_b_sims_per_s=G * sims * M / loop_b, loop_b_positions_per_s=G * M / loop_b,
        search_ms_per_move_a=1e3 * t["a_search"] / M, search_ms_per_move_b=1e3 * t["b_search"] / M,
        selfplay_step_ms_per_move=1e3 * t["a_step"] / M, selfplay_step_device_ms_per_move=1e3 * t["a_step_events"] / M,
        host_loop_ms_per_move=1e3 * t["b_host"] / M,
        finished_games=finished, records_drained=int(drained), slots_compared_mismatch=mismatch,
        gpu=name, power_limit=limit)
    print(json.dumps(out))
    ea.close()
    eb.close()
    if mismatch:
        sys.exit("loops (a) and (b) chose different moves in %d slot-plies" % mismatch)


if __name__ == "__main__":
    main()
