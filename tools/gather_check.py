"""The real-engine N-rank == 1-rank check (SURVEY.md §4 "Multi-GPU" row; ref: learner_concurrent.rs:201-230, :281-288).
Launch:  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/gather_check.py [--game chess]
Every rank plays its shard of the games (global ids by game_id_base / game_id_stride) for a few plies, the finished
trajectories are gathered to rank 0 over the C ABI (spb_gather_trajectories / spb_chess_gather_trajectories: NCCL all-gather
of counts + grouped send/recv); rank 0 then plays ALL the games on its own GPU and compares the SHA-256 of the two byte
streams.  Chess games start from the synthetic roots with their history filled to 500 plies, so every game ends at the
history cap within 13 plies and restarts from its root."""
import argparse
import hashlib
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import selfplay_b200 as S
from selfplay_b200.distributed import comm_init_over_process_group
from selfplay_b200.synth import synthetic_chess_roots_device, synthetic_roots_device
from selfplay_b200.weights_init import random_checkpoint, random_chess_checkpoint

ap = argparse.ArgumentParser()
ap.add_argument("--game", choices=("c4", "chess"), default="c4")
GAME = ap.parse_args().game

rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
os.environ.setdefault("MASTER_PORT", "29533")
torch.cuda.set_device(local)
dist.init_process_group("gloo", rank=rank, world_size=world)     # carries only the 128-byte id
G, PLIES, SIMS = (256, 12, 60) if GAME == "c4" else (128, 16, 40)


def generation(evaluator, device, g, base, stride, comm):
    with S.Engine(game=S.GAME_C4, num_games=g, evaluator=evaluator, device=device, game_id_base=base, game_id_stride=stride) as e:
        if evaluator == S.EVAL_NET:
            e.load_weights(random_checkpoint(1, 0))
        if comm:
            comm_init_over_process_group(e, rank, world)
        roots = synthetic_roots_device(e, g, start=base)
        e.reset_games(roots)
        for _ in range(PLIES):
            e.search(SIMS)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)
        pos, ids = e.gather_trajectories(0) if comm else e.drain_trajectories()
        if comm:
            e.comm_destroy()
    return pos, ids


def chess_roots(e, g, base):
    st, hist = synthetic_chess_roots_device(e, g, start=base)
    for i in range(g):                                                 # history to 500 plies, seeded per global game id
        h0 = int(st[i]["hist_len"])
        hist[i, h0:500] = np.random.default_rng(base + i).integers(1 << 40, 1 << 62, 500 - h0, dtype=np.uint64)
        st[i]["hist_len"] = 500
    return st, hist


def chess_generation(evaluator, device, g, base, stride, comm):
    with S.chess.ChessEngine(num_games=g, evaluator=evaluator, device=device, game_id_base=base, game_id_stride=stride) as e:
        if evaluator == S.EVAL_NET:
            e.load_weights(random_chess_checkpoint(seed=2))
        if comm:
            comm_init_over_process_group(e, rank, world)
        st, hist = chess_roots(e, g, base)
        e.reset_games(st, hist)
        for _ in range(PLIES):
            e.search(SIMS)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=st, restart_history=hist)
        pos, ids = e.gather_trajectories(0) if comm else e.drain_trajectories()
        if comm:
            e.comm_destroy()
    return pos, ids


if GAME == "chess":
    generation = chess_generation  # noqa: F811
ok = True
for name, ev in (("DetEval", S.EVAL_DET), ("network", S.EVAL_NET)):
    pos, ids = generation(ev, local, G, rank * G, world * G, True)
    if rank == 0:
        sha_n = hashlib.sha256(pos.tobytes() + ids.tobytes()).hexdigest()
        pos1, ids1 = generation(ev, local, world * G, 0, world * G, False)
        sha_1 = hashlib.sha256(pos1.tobytes() + ids1.tobytes()).hexdigest()
        same = sha_n == sha_1
        ok = ok and same
        print("%s%-8s %d ranks x %d games, %d plies x %d sims: %d positions gathered, sha256 %s | 1 rank x %d games: %d positions, sha256 %s | %s" % (
            "chess " if GAME == "chess" else "", name, world, G, PLIES, SIMS, len(pos), sha_n[:16], world * G, len(pos1), sha_1[:16], "IDENTICAL" if same else "DIFFERENT"), flush=True)
    else:
        assert len(pos) == 0
dist.barrier()
dist.destroy_process_group()
sys.exit(0 if ok else 1)
