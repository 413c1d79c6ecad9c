#!/usr/bin/env python
"""bench.py — MCTS simulations/sec for Connect4 at 800 sims/move (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W          # this framework, one rank per GPU
    python bench.py --impl reference ...                   # the reference's algorithm on the host CPU cores
    python bench.py --leaves 16                            # configs[3]: 16 leaves in flight per tree (virtual loss, lock-step)
    python bench.py --game ttt --sims 600                  # configs[0]: tic-tac-toe
    python bench.py --game chess                           # configs[4]: chess, 200 sims/move, the 10x256 net (lock-step)

One "step" = one `search` call (ref: Mcts::search, src/mcts.rs:196) of 800 simulations over 4,096 concurrent
Connect4 games per GPU, every tree fresh at a seeded synthetic root (SURVEY.md §8d), evaluator = the
reference's 4x64 conv ResNet with random-init weights (bf16 on tcgen05, fp32 accumulate).  Work per GPU is
fixed (weak scaling); `value` is the whole-job aggregate.

  value     sims/s with the roots already resident in HBM; device time (CUDA events on the engine's stream),
            max over ranks.
  e2e       the same metric through the C ABI with HOST buffers: spb_reset_games (H2D) + spb_search +
            spb_root_children_all (D2H) per step, page-locked host buffers allocated once, wall clock between
            synchronisations, max over ranks.  The K value steps
            and the K e2e steps alternate, so that both are measured in the same power state of the board.
  roofline  the dominant kernel.  Default (asynchronous pipeline): ONE resident kernel per search that holds the tcgen05
            evaluator and the tree warps; achieved = evaluated positions x FLOPs per position / the search's device time
            (CUDA events on the engine's stream), against the measured sustained bf16 peak of MEASURED_PEAKS.json.
            `traffic` is read from the committed ncu summary of that kernel (profiles/, named in the line).
  cpu_baseline  the C++ restatement of the reference (oracle/) with the torch CPU fp32 net, one PROCESS per host core
            (the reference's workers share nothing: src/main.rs:169), 100 games each, one full 800-simulation search
            (rank 0, N = 1 only).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GAMES_PER_GPU = 4096
SIMS = 800
REF_GAMES_PER_THREAD = 100        # learner_concurrent.rs:56 num_batched_self_play_games
REF_SEGMENT = 100                 # the CPU arm's step: 100 consecutive simulations of an 800-simulation search
METRIC = "MCTS simulations/sec (whole box) Connect4 @800 sims/move"
WORKLOAD = "connect4_6x7_batched_selfplay_4096_games_x_800_sims_per_gpu"
NCU_SUMMARY = os.path.join("profiles", "r02_ncu_eval_async_summary.json")   # source of roofline.traffic


def workload_name(game, games, sims, leaves):
    if game == "ttt":
        return "tictactoe_3x3_selfplay_%d_games_x_%d_sims_per_gpu" % (games, sims)
    if leaves > 1:
        return "connect4_6x7_parallel_tree_search_virtual_loss_%d_leaves_per_tree_%d_games_x_%d_sims_per_gpu" % (leaves, games, sims)
    if (games, sims) == (GAMES_PER_GPU, SIMS):
        return WORKLOAD
    return "connect4_6x7_batched_selfplay_%d_games_x_%d_sims_per_gpu" % (games, sims)


def metric_name(game, sims):
    return METRIC if (game, sims) == ("c4", SIMS) else "MCTS simulations/sec (whole box) %s @%d sims/move" % (
        "Connect4" if game == "c4" else "tic-tac-toe", sims)


NCU_SUMMARY_CHESS = os.path.join("profiles", "r02_ncu_chess_conv_summary.json")   # k_conv<8,9,256> over 2,048 positions


def pinned(arr):
    """A copy of `arr` in page-locked host memory (the e2e steps copy their inputs from / their results to pinned buffers)."""
    import numpy as np
    import torch
    t = torch.empty(max(1, arr.nbytes), dtype=torch.uint8, pin_memory=True)
    out = t.numpy()[:arr.nbytes].view(arr.dtype).reshape(arr.shape)
    out[...] = arr
    out.flags.writeable = True
    _PINNED_KEEPALIVE.append(t)
    return out


_PINNED_KEEPALIVE = []

DUMP_BYTES = 64 * 10 ** 6         # --dump-outputs: at most this much data in all


def dump_outputs(path, arrays):
    """--dump-outputs: writes the per-game arrays a caller of the timed path received in its last step as <path>/<name>.npy
    in float64 (exact for their integer values), and <path>/game_index.npy, the games (rows) written.  A result larger than
    DUMP_BYTES is cut to a fixed, seeded sample of games, so that two builds run with the same arguments write the same rows."""
    import numpy as np
    games = len(next(iter(arrays.values())))
    row_bytes = 8 * (1 + sum(a[0].size for a in arrays.values()))
    keep = np.arange(games)
    if games * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(games, (DUMP_BYTES - 1024 * (len(arrays) + 1)) // row_bytes, replace=False))
    os.makedirs(path, exist_ok=True)
    for name, a in dict({k: a[keep] for k, a in arrays.items()}, game_index=keep).items():
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


def ncu_traffic(summary=None):
    """DRAM bytes (read + write) per launch of the dominant kernel, from the committed `ncu --set full` summary."""
    summary = summary or NCU_SUMMARY
    try:
        with open(os.path.join(ROOT, summary)) as f:
            j = json.load(f)
        return j.get("traffic_bytes_per_launch"), summary
    except Exception:
        return None, None


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json, sustained)"
    except Exception:
        return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx, self.proc, self.lines = device_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# -------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle (C++ restatement of mcts.rs + connect_four.rs) with the torch CPU net
# -------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's self-play workers on the host cores: one process per worker (oracle/cpu_worker.py), each an
    independent `search` over its own 100 games (learner_concurrent.rs:56) with its own copy of the net — the shape of
    main.rs:169's SelfPlayWorkers.  A step = `segment` consecutive simulations; the trees persist until `sims` simulations
    have been run on them (one full search), then every worker starts fresh trees."""

    def __init__(self, game: str, sims: int, blob: bytes, workers: int | None = None, segment: int = REF_SEGMENT):
        import tempfile
        self.workers = workers or (os.cpu_count() or 1)
        self.sims, self.segment = sims, min(segment, sims)
        self.done_on_trees = 0
        self.tmp = tempfile.NamedTemporaryFile(suffix=".safetensors", delete=False)
        self.tmp.write(blob)
        self.tmp.close()
        gid = 1 if game == "c4" else 0
        env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
        self.procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "cpu_worker.py"), str(gid), str(w),
                                        str(REF_GAMES_PER_THREAD), self.tmp.name], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                       stderr=subprocess.DEVNULL, text=True, env=env) for w in range(self.workers)]
        for p in self.procs:
            if p.stdout.readline().strip() != "ready":
                raise RuntimeError("CPU worker failed to start")

    def _all(self, cmd):
        for p in self.procs:
            p.stdin.write(cmd + "\n")
            p.stdin.flush()
        return [p.stdout.readline().split() for p in self.procs]

    def step(self):
        """-> (simulations, evaluations, terminal leaves, wall seconds) of one step over all workers."""
        if self.done_on_trees >= self.sims:
            self._all("reset")                                   # Tree::with_root_state: next search, untimed
            self.done_on_trees = 0
        n = min(self.segment, self.sims - self.done_on_trees)
        t0 = time.perf_counter()
        rep = self._all("step %d" % n)
        dt = time.perf_counter() - t0
        self.done_on_trees += n
        return sum(int(r[0]) for r in rep), sum(int(r[1]) for r in rep), sum(int(r[2]) for r in rep), dt

    def sample(self):
        return ("%d worker processes x %d games, each step = %d consecutive simulations of a %d-simulation search (trees persist for "
                "%d steps, then fresh trees at the same seeded roots); torch CPU fp32 evaluator, 1 intra-op thread per worker" % (
                    self.workers, REF_GAMES_PER_THREAD, self.segment, self.sims, -(-self.sims // self.segment)))

    def close(self):
        for p in self.procs:
            try:
                p.stdin.write("quit\n")
                p.stdin.flush()
            except Exception:
                pass
        for p in self.procs:
            try:
                p.wait(timeout=10)
            except Exception:
                p.kill()
        os.unlink(self.tmp.name)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0                                          # rank 0 alone runs the CPU arm
    from selfplay_b200.weights_init import random_checkpoint
    arm = CpuArm(args.game, args.sims, random_checkpoint(1 if args.game == "c4" else 0, 0), segment=args.ref_segment)
    tot = [0, 0, 0, 0.0]
    try:
        for i in range(args.warmup + args.steps):
            r = arm.step()
            if i >= args.warmup:
                tot = [a + b for a, b in zip(tot, r)]
    finally:
        sample = arm.sample()
        threads = arm.workers
        arm.close()
    value = tot[0] / tot[3]
    line = {
        "impl": "reference", "metric": metric_name(args.game, args.sims), "value": value, "unit": "sims/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot[3] / max(1, args.steps), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.game, args.games, args.sims, 1),
                   "reference_arm": "oracle port of src/mcts.rs + src/game/*.rs (the Rust crate cannot be built here: no rustc/cargo), evaluator = torch CPU fp32",
                   "sample": sample, "terminal_leaf_fraction": tot[2] / max(1, tot[0])},
        "cpu_baseline": {"value": value, "unit": "sims/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


# -------------------------------------------------------------------------------------------------
# this framework
# -------------------------------------------------------------------------------------------------
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import selfplay_b200 as S
    from selfplay_b200.synth import synthetic_roots_device
    from selfplay_b200.weights_init import random_checkpoint

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")

    G, sims, K = args.games, args.sims, args.leaves
    game = S.GAME_C4 if args.game == "c4" else S.GAME_TTT
    A_branch = 7 if args.game == "c4" else 9
    blob = random_checkpoint(1 if args.game == "c4" else 0, 0)
    # node pools sized for the full-game leg (a tree can carry nearly all of its nodes through a re-root and adds at most
    # A per simulation), so that no pool growth (spb_search widens the pools on demand) lands inside a timed region
    eng = S.Engine(game=game, num_games=G, evaluator=S.EVAL_NET, device=local_rank, leaves_per_tree=K,
                   game_id_base=rank * G, game_id_stride=world * G,
                   max_nodes_per_tree=1024 * ((A_branch * sims * (args.full_game_moves + 1) + 1024) // 1024))
    eng.load_weights(blob)
    # games are sharded by rank: rank r owns ids [r*G, (r+1)*G)
    roots = synthetic_roots_device(eng, G, start=rank * G, max_ply=21 if args.game == "c4" else 5)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- warm-up ------------------------------------------------------------------------------------
    roots = pinned(roots)                 # host buffers of the e2e steps: page-locked, allocated once
    out_bufs = tuple(pinned(x) for x in eng.root_children_all())
    for _ in range(args.warmup):
        eng.reset_games(roots)
        eng.search(sims)
        eng.root_children_all(out_bufs)

    # ---- timed regions: device-resident (`value`) and end to end through the C ABI with host buffers (`e2e`) ----------
    # K steps each, ALTERNATING (value step, e2e step, value step, ...): the board sits at its power cap and its clocks drift
    # over seconds, so two loops run one after the other would be measured in two different power states.  `value` sums
    # the device time of its K searches (CUDA events on the engine stream inside spb_search); `e2e` sums the wall time of
    # its K steps, each = H2D of the step's inputs + search + D2H of the step's result (synchronous calls).
    sampler = ClockSampler(local_rank)
    sampler.start()
    ADDITIVE = ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "kernel_launches")
    ctr, stats = None, None
    barrier()
    dev_ms, wall_s, e2e_s = 0.0, 0.0, 0.0
    for _ in range(args.steps):
        eng.reset_counters()
        t0 = time.perf_counter()
        eng.reset_games(roots)            # untimed part of `value`: fresh trees; roots then live in HBM
        eng.search(sims)                  # synchronous; its device time is measured with CUDA events inside
        wall_s += time.perf_counter() - t0
        dev_ms += eng.last_search_timing()[0]
        c = eng.counters()
        ctr = c if ctr is None else {k: (ctr[k] + c[k] if k in ADDITIVE else c[k]) for k in c}
        stats, stats_ms = eng.async_stats(), eng.last_search_timing()[0]
        t0 = time.perf_counter()
        eng.reset_games(roots)            # H2D of the step's inputs
        eng.search(sims)
        acts, counts, ids, ncs = eng.root_children_all(out_bufs)   # D2H of the step's result
        e2e_s += time.perf_counter() - t0
    barrier()
    launches = ctr["kernel_launches"]
    dev_ms = rank_max(dev_ms)
    wall_s = rank_max(wall_s)
    e2e_s = rank_max(e2e_s)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"actions": acts, "visit_counts": counts, "child_ids": ids, "n_children": ncs})
    h2d = G * 16
    d2h = G * (2 * 4 * S.MAX_ACTIONS + 4 + S.MAX_ACTIONS)
    assert int(counts[0].sum()) == sims - (K if K > 1 else 1)

    # ---- roofline of the dominant kernel, measured live ------------------------------------------------
    peak_tf, peak_hbm, peak_src = _peaks()
    total_sims = world * G * sims * args.steps
    value = total_sims / (dev_ms * 1e-3)
    D = ctr["path_length_sum"] / max(1, ctr["simulations"])
    bbar = ctr["children_created"] / max(1, ctr["evaluations"])
    tree_bytes_per_sim = 16 * bbar * D + 36 * bbar + 16 * D + 96            # SURVEY.md §8(d)
    static_ms, static_n, flops_pos = eng.time_evaluator(iters=10)            # also: FLOPs per position
    if K == 1:
        # asynchronous pipeline: one resident kernel per search = evaluator CTAs + tree warps.  Its duration is the search's
        # device time (the ring reset and the queueing kernel in front of it take microseconds).
        evals_per_launch = ctr["evaluations"] / args.steps
        launch_ms = dev_ms / args.steps
        kernel = "umma::k_eval_umma<%s, RING=true> (resident: tcgen05 evaluator + tree warps)" % ("Connect4" if args.game == "c4" else "TicTacToe")
        traffic, traffic_src = ncu_traffic() if (args.game, G, sims) == ("c4", GAMES_PER_GPU, SIMS) else (None, None)
    else:
        evals_per_launch, launch_ms = static_n, static_ms
        kernel = "umma::k_eval_umma<Connect4, RING=false> (one launch per lock-step, %d leaves per tree)" % K
        traffic, traffic_src = None, None
    achieved_tf = flops_pos * evals_per_launch / (launch_ms * 1e-3) / 1e12
    roof = {"bound": "tensor", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
            "traffic": traffic, "traffic_source": traffic_src, "kernel": kernel, "peak_source": peak_src,
            "positions_per_launch": evals_per_launch, "flops_per_position": flops_pos, "avg_launch_ms": launch_ms,
            "static_list_launch": {"positions": static_n, "ms": static_ms,
                                   "tflops": flops_pos * static_n / (static_ms * 1e-3) / 1e12,
                                   "note": "the same evaluator on one static list (spb_predict / lock-step shape), timed alone"}}
    line = {
        "metric": metric_name(args.game, sims), "value": value, "unit": "sims/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": workload_name(args.game, G, sims, K),
                   "games_per_gpu": G, "sims_per_move": sims, "leaves_per_tree": K,
                   "pipeline": "asynchronous (trees and leaves circulate between tree warps and resident evaluator CTAs)" if K == 1 else "lock-step with virtual loss",
                   "evaluator": "%s 4x64 conv ResNet, random init (numpy seed 0), BN folded" % ("connect4" if args.game == "c4" else "tic-tac-toe"),
                   "parallelism": "games sharded by rank, no collective on the search path",
                   "cache": "inputs larger than L2: per-GPU node pools touched per step ~%d MB" % (ctr["nodes_live"] * 20 // (1 << 20)),
                   "timing": "CUDA events on the engine stream around each search, max over ranks; wall clock %.3f s; value and e2e steps alternate (same power state)" % wall_s},
        "e2e": {"value": total_sims / e2e_s, "unit": "sims/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "tree_side": {"bytes_per_sim_algorithmic": tree_bytes_per_sim, "mean_path_length": D, "mean_branching": bbar,
                      "algorithmic_gbs": tree_bytes_per_sim * G * sims * args.steps / (dev_ms * 1e-3) / 1e9, "hbm_peak_gbs": peak_hbm,
                      "tree_warps": stats["tree_warps"], "tree_warp_busy_frac": stats["tree_busy_ns"] / max(1, stats["tree_warps"]) / max(1e-9, stats_ms * 1e6),
                      "us_per_tree_visit": stats["tree_busy_ns"] / max(1, stats["tree_visits"]) / 1e3,
                      "boards_per_evaluator_batch": stats["boards"] / max(1, stats["batches"]),
                      "note": "latency-bound pointer chasing that runs under the evaluator in the same kernel; statistics of the last search (spb_last_async_stats)"},
        "counters": {k: ctr[k] for k in ("simulations", "evaluations", "terminal_leaves")},
        "terminal_leaf_fraction": ctr["terminal_leaves"] / max(1, ctr["simulations"]),
    }
    # ---- full-game leg: greedy last-max moves, subtree reuse, finished slots refilled from the same roots ------
    if args.full_game_moves > 0:
        eng.reset_games(roots)
        eng.drain_trajectories()
        barrier()
        t0 = time.perf_counter()
        finished = 0
        for _ in range(args.full_game_moves):
            eng.search(sims)                                   # carry + 800 more simulations per move (mcts.rs:161-192)
            finished += eng.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)
        barrier()
        fg_s = rank_max(time.perf_counter() - t0)
        pos, _ = eng.drain_trajectories()
        line["full_game"] = {"moves": args.full_game_moves, "value": world * G * sims * args.full_game_moves / fg_s, "unit": "sims/s",
                             "finished_games_rank0": int(finished), "trajectory_positions_rank0": int(len(pos)),
                             "note": "search + on-device move selection + use_subtree per move, wall clock"}
    # ---- CPU baseline beside it (rank 0, N = 1 only): ONE full search of `sims` simulations on every host core ----------
    if world == 1 and not args.no_cpu_baseline:
        eng.close()
        arm = CpuArm(args.game, sims, blob, segment=args.ref_segment)
        tot = [0, 0, 0, 0.0]
        try:
            for _ in range(-(-sims // arm.segment)):
                tot = [a + b for a, b in zip(tot, arm.step())]
        finally:
            sample, threads = arm.sample(), arm.workers
            arm.close()
        line["cpu_baseline"] = {"value": tot[0] / tot[3], "unit": "sims/s", "cores": threads, "kind": "port",
                                "sample": sample + "; one full search, same seeded roots and weights as the GPU arm",
                                "terminal_leaf_fraction": tot[2] / max(1, tot[0])}
    else:
        line["cpu_baseline"] = None
    # ---- multi-GPU: the one exchange of the path — trajectories to the learner rank over the C ABI (NCCL) -------------
    if world > 1:
        import hashlib
        from selfplay_b200.distributed import comm_init_over_process_group
        eng.drain_trajectories()
        comm_init_over_process_group(eng, rank, world)
        eng.reset_games(roots)
        for _ in range(2):
            eng.search(sims)
            eng.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)
        eng.gather_trajectories(0)                               # first use sets up NCCL's connections
        eng.search(sims)
        eng.selfplay_step(S.MOVE_GREEDY_LAST_MAX, restart_roots=roots)
        barrier()
        t0 = time.perf_counter()
        pos, gids = eng.gather_trajectories(0)
        dt = time.perf_counter() - t0
        eng.comm_destroy()
        line["trajectory_gather"] = {"positions": int(len(pos)) if rank == 0 else None, "seconds": dt,
                                     "sha256": hashlib.sha256(pos.tobytes() + gids.tobytes()).hexdigest() if rank == 0 else None,
                                     "transport": "spb_gather_trajectories (C ABI): NCCL all-gather of counts + grouped send/recv, ordered by (game id, ply)",
                                     "n_rank_equals_1_rank": "tools/gather_check.py (profiles/r02_gather_check.txt)"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


# -------------------------------------------------------------------------------------------------
# chess (BASELINE.json configs[4]): bitboard move generation + MCTS at 200 sims/move with the 10x256 net
# -------------------------------------------------------------------------------------------------
CHESS_SIMS = 200
CHESS_GAMES_PER_GPU = 4096
CHESS_MAX_PLY = 41


class ChessCpuArm(CpuArm):
    """The CPU arm for chess: oracle/chess_cpu_worker.py processes (oracle MCTS over chess + torch CPU fp32 net)."""

    def __init__(self, sims: int, blob: bytes, games_per_worker: int, workers: int | None = None, segment: int = 4):
        import tempfile
        self.workers = workers or (os.cpu_count() or 1)
        self.sims, self.segment, self.games = sims, min(segment, sims), games_per_worker
        self.done_on_trees = 0
        self.tmp = tempfile.NamedTemporaryFile(suffix=".safetensors", delete=False)
        self.tmp.write(blob)
        self.tmp.close()
        env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1")
        self.procs = [subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "chess_cpu_worker.py"), str(w), str(games_per_worker),
                                        self.tmp.name, str(CHESS_MAX_PLY)], stdin=subprocess.PIPE, stdout=subprocess.PIPE,
                                       stderr=subprocess.DEVNULL, text=True, env=env) for w in range(self.workers)]
        for p in self.procs:
            if p.stdout.readline().strip() != "ready":
                raise RuntimeError("chess CPU worker failed to start")

    def sample(self):
        return ("%d worker processes x %d games, each step = %d consecutive simulations per tree from the seeded roots (a bounded "
                "sample of the %d-simulation search: the first simulations of every tree); torch CPU fp32 10x256 net, 1 intra-op thread "
                "per worker" % (self.workers, self.games, self.segment, self.sims))


def chess_workload(games, sims):
    return "chess_8x8_bitboard_movegen_mcts_%d_games_x_%d_sims_per_gpu" % (games, sims)


def run_chess_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    from selfplay_b200.weights_init import random_chess_checkpoint
    arm = ChessCpuArm(args.sims, random_chess_checkpoint(0), games_per_worker=8, segment=args.ref_segment if args.ref_segment != REF_SEGMENT else 4)
    tot = [0, 0, 0, 0.0]
    try:
        for i in range(args.warmup + args.steps):
            r = arm.step()
            if i >= args.warmup:
                tot = [a + b for a, b in zip(tot, r)]
    finally:
        sample, threads = arm.sample(), arm.workers
        arm.close()
    value = tot[0] / tot[3]
    print(json.dumps({
        "impl": "reference", "metric": "MCTS simulations/sec (whole box) chess @%d sims/move" % args.sims, "value": value, "unit": "sims/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot[3] / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": chess_workload(args.games, args.sims), "sample": sample,
                   "reference_arm": "oracle port of src/mcts.rs + src/game/chess.rs (no rustc/cargo here), evaluator = torch CPU fp32"},
        "cpu_baseline": {"value": value, "unit": "sims/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)
    return 0


def run_chess(args):
    import torch
    import torch.distributed as dist

    import selfplay_b200 as S
    from selfplay_b200.synth import synthetic_chess_roots_device
    from selfplay_b200.weights_init import random_chess_checkpoint

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")
    G, sims = args.games, args.sims
    blob = random_chess_checkpoint(0)
    eng = S.ChessEngine(num_games=G, evaluator=S.EVAL_NET, device=local_rank, max_nodes_per_tree=1024 * ((64 * sims + 2048) // 1024))
    eng.load_weights(blob)
    roots, hist = synthetic_chess_roots_device(eng, G, start=rank * G, max_ply=CHESS_MAX_PLY)   # games sharded by rank

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    roots, hist = pinned(roots), pinned(hist)   # host buffers of the e2e steps: page-locked, allocated once
    out_bufs = tuple(pinned(x) for x in eng.root_children_all())
    for _ in range(args.warmup):
        eng.reset_games(roots, hist)
        eng.search(sims)
        eng.root_children_all(out_bufs)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ADDITIVE = ("simulations", "evaluations", "terminal_leaves", "path_length_sum", "children_created", "kernel_launches")
    ctr = None
    barrier()
    dev_ms, wall_s, e2e_s = 0.0, 0.0, 0.0
    for _ in range(args.steps):           # value step, e2e step, value step, ...: both measured in the same power state
        eng.reset_counters()
        t0 = time.perf_counter()
        eng.reset_games(roots, hist)
        eng.search(sims)
        wall_s += time.perf_counter() - t0
        dev_ms += eng.last_search_ms()
        c = eng.counters()
        ctr = c if ctr is None else {k: (ctr[k] + c[k] if k in ADDITIVE else c[k]) for k in c}
        t0 = time.perf_counter()
        eng.reset_games(roots, hist)                        # H2D: states + game histories
        eng.search(sims)
        mv, cnt, ids, ncs = eng.root_children_all(out_bufs)   # D2H: moves, visit counts, child ids
        e2e_s += time.perf_counter() - t0
    barrier()
    wall_s = rank_max(wall_s)
    dev_ms = rank_max(dev_ms)
    e2e_s = rank_max(e2e_s)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"moves": mv, "visit_counts": cnt, "child_ids": ids, "n_children": ncs})
    assert int(cnt[0].sum()) == sims - 1
    peak_tf, peak_hbm, peak_src = _peaks()
    conv_ms, conv_n, conv_flops, flops_pos = eng.time_conv(iters=20)
    total_sims = world * G * sims * args.steps
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12
    evals = ctr["evaluations"]
    line = {
        "metric": "MCTS simulations/sec (whole box) chess @%d sims/move" % sims, "value": total_sims / (dev_ms * 1e-3), "unit": "sims/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": chess_workload(G, sims), "games_per_gpu": G, "sims_per_move": sims, "leaves_per_tree": 1,
                   "pipeline": "lock-step (the reference's loop: select, one network batch, expand + backup), run as two half-loops over the two halves of the trees on two streams",
                   "evaluator": "chess 10x256 conv ResNet, random init (numpy seed 0), BN folded, bf16 operands / f32 accumulate",
                   "roots": "seeded random playouts of 0..%d plies from the start position (device rules)" % (CHESS_MAX_PLY - 1),
                   "parallelism": "games sharded by rank, no collective on the search path",
                   "cache": "inputs larger than L2: activations of one layer %d MB, node pools touched ~%d MB" % (
                       G * 81 * 512 // (1 << 20), ctr["nodes_live"] * 32 // (1 << 20)),
                   "timing": "CUDA events on the engine stream around each search, max over ranks; wall clock %.3f s; value and e2e steps alternate (same power state)" % wall_s},
        "e2e": {"value": total_sims / e2e_s, "unit": "sims/s", "h2d_bytes_per_step": int(roots.nbytes + hist.nbytes),
                "d2h_bytes_per_step": int(mv.nbytes + cnt.nbytes + ids.nbytes + ncs.nbytes)},
        "gpu_launches": int(ctr["kernel_launches"]),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                     "traffic": ncu_traffic(NCU_SUMMARY_CHESS)[0] if conv_n == 2048 else None,
                     "traffic_source": NCU_SUMMARY_CHESS if conv_n == 2048 else None,
                     "kernel": "chess::k_conv<8, 9, 256> (one 256->256 3x3 residual convolution over the leaf batch; 20 of the 25 launches "
                               "per evaluation and 99 % of its FLOPs)",
                     "peak_source": peak_src, "positions_per_launch": conv_n, "flops_per_launch": conv_flops, "avg_launch_ms": conv_ms,
                     "useful_row_fraction": 64.0 / 72.0,   # an M tile is 16 board rows of 8 cells: 8 of 9 board rows of a position are real
                     "whole_network": {"flops_per_position": flops_pos,
                                       "tflops_over_search": flops_pos * evals / (dev_ms * 1e-3) / 1e12,
                                       "note": "all evaluations x FLOPs per evaluation / device time of the searches (tree kernels included)"}},
        "counters": {k: ctr[k] for k in ("simulations", "evaluations", "terminal_leaves")},
        "tree_side": {"mean_path_length": ctr["path_length_sum"] / max(1, ctr["simulations"]),
                      "mean_branching": ctr["children_created"] / max(1, ctr["evaluations"]), "largest_arena": ctr["largest_arena"]},
    }
    if world == 1 and not args.no_cpu_baseline:
        eng.close()
        arm = ChessCpuArm(sims, blob, games_per_worker=8)
        tot = [0, 0, 0, 0.0]
        try:
            for _ in range(3):
                tot = [a + b for a, b in zip(tot, arm.step())]
        finally:
            sample, threads = arm.sample(), arm.workers
            arm.close()
        line["cpu_baseline"] = {"value": tot[0] / tot[3], "unit": "sims/s", "cores": threads, "kind": "port", "sample": sample}
    else:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--games", type=int, default=None)
    ap.add_argument("--sims", type=int, default=None)
    ap.add_argument("--ref-segment", type=int, default=REF_SEGMENT, help="CPU arm: simulations per step (consecutive segments of one --sims search)")
    ap.add_argument("--leaves", type=int, default=1, help="leaves in flight per tree (configs[3]: 16); > 1 runs the lock-step virtual-loss pipeline")
    ap.add_argument("--game", default="c4", choices=["c4", "ttt", "chess"], help="configs[0] is tic-tac-toe, configs[4] chess")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-game-moves", type=int, default=4, help="extra leg: self-play moves with subtree reuse (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the root children of every game (rank 0's games under --gpus > 1) that the last "
                         "step returned as DIR/<name>.npy (float64, at most 64 MB: a seeded sample of games beyond that)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results; the reference arm runs in worker processes and returns none")
    if args.games is None:
        args.games = CHESS_GAMES_PER_GPU if args.game == "chess" else GAMES_PER_GPU
    if args.sims is None:
        args.sims = CHESS_SIMS if args.game == "chess" else SIMS
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:
        # not under torchrun: launch one rank per GPU ourselves
        import socket
        with socket.socket() as sk:
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    # stdout carries exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version there) are sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(json_fd, "w")
    if args.game == "chess":
        return run_chess_reference(args) if args.impl == "reference" else run_chess(args)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
