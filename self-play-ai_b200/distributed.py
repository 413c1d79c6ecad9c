"""Multi-GPU plumbing: games are sharded by rank (rank r owns global game ids r*G .. (r+1)*G-1 and every id
congruent to them modulo world*G); nothing is exchanged on the search path.  The one exchange of the path is
the variable-length gather of finished trajectories to the learner rank (SURVEY.md §8e), done with
torch.distributed (NCCL on GPUs, gloo in CPU tests): all-gather of per-rank counts, then one padded
all-gather of the records; the learner orders positions by (global game id, ply), which makes an R-rank run
byte-identical to a 1-rank run of the same games.
"""
from __future__ import annotations

import numpy as np

from .engine import POSITION_DTYPE


def shard_range(num_games_total: int, rank: int, world: int):
    """Contiguous partition of the global game ids [0, num_games_total) over ranks (ref: independent trees,
    mcts.rs:236 — no tree reads another)."""
    per = num_games_total // world
    extra = num_games_total % world
    lo = rank * per + min(rank, extra)
    return lo, lo + per + (1 if rank < extra else 0)


def merge_trajectories(parts, dtype=POSITION_DTYPE):
    """parts: list of (positions, game_ids[u64]) from every rank -> one (positions, ids) ordered by (game id, ply).  The
    record type is that of the parts (POSITION_DTYPE, chess.CHESS_POSITION_DTYPE); `dtype` types an empty result."""
    pos = np.concatenate([p for p, _ in parts]) if parts else np.zeros(0, dtype)
    ids = np.concatenate([g for _, g in parts]) if parts else np.zeros(0, np.uint64)
    order = np.lexsort((pos["ply"], ids))
    return pos[order], ids[order]


def gather_records(pos: np.ndarray, ids: np.ndarray, dst: int = 0, device=None, dtype=None):
    """Variable-length gather of (positions, game ids) to rank `dst` over the default process group.  The record type is
    that of `pos` (POSITION_DTYPE or chess.CHESS_POSITION_DTYPE), or `dtype` when given; every rank passes the same."""
    import torch
    import torch.distributed as dist

    dtype = np.dtype(dtype) if dtype is not None else (pos.dtype if pos.dtype.names else POSITION_DTYPE)
    world, rank = dist.get_world_size(), dist.get_rank()
    dev = device if device is not None else (torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu"))
    n = torch.tensor([len(pos)], dtype=torch.int64, device=dev)
    counts = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
    dist.all_gather(counts, n)
    counts = [int(c.item()) for c in counts]
    cap = max(1, max(counts))
    size = dtype.itemsize
    buf = np.zeros((cap, size + 8), np.uint8)
    if len(pos):
        buf[:len(pos), :size] = np.ascontiguousarray(pos, dtype=dtype).view(np.uint8).reshape(len(pos), -1)
        buf[:len(pos), size:] = np.ascontiguousarray(ids, dtype=np.uint64).view(np.uint8).reshape(len(pos), 8)
    mine = torch.from_numpy(buf).to(dev)
    out = [torch.zeros_like(mine) for _ in range(world)] if rank == dst else None
    dist.gather(mine, out, dst=dst)
    if rank != dst:
        return np.zeros(0, dtype), np.zeros(0, np.uint64)
    parts = []
    for r in range(world):
        a = out[r].cpu().numpy()[:counts[r]]
        p = np.ascontiguousarray(a[:, :size]).view(dtype).reshape(-1)
        g = np.ascontiguousarray(a[:, size:]).view(np.uint64).reshape(-1)
        parts.append((p, g))
    return merge_trajectories(parts, dtype)


def gather_trajectories(engine, dst: int = 0):
    """Drains this rank's finished trajectories and gathers them to the learner rank."""
    pos, ids = engine.drain_trajectories()
    return gather_records(pos, ids, dst=dst)


def comm_init_over_process_group(engine, rank: int | None = None, world: int | None = None):
    """Joins `engine` to a C-ABI communicator (spb_comm_init) spanning the default torch.distributed process group: rank 0
    creates the NCCL id (spb_comm_unique_id) and the process group only carries its 128 bytes.  A Rust host distributes the
    id by its own means (INTEGRATION.md)."""
    import torch.distributed as dist
    from .engine import comm_unique_id
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    box = [comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    engine.comm_init(box[0], rank, world)
