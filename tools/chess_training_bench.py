"""Chess training tensors from self-play records: the host builder against the device builder (one JSON line on stdout).

Records come from real self-play: 1,024 games from the bench's synthetic roots with their history filled to 500 plies, so
that every game ends at the history cap within 13 plies (DetEval, 64 simulations a move).  They are replicated to the sizes
below; nothing is downloaded.  A record is 1,624 bytes, its tensors 19*64*4 + 4,672*4 + 4 = 23,556 bytes.
  (1) host: spb_chess_positions_to_training on --host-rows rows, wall clock.
  (2) device: spb_chess_positions_to_training_device on --rows rows held in device memory (outputs of 23,556 bytes a row,
      6.2 GB at the default, far more than the 126 MB L2), warmed up, then --iters calls between CUDA events.  Each call is
      the validation kernel, a 8-byte read back, and the writer kernel.  A torch.profiler pass afterwards gives the device
      time of each kernel; GB/s written are output bytes over the writer kernel's time, and the share is of the 6,545 GB/s
      HBM rate measured in DESIGN.md section 4.1.
  (3) PCIe: copying the --host-rows records from pinned host memory against copying their host-built tensors.
  (4) minibatches: --batch random indices into a device-resident buffer of --buffer records, microseconds per call.

usage: python tools/chess_training_bench.py [--rows 262144] [--iters 20] [--host-rows 32768] [--buffer 1048576] [--batch 4096]
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

HBM_GBS = 6545.0                                                       # DESIGN.md section 4.1, measured on this board
REC_BYTES, OUT_BYTES = 1624, 19 * 64 * 4 + 4672 * 4 + 4


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception as ex:                                           # the numbers are still printed, without the card
        return "unknown (%s)" % ex, "unknown"


def selfplay_records(S, CH, games):
    from selfplay_b200.synth import synthetic_chess_roots_device
    with CH.ChessEngine(num_games=games, evaluator=S.EVAL_DET) as e:
        st, hist = synthetic_chess_roots_device(e, games)
        rng = np.random.default_rng(9)
        for i in range(games):
            h0 = int(st[i]["hist_len"])
            hist[i, h0:500] = rng.integers(1 << 40, 1 << 62, 500 - h0, dtype=np.uint64)
            st[i]["hist_len"] = 500
        e.reset_games(st, hist)
        for _ in range(13):
            e.search(64)
            e.selfplay_step(S.MOVE_GREEDY_LAST_MAX)
        pos, _ = e.drain_trajectories()
    return pos


def replicate(pos, n):
    return np.ascontiguousarray(np.resize(pos, n))


def kernel_times_us(torch, fn, calls):
    """Device time per launch of each k_chess_training* kernel over `calls` calls of fn, by torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "k_chess_training" in ev.key:
            total = getattr(ev, "device_time_total", None)
            if total is None:
                total = ev.cuda_time_total
            name = "check" if "check" in ev.key else "writer"
            out[name] = total / max(ev.count, 1)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--games", type=int, default=1024)
    ap.add_argument("--rows", type=int, default=262144)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--host-rows", type=int, default=32768)
    ap.add_argument("--buffer", type=int, default=1 << 20)
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--batches", type=int, default=200)
    a = ap.parse_args()

    import torch

    import selfplay_b200 as S
    CH = S.chess
    assert torch.cuda.is_available(), "the device builder runs on the GPU; there is no CPU fallback"
    name, limit = card()
    base = selfplay_records(S, CH, a.games)
    res = dict(tool="chess_training_bench", gpu=name, power_limit=limit, selfplay_games=a.games, selfplay_records=len(base),
               record_bytes=REC_BYTES, tensor_bytes_per_row=OUT_BYTES)

    # (1) host builder
    host = replicate(base, a.host_rows)
    CH.positions_to_training(host[:1024])
    t0 = time.perf_counter()
    want = CH.positions_to_training(host)
    t_host = time.perf_counter() - t0
    res.update(host_rows=a.host_rows, host_s=t_host, host_rows_per_s=a.host_rows / t_host, host_gb_per_s_written=a.host_rows * OUT_BYTES / t_host / 1e9)

    with CH.ChessEngine(num_games=1, evaluator=S.EVAL_DET) as e:
        # the device builder reproduces the host builder on these rows
        got = CH.positions_to_training_device(e, host)
        res["device_equals_host"] = all(np.array_equal(g.cpu().numpy().view(np.uint32), w.view(np.uint32)) for g, w in zip(got, want))
        del got

        # (2) device builder, whole buffer
        recs = torch.from_numpy(replicate(base, a.rows).view(np.uint8).reshape(a.rows, REC_BYTES)).cuda()
        enc = torch.empty((a.rows, 19, 8, 8), dtype=torch.float32, device="cuda")
        pol = torch.empty((a.rows, 4672), dtype=torch.float32, device="cuda")
        val = torch.empty((a.rows, 1), dtype=torch.float32, device="cuda")
        L = S.load_library()

        def call(pos_t, n_pos, idx, n, outs):
            rc = L.spb_chess_positions_to_training_device(e._h, pos_t.data_ptr(), n_pos, None if idx is None else idx.data_ptr(), n,
                                                           outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr())
            assert rc == 0, L.spb_chess_last_error(e._h).decode()

        torch.cuda.synchronize()
        for _ in range(3):
            call(recs, a.rows, None, a.rows, (enc, pol, val))
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(a.iters):
            call(recs, a.rows, None, a.rows, (enc, pol, val))
        ev1.record()
        torch.cuda.synchronize()
        call_ms = ev0.elapsed_time(ev1) / a.iters
        k = kernel_times_us(torch, lambda: call(recs, a.rows, None, a.rows, (enc, pol, val)), 5)
        out_bytes = a.rows * OUT_BYTES
        res.update(device_rows=a.rows, device_output_gb=out_bytes / 1e9, device_iters=a.iters, device_call_ms=call_ms,
                   device_call_gb_per_s_written=out_bytes / (call_ms * 1e-3) / 1e9,
                   check_kernel_us=k.get("check"), writer_kernel_us=k.get("writer"))
        if k.get("writer"):
            gbs = out_bytes / (k["writer"] * 1e-6) / 1e9
            res.update(writer_gb_per_s_written=gbs, writer_gb_per_s_moved=a.rows * (OUT_BYTES + REC_BYTES) / (k["writer"] * 1e-6) / 1e9,
                       writer_share_of_measured_hbm=gbs / HBM_GBS)
        del enc, pol, val, recs
        torch.cuda.empty_cache()

        # (3) PCIe: records against host-built tensors, from pinned memory
        rec_h = torch.from_numpy(host.view(np.uint8).reshape(len(host), REC_BYTES)).pin_memory()
        ten_h = [torch.from_numpy(w).pin_memory() for w in want]
        rec_d = torch.empty_like(rec_h, device="cuda")
        ten_d = [torch.empty_like(t, device="cuda") for t in ten_h]

        def timed(fn, reps=10):
            fn()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(reps):
                fn()
            ev1.record()
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1) / reps

        rec_ms = timed(lambda: rec_d.copy_(rec_h, non_blocking=True))
        ten_ms = timed(lambda: [d.copy_(h, non_blocking=True) for d, h in zip(ten_d, ten_h)])
        res.update(h2d_rows=len(host), h2d_records_ms=rec_ms, h2d_tensors_ms=ten_ms,
                   h2d_records_gb_per_s=rec_h.numel() / (rec_ms * 1e-3) / 1e9,
                   h2d_tensors_gb_per_s=sum(t.numel() * 4 for t in ten_h) / (ten_ms * 1e-3) / 1e9)
        del rec_h, ten_h, rec_d, ten_d

        # (4) minibatches from a device-resident replay buffer
        buf = torch.from_numpy(replicate(base, a.buffer).view(np.uint8).reshape(a.buffer, REC_BYTES)).cuda()
        gen = torch.Generator(device="cuda").manual_seed(5)
        idx = torch.randint(0, a.buffer, (a.batches, a.batch), device="cuda", generator=gen, dtype=torch.int64)
        outs = (torch.empty((a.batch, 19, 8, 8), device="cuda"), torch.empty((a.batch, 4672), device="cuda"), torch.empty((a.batch, 1), device="cuda"))
        torch.cuda.synchronize()
        for b in range(5):
            call(buf, a.buffer, idx[b], a.batch, outs)
        ev0.record()
        for b in range(a.batches):
            call(buf, a.buffer, idx[b], a.batch, outs)
        ev1.record()
        torch.cuda.synchronize()
        mb_us = ev0.elapsed_time(ev1) * 1e3 / a.batches
        kb = kernel_times_us(torch, lambda: call(buf, a.buffer, idx[0], a.batch, outs), 20)
        res.update(minibatch_buffer_records=a.buffer, minibatch_rows=a.batch, minibatch_calls=a.batches, minibatch_call_us=mb_us,
                   minibatch_check_kernel_us=kb.get("check"), minibatch_writer_kernel_us=kb.get("writer"),
                   minibatch_rows_per_s=a.batch / (mb_us * 1e-6))
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
