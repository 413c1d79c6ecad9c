"""Error of the evaluator kernels over several nets.  Connect4 / tic-tac-toe against the torch fp32 network: fresh (random
init, randomised BatchNorm) and trained-like (BatchNorm gammas 0.5..2, shifted statistics, larger heads); reported per net:
max |dlogit| / max |logit| (the bound of tests/test_gpu_evaluator.py), the worst per-position relative L2 error of the logit
vector, the largest change of a softmax probability, max |dvalue|.  The chess 10x256 network, fresh (seed 0) and calibrated
(make_chess_net(calibrated=True)), on the 4,096 distinct positions of tests/test_net_numerics.py at every batch size of
its tile-loop regimes, against the bf16-faithful reference (tests/chess_net_ref.py; |dlogit| over the logit's
position-dependent spread, the bound of that test) and against torch fp32.  Connect4 / tic-tac-toe again, on the nets,
positions and batch sizes of tests/test_eval_numerics.py, per kernel: against the bf16-faithful reference
(tests/small_net_ref.py; the metrics of that test) next to torch fp32.  Needs a B200; prints the card and its power
limit first."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np  # noqa: E402

import selfplay_b200 as S  # noqa: E402
from helpers import random_states  # noqa: E402
from oracle import pyoracle as O, torch_net  # noqa: E402

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip(),
      flush=True)


def report(tag, lg, v, logit_ref, v_ref):
    scale = float(np.abs(logit_ref).max())
    rel_l2 = np.linalg.norm(lg - logit_ref, axis=1) / np.maximum(np.linalg.norm(logit_ref, axis=1), 1e-6)
    sm = lambda x: np.exp(x - x.max(1, keepdims=True)) / np.exp(x - x.max(1, keepdims=True)).sum(1, keepdims=True)   # noqa: E731
    print("%s (logit scale %.3f): max|dlogit|/scale %.2e | worst rel L2 per position %.2e | max|dp| %.2e | max|dvalue| %.2e" % (
        tag, scale, np.abs(lg - logit_ref).max() / scale, rel_l2.max(), np.abs(sm(lg) - sm(logit_ref)).max(), np.abs(v - v_ref).max()), flush=True)


for game, tag in ((S.GAME_C4, "c4"), (S.GAME_TTT, "ttt")):
    for trained in (False, True):
        for seed in range(4):
            net = torch_net.make_net(game, seed=seed, trained_like=trained)
            states = random_states(game, 1500, seed=100 + seed, include_terminal=False)
            enc = np.stack([O.encode(game, s) for s in states])
            _, v_ref, logit_ref = torch_net.forward_probs(net, enc)
            for flags, name in ((0, "tcgen05"), (S.FLAG_EVAL_SIMT, "simt")):
                with S.Engine(game=game, num_games=4, evaluator=S.EVAL_NET, flags=flags) as e:
                    e.load_weights(torch_net.to_safetensors_tch(net))
                    _, v, lg = e.predict(states, want_logits=True)
                report("%s %s seed %d %s" % (tag, "trained-like" if trained else "fresh", seed, name), lg, v, logit_ref, v_ref)

import torch  # noqa: E402

import chess_net_ref as R  # noqa: E402
import test_net_numerics as T  # noqa: E402

torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False
with S.ChessEngine(num_games=T.G, evaluator=S.EVAL_NET) as e:
    st, hist = T.distinct_positions(e, T.G)
    enc = e.encode(st, hist)
    pairs = T.conv_pairs(T.G, torch.cuda.get_device_properties(0).multi_processor_count)
    for name, kw in T.NETS.items():
        net = torch_net.make_chess_net(**kw)
        ref_lg, ref_v = R.ChessNetRef(net, device="cuda").forward(enc)
        spread = ref_lg.std(0)
        with torch.no_grad():
            out = [net.cuda()(torch.from_numpy(enc[i:i + 512]).cuda()) for i in range(0, T.G, 512)]
        lg32 = torch.cat([o[0] for o in out]).cpu().numpy()
        v32 = torch.cat([o[1] for o in out]).reshape(-1).cpu().numpy()
        e.load_weights(torch_net.chess_to_safetensors_explicit(net.cpu()))
        print("chess 10x256 %s: value std %.3f, logit scale %.1f, position-dependent logit spread %.3g (median per logit %.3g)" % (
            name, ref_v.std(), np.abs(ref_lg).max(), torch_net.chess_logit_deviation(ref_lg), np.median(spread)), flush=True)
        for n in T.batch_sizes(pairs):
            _, v, lg = e.predict(st[:n], hist[:n], want_logits=True)
            r = np.abs(lg - ref_lg[:n]) / spread
            dv = np.abs(v - ref_v[:n])
            print("  n %4d it<=%2d | vs bf16 reference: |dlogit|/spread max %.2e p99.99 %.2e median %.2e; |dv| max %.2e p99 %.2e "
                  "| vs fp32: max|dlogit|/scale %.2e |dlogit|/spread max %.2e |dv| max %.2e" % (
                      n, T.max_pass(n, pairs), r.max(), np.quantile(r, 0.9999), np.median(r), dv.max(), np.quantile(dv, 0.99),
                      np.abs(lg - lg32[:n]).max() / np.abs(lg32[:n]).max(), (np.abs(lg - lg32[:n]) / spread).max(),
                      np.abs(v - v32[:n]).max()), flush=True)

# ---- Connect4 / tic-tac-toe against the bf16-faithful reference (tests/small_net_ref.py) --------------------------------
import small_net_ref as SR  # noqa: E402
import test_eval_numerics as EN  # noqa: E402

sms = torch.cuda.get_device_properties(0).multi_processor_count
for tag in EN.GAMES:
    for name in EN.NETS:
        c = EN.case(tag, name)
        _, v32, lg32 = torch_net.forward_probs(c["net"], c["enc"])
        print("%s %s: %d positions, value std %.3f, logit scale %.2f, position-dependent logit spread %.3g (median per logit %.3g)" % (
            tag, name, len(c["enc"]), c["ref_v"].std(), np.abs(c["ref_lg"]).max(), torch_net.chess_logit_deviation(c["ref_lg"]),
            np.median(c["spread"])), flush=True)
        for kernel, flags in EN.KERNELS.items():
            with S.Engine(game=EN.GAMES[tag], num_games=4, evaluator=S.EVAL_NET, flags=flags) as e:
                e.load_weights(c["blob"])
                for n in [len(c["enc"])] + EN.batch_sizes(EN.GAMES[tag], sms):
                    idx = np.arange(n) % len(c["enc"])
                    pol, v, lg = e.predict(c["states"][idx], want_logits=True)
                    m = EN.metrics(c, lg, v, pol, idx=idx)
                    print("  %-7s n %5d | vs bf16 reference: |dlogit|/spread max %.2e, position RMS max %.2e median %.2e, |dv| max %.2e, |dp| max %.2e "
                          "| vs fp32: max|dlogit|/scale %.2e |dv| max %.2e" % (
                              (kernel, n) + m + (np.abs(lg - lg32[idx]).max() / np.abs(lg32[idx]).max(), np.abs(v - v32[idx]).max())), flush=True)
