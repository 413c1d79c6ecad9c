"""bf16-faithful reference of the Connect4 / tic-tac-toe network (csrc/evaluator_umma.cu, csrc/evaluator.cu), for the
numerics tests.

The same operations as the device, rounded where k_eval_umma rounds and carried in float64 everywhere else, so that what
is left between the kernels and this reference is the f32 accumulation order:
  * weights: BatchNorm folded as weights.cu::fold_conv folds it (float64 scale g / sqrt(var + eps), the product cast to
    float32), then rounded to bf16 as f2bf rounds (nearest, ties to even).  Conv biases stay float32, and so do the
    Linear layers' weights and biases (f32 in the weight image);
  * input: the three planes of get_encoding, exact in bf16;
  * the stem and every residual conv: acc + bias (+ the bf16-stored block input), ReLU, stored as bf16;
  * the head conv (32 policy + 3 value channels, one fused conv on the device): acc + bias, ReLU, stored as bf16;
  * the Linear heads over the flat index channel * P + row * C + col, then softmax over the A actions and tanh.
`rounding=False` turns every rounding point off (folded weights kept in float64): the network is then torch_net.Net's to
float32 accuracy, a check of folding, layouts and head wiring that needs no GPU.
Tensors and the head rounding are attributes, so that a test can perturb one of them.  Runs on any torch device in
float64; its speed is not measured.
"""
import numpy as np
import torch
import torch.nn.functional as F

from chess_net_ref import BN_EPS, bf16_round


class SmallNetRef:
    """The device arithmetic of one torch_net.Net (Connect4 or tic-tac-toe)."""

    def __init__(self, net, rounding=True, device="cpu", dtype=torch.float64):
        self.rows, self.cols, self.actions = net.rows, net.cols, net.actions
        self.rounding, self.round_head, self.device, self.dtype = rounding, rounding, device, dtype
        d = lambda t: t.detach().to(torch.float64)                          # noqa: E731
        f32 = lambda t: t.to(torch.float32).to(torch.float64) if rounding else t   # noqa: E731
        bf = lambda t: bf16_round(t) if rounding else t                     # noqa: E731
        put = lambda t: t.to(device=device, dtype=dtype)                    # noqa: E731
        folded = []
        for conv, bn in net.conv_bn_pairs():
            s = d(bn.weight) / torch.sqrt(d(bn.running_var) + BN_EPS)
            w = bf(f32(d(conv.weight) * s[:, None, None, None]))
            b = f32((d(conv.bias) - d(bn.running_mean)) * s + d(bn.bias))
            folded.append((put(w), put(b)))
        self.convs = folded[:-2]                                             # stem + 8 residual convs
        # the head conv: policy channels 0..31, value channels 32..34 (one conv of 35 output channels on the device)
        self.hw = torch.cat([folded[-2][0], folded[-1][0]])
        self.hb = torch.cat([folded[-2][1], folded[-1][1]])
        self.pw, self.pb = put(d(net.pfc.weight)), put(d(net.pfc.bias))
        self.vw, self.vb = put(d(net.vfc.weight)), put(d(net.vfc.bias))
        self.policy_ch = net.pconv.out_channels

    def _bf(self, t):
        return bf16_round(t) if self.rounding else t

    def _conv(self, x, k, skip=None):
        w, b = self.convs[k]
        y = F.conv2d(x, w, padding=1) + b[None, :, None, None]
        return y if skip is None else y + skip

    def torso(self, enc):
        """enc [n, 3, R, C] (or flat [n, 3 R C]) -> the bf16-stored output of the last residual block."""
        x = torch.as_tensor(np.asarray(enc, np.float32)).reshape(-1, 3, self.rows, self.cols)
        x = self._bf(x.to(device=self.device, dtype=self.dtype))
        x = self._bf(torch.relu(self._conv(x, 0)))
        for blk in range((len(self.convs) - 1) // 2):
            y = self._bf(torch.relu(self._conv(x, 1 + 2 * blk)))
            x = self._bf(torch.relu(self._conv(y, 2 + 2 * blk, skip=x)))
        return x

    def head(self, x):
        """The head conv's activations [n, 35, R, C]: policy channels, then value channels."""
        h = torch.relu(F.conv2d(x, self.hw, padding=1) + self.hb[None, :, None, None])
        return bf16_round(h) if self.round_head else h

    def linear(self, h):
        """-> (logits [n, A], the value before tanh [n])."""
        p = h[:, :self.policy_ch].flatten(1)
        v = h[:, self.policy_ch:].flatten(1)
        return p @ self.pw.T + self.pb, (v @ self.vw.T + self.vb).reshape(-1)

    def forward(self, enc, chunk=4096):
        """-> (logits [n, A], values [n]) as float64 numpy arrays."""
        lg, v = [], []
        with torch.no_grad():
            for i in range(0, len(enc), chunk):
                logit, z = self.linear(self.head(self.torso(enc[i:i + chunk])))
                lg.append(logit.double().cpu().numpy())
                v.append(torch.tanh(z).double().cpu().numpy())
        return np.concatenate(lg), np.concatenate(v)


def softmax(logits):
    """Softmax over the last axis in float64."""
    lg = np.asarray(logits, np.float64)
    e = np.exp(lg - lg.max(-1, keepdims=True))
    return e / e.sum(-1, keepdims=True)
