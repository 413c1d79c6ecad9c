"""bf16-faithful reference of the chess 10x256 network (csrc/chess_net.cu), for the numerics tests.

The same operations as the device, rounded where the device rounds and carried in float64 everywhere else, so that what
is left between the kernels and this reference is the f32 accumulation order of the tensor cores:
  * weights: BatchNorm folded as weights.cu::parse_safetensors_chess folds it (float64 product, cast to float32), then
    rounded to bf16 as chess_net.cu::f2bf rounds (nearest, ties to even); policy_conv1 / policy_conv2 are rounded without
    folding.  Biases, the value conv's 1x1 weights and fc1 / fc2 stay float32 (the f32 parameter block of net_upload);
  * input planes rounded to bf16 (k_encode_input): planes 17 (fifty / 100) and 18 ((plies / 2) / 50) are not exact;
  * every conv of the torso and the first policy conv: acc + bias (+ the bf16-stored block input), ReLU, stored as bf16;
  * the value head's 1x1 conv (`vcell`) is formed from the UNROUNDED ReLU output of the last torso conv
    (EPI_SKIP_RELU_VALUE), while the policy head reads the bf16-stored tensor;
  * logits: accumulator + bias, no rounding; k_value_head is f32 throughout (float64 here).
`rounding=False` turns every rounding point off (folded weights kept in float64): the network is then torch_net.ChessNet's
to float32 accuracy, a check of layouts, folding and head wiring that needs no GPU.
Runs on any torch device in float64; its speed is not measured.
"""
import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = float(np.float32(1e-5))          # NET_BN_EPS, a float widened to double in the fold


def f2bf_bits(f32_bits):
    """chess_net.cu::f2bf on the bit pattern of a float32 -> the bf16 bit pattern (inf / NaN are truncated)."""
    u = int(f32_bits) & 0xFFFFFFFF
    if (u & 0x7F800000) == 0x7F800000:
        return u >> 16
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFFFFFF
    return u >> 16


def bf16_round(t):
    """Rounds to float32, then to bf16 as f2bf does; returned in t's dtype."""
    u = t.to(torch.float32).view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    special = (u & 0x7F800000) == 0x7F800000
    r = torch.where(special, u, u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    r = torch.where(r >= 1 << 31, r - (1 << 32), r).to(torch.int32)
    return r.view(torch.float32).to(t.dtype)


class ChessNetRef:
    """The device arithmetic of one torch_net.ChessNet.  Tensors are attributes, so a test can perturb one of them."""

    def __init__(self, net, rounding=True, device="cpu", dtype=torch.float64):
        self.rounding, self.device, self.dtype = rounding, device, dtype
        d = lambda t: t.detach().to(torch.float64)                          # noqa: E731
        f32 = lambda t: t.to(torch.float32).to(torch.float64) if rounding else t   # noqa: E731
        bf = lambda t: bf16_round(t) if rounding else t                     # noqa: E731
        put = lambda t: t.to(device=device, dtype=dtype)                    # noqa: E731
        self.convs = []                                                      # (weight, bias) of the stem and 20 residual convs
        for conv, bn in net.conv_bn_pairs():
            s = d(bn.weight) / torch.sqrt(d(bn.running_var) + BN_EPS)
            w = bf(f32(d(conv.weight) * s[:, None, None, None]))
            b = f32((d(conv.bias) - d(bn.running_mean)) * s + d(bn.bias))
            self.convs.append((put(w), put(b)))
        self.p1w, self.p1b = put(bf(d(net.p1.weight))), put(d(net.p1.bias))
        self.p2w, self.p2b = put(bf(d(net.p2.weight))), put(d(net.p2.bias))
        self.vw, self.vb = put(d(net.vconv.weight).reshape(-1)), put(d(net.vconv.bias))
        self.f1w, self.f1b = put(d(net.fc1.weight)), put(d(net.fc1.bias))
        self.f2w, self.f2b = put(d(net.fc2.weight)), put(d(net.fc2.bias))

    def _bf(self, t):
        return bf16_round(t) if self.rounding else t

    def _conv(self, x, k, skip=None):
        w, b = self.convs[k]
        y = F.conv2d(x, w, padding=1) + b[None, :, None, None]
        return y if skip is None else y + skip

    def torso(self, enc):
        """-> (bf16-stored torso output, the last conv's ReLU output before it is stored)."""
        x = self._bf(torch.as_tensor(np.asarray(enc, np.float32)).to(device=self.device, dtype=self.dtype))
        x = self._bf(torch.relu(self._conv(x, 0)))
        for blk in range((len(self.convs) - 1) // 2):
            y = self._bf(torch.relu(self._conv(x, 1 + 2 * blk)))
            last = torch.relu(self._conv(y, 2 + 2 * blk, skip=x))
            x = self._bf(last)
        return x, last

    def vcell(self, last):
        """The value head's 1x1 conv before bias and ReLU, [n, 64] (EPI_SKIP_RELU_VALUE)."""
        return torch.einsum("nchw,c->nhw", last, self.vw).reshape(len(last), 64)

    def value(self, vcell):
        h = torch.relu(torch.relu(vcell + self.vb) @ self.f1w.T + self.f1b)
        return torch.tanh(h @ self.f2w.T + self.f2b).reshape(-1)

    def logits(self, x):
        y = self._bf(torch.relu(F.conv2d(x, self.p1w) + self.p1b[None, :, None, None]))
        return (F.conv2d(y, self.p2w) + self.p2b[None, :, None, None]).flatten(1)

    def forward(self, enc, chunk=512):
        """enc [n, 19, 8, 8] -> (logits [n, 4672], values [n]) as float64 numpy arrays."""
        lg, v = [], []
        with torch.no_grad():
            for i in range(0, len(enc), chunk):
                x, last = self.torso(enc[i:i + chunk])
                lg.append(self.logits(x).double().cpu().numpy())
                v.append(self.value(self.vcell(last)).double().cpu().numpy())
        return np.concatenate(lg), np.concatenate(v)
