"""PyTorch fp32 restatement of the reference's policy/value nets (test infrastructure).

ref: src/model/mod.rs:152-184 (resnet_block / new_resnet), src/model/connect_four.rs:50-81,
src/model/tictactoe.rs:50-81.  tch is a libtorch binding, so torch CPU fp32 is the same arithmetic
library the reference calls.  Also writes safetensors files with the names tch's VarStore produces
when every layer is created on the root path (name de-duplication by "__{count}" suffix).
"""
import io
import struct
import json

import numpy as np
import torch
import torch.nn as nn


class ResBlock(nn.Module):
    def __init__(self, h):
        super().__init__()
        self.conv1 = nn.Conv2d(h, h, 3, padding=1)
        self.bn1 = nn.BatchNorm2d(h)
        self.conv2 = nn.Conv2d(h, h, 3, padding=1)
        self.bn2 = nn.BatchNorm2d(h)

    def forward(self, x):
        f = self.bn2(self.conv2(torch.relu(self.bn1(self.conv1(x)))))
        return torch.relu(x + f)


class Net(nn.Module):
    """Connect4: rows=6, cols=7, actions=7.  Tic-tac-toe: 3, 3, 9."""

    def __init__(self, rows, cols, actions, blocks=4, hidden=64):
        super().__init__()
        self.rows, self.cols, self.actions = rows, cols, actions
        self.stem = nn.Conv2d(3, hidden, 3, padding=1)
        self.stem_bn = nn.BatchNorm2d(hidden)
        self.blocks = nn.ModuleList([ResBlock(hidden) for _ in range(blocks)])
        self.pconv = nn.Conv2d(hidden, 32, 3, padding=1)
        self.pbn = nn.BatchNorm2d(32)
        self.pfc = nn.Linear(32 * rows * cols, actions)
        self.vconv = nn.Conv2d(hidden, 3, 3, padding=1)
        self.vbn = nn.BatchNorm2d(3)
        self.vfc = nn.Linear(3 * rows * cols, 1)

    def forward(self, x):
        x = x.view(-1, 3, self.rows, self.cols)
        x = torch.relu(self.stem_bn(self.stem(x)))
        for b in self.blocks:
            x = b(x)
        p = self.pfc(torch.relu(self.pbn(self.pconv(x))).flatten(1))
        v = torch.tanh(self.vfc(torch.relu(self.vbn(self.vconv(x))).flatten(1)))
        return p, v

    def conv_bn_pairs(self):
        pairs = [(self.stem, self.stem_bn)]
        for b in self.blocks:
            pairs += [(b.conv1, b.bn1), (b.conv2, b.bn2)]
        pairs += [(self.pconv, self.pbn), (self.vconv, self.vbn)]
        return pairs


def make_net(game, seed=0, randomize_bn=True, trained_like=False, calibrated=False):
    """game: 0 tic-tac-toe, 1 connect4.  Default torch init under manual_seed; BN running stats and affine
    parameters are randomised (when asked) so that BN folding is actually exercised.  trained_like: statistics of a net
    that has been trained for a while instead of a fresh one — BatchNorm gammas spread over 0.5..2, shifted and scaled
    running statistics, larger head weights (logits of several units, tanh driven towards saturation).
    calibrated: the counterpart of make_chess_net(calibrated=True), calibrated on calibration_encodings(game).  BatchNorm
    gammas 0.5..2 and shifted betas, running statistics that are those of the conv outputs they normalise (head convs
    included); value_fc scaled so that the value before tanh has mean 0 and standard deviation 0.8, and every row of
    policy_fc so that its logit's position-dependent part (the logit minus its mean over the positions) has standard
    deviation 1.  A fresh or trained-like net's value hardly depends on the position (standard deviation 0.02 over
    random positions), so a comparison against it cannot see the value head."""
    rows, cols, actions = (6, 7, 7) if game == 1 else (3, 3, 9)
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    net = Net(rows, cols, actions).eval()
    if calibrated:
        with torch.no_grad():
            for _, bn in net.conv_bn_pairs():
                bn.weight.copy_(torch.rand(bn.num_features, generator=g) * 1.5 + 0.5)
                bn.bias.copy_(torch.randn(bn.num_features, generator=g) * 0.3)
            _calibrate_net(net, calibration_encodings(game))
        return net
    if trained_like:
        with torch.no_grad():
            for _, bn in net.conv_bn_pairs():
                bn.running_mean.copy_(torch.randn(bn.num_features, generator=g) * 0.5)
                bn.running_var.copy_(torch.rand(bn.num_features, generator=g) * 1.8 + 0.2)
                bn.weight.copy_(torch.rand(bn.num_features, generator=g) * 1.5 + 0.5)
                bn.bias.copy_(torch.randn(bn.num_features, generator=g) * 0.3)
            net.pfc.weight.mul_(4.0)
            net.vfc.weight.mul_(2.0)
        return net
    if randomize_bn:
        with torch.no_grad():
            for _, bn in net.conv_bn_pairs():
                bn.running_mean.copy_(torch.randn(bn.num_features, generator=g) * 0.1)
                bn.running_var.copy_(torch.rand(bn.num_features, generator=g) * 0.5 + 0.75)
                bn.weight.copy_(torch.rand(bn.num_features, generator=g) * 0.5 + 0.75)
                bn.bias.copy_(torch.randn(bn.num_features, generator=g) * 0.1)
    return net


def calibration_states(game, n=256, seed=97):
    """n fixed ongoing positions: the position after a uniform random playout of a random length (oracle rules, seeded)."""
    from . import pyoracle as O
    rng = np.random.default_rng(seed)
    max_len = 42 if game == O.GAME_C4 else 9
    out = []
    while len(out) < n:
        s = O.State()
        for _ in range(int(rng.integers(0, max_len))):
            s = O.next_state(game, s, int(rng.choice(O.valid_actions(game, s))))
            if s.status != O.ONGOING:
                break
        if s.status == O.ONGOING:
            out.append(s)
    return out


def calibration_encodings(game, n=256, seed=97):
    from . import pyoracle as O
    return np.stack([O.encode(game, s) for s in calibration_states(game, n, seed)])


def _calibrate_net(net, enc):
    def bn_from(conv, bn, x):
        u = conv(x)
        bn.running_mean.copy_(u.mean((0, 2, 3)))
        bn.running_var.copy_(u.var((0, 2, 3)))
        return bn(u)
    x = torch.from_numpy(np.ascontiguousarray(enc, dtype=np.float32)).view(-1, 3, net.rows, net.cols)
    x = torch.relu(bn_from(net.stem, net.stem_bn, x))
    for b in net.blocks:
        x = torch.relu(x + bn_from(b.conv2, b.bn2, torch.relu(bn_from(b.conv1, b.bn1, x))))
    z = net.vfc(torch.relu(bn_from(net.vconv, net.vbn, x)).flatten(1))
    m, s = z.mean(), z.std() / 0.8
    net.vfc.weight.div_(s)
    net.vfc.bias.sub_(m).div_(s)
    lg = net.pfc(torch.relu(bn_from(net.pconv, net.pbn, x)).flatten(1))
    net.pfc.weight.div_(lg.std(0)[:, None])


def _write_safetensors(tensors):
    """tensors: list[(name, np.ndarray f32)] in file order."""
    header, off, chunks = {}, 0, []
    for name, arr in tensors:
        arr = np.ascontiguousarray(arr, dtype=np.float32)
        b = arr.tobytes()
        header[name] = {"dtype": "F32", "shape": list(arr.shape), "data_offsets": [off, off + len(b)]}
        off += len(b)
        chunks.append(b)
    hj = json.dumps(header, separators=(",", ":")).encode()
    hj += b" " * ((8 - len(hj) % 8) % 8)
    return struct.pack("<Q", len(hj)) + hj + b"".join(chunks)


def to_safetensors_explicit(net) -> bytes:
    out = []
    for i, (conv, bn) in enumerate(net.conv_bn_pairs()):
        out += [("conv%d.weight" % i, conv.weight), ("conv%d.bias" % i, conv.bias), ("bn%d.weight" % i, bn.weight),
                ("bn%d.bias" % i, bn.bias), ("bn%d.running_mean" % i, bn.running_mean), ("bn%d.running_var" % i, bn.running_var)]
    out += [("policy_fc.weight", net.pfc.weight), ("policy_fc.bias", net.pfc.bias),
            ("value_fc.weight", net.vfc.weight), ("value_fc.bias", net.vfc.bias)]
    return _write_safetensors([(n, t.detach().numpy()) for n, t in out])


def to_safetensors_tch(net, bn_order=("weight", "bias", "running_mean", "running_var"), shuffle_seed=None) -> bytes:
    """Names as tch's VarStore makes them when all layers share the root path: the first variable called
    `weight` keeps its name, later ones become `weight__{number of variables created so far}`."""
    created = []   # (base name, tensor) in creation order
    def conv(c):
        created.extend([("bias", c.bias), ("weight", c.weight)])
    def bn(b):
        for k in bn_order:
            created.append((k, getattr(b, k)))
    def linear(l):
        created.extend([("bias", l.bias), ("weight", l.weight)])
    pairs = net.conv_bn_pairs()
    for c, b in pairs[:-2]:
        conv(c); bn(b)
    conv(net.pconv); bn(net.pbn); linear(net.pfc)
    conv(net.vconv); bn(net.vbn); linear(net.vfc)
    named, seen = [], set()
    for base, t in created:
        name = base if base not in seen else "%s__%d" % (base, len(named))
        seen.add(base)
        named.append((name, t.detach().numpy()))
    if shuffle_seed is not None:   # file order is not creation order (safetensors sorts by dtype/name)
        rng = np.random.default_rng(shuffle_seed)
        named = [named[i] for i in rng.permutation(len(named))]
    return _write_safetensors(named)


def forward_probs(net, enc):
    """The tensor part of Model::predict (model/mod.rs:60-67,95): softmax(logits), value."""
    with torch.no_grad():
        x = torch.from_numpy(np.ascontiguousarray(enc, dtype=np.float32))
        p, v = net(x)
        return torch.softmax(p, -1).numpy(), v.reshape(-1).numpy(), p.numpy()


def load_tch_safetensors(blob: bytes, game: int):
    """Builds the torch net from a tch-style checkpoint (names de-duplicated with "__{n}", creation order)."""
    hlen = struct.unpack("<Q", blob[:8])[0]
    header = json.loads(blob[8:8 + hlen])
    data = blob[8 + hlen:]
    items = []
    for name, meta in header.items():
        if name == "__metadata__":
            continue
        base, _, idx = name.partition("__")
        arr = np.frombuffer(data[meta["data_offsets"][0]:meta["data_offsets"][1]], dtype=np.float32).reshape(meta["shape"])
        items.append((int(idx) if idx else -1, base, arr))
    items.sort(key=lambda t: t[0])
    rows, cols, actions = (6, 7, 7) if game == 1 else (3, 3, 9)
    net = Net(rows, cols, actions).eval()
    it = iter(items)
    def take(n):
        got = {}
        for _ in range(n):
            _, base, arr = next(it)
            got[base] = torch.from_numpy(arr.copy())
        return got
    with torch.no_grad():
        def fill_conv(c):
            g = take(2); c.weight.copy_(g["weight"]); c.bias.copy_(g["bias"])
        def fill_bn(b):
            g = take(4); b.weight.copy_(g["weight"]); b.bias.copy_(g["bias"]); b.running_mean.copy_(g["running_mean"]); b.running_var.copy_(g["running_var"])
        pairs = net.conv_bn_pairs()
        for c, b in pairs[:-2]:
            fill_conv(c); fill_bn(b)
        fill_conv(net.pconv); fill_bn(net.pbn); fill_conv(net.pfc)
        fill_conv(net.vconv); fill_bn(net.vbn); fill_conv(net.vfc)
    return net


# ---- chess (ref: src/model/chess.rs:50-83) ---------------------------------------------------------------------------

class ChessNet(nn.Module):
    """19 -> 256 stem, 10 residual blocks, policy head conv1x1 256 -> 256, ReLU, conv1x1 256 -> 73 (flat 73*8*8), value head
    conv1x1 256 -> 1, ReLU, Linear 64 -> 256, ReLU, Linear 256 -> 1, tanh."""

    def __init__(self, blocks=10, hidden=256):
        super().__init__()
        self.stem = nn.Conv2d(19, hidden, 3, padding=1)
        self.stem_bn = nn.BatchNorm2d(hidden)
        self.blocks = nn.ModuleList([ResBlock(hidden) for _ in range(blocks)])
        self.p1 = nn.Conv2d(hidden, 256, 1)
        self.p2 = nn.Conv2d(256, 73, 1)
        self.vconv = nn.Conv2d(hidden, 1, 1)
        self.fc1 = nn.Linear(64, 256)
        self.fc2 = nn.Linear(256, 1)

    def forward(self, x):
        x = x.view(-1, 19, 8, 8)
        x = torch.relu(self.stem_bn(self.stem(x)))
        for b in self.blocks:
            x = b(x)
        p = self.p2(torch.relu(self.p1(x))).flatten(1)
        v = torch.tanh(self.fc2(torch.relu(self.fc1(torch.relu(self.vconv(x)).flatten(1)))))
        return p, v

    def conv_bn_pairs(self):
        pairs = [(self.stem, self.stem_bn)]
        for b in self.blocks:
            pairs += [(b.conv1, b.bn1), (b.conv2, b.bn2)]
        return pairs


def make_chess_net(seed=0, randomize_bn=True, blocks=10, calibrated=False):
    """calibrated: the counterpart of make_net(trained_like=True), calibrated on chess_calibration_encodings().  BatchNorm
    as after training: gammas 0.5..2, shifted betas, and running statistics that are those of the conv outputs they normalise
    (random statistics would make the torso blow small differences up, which a trained torso does not).  Heads: the value
    conv's pre-activation is standardised, fc2's pre-tanh scaled to mean 0 and standard deviation 0.8 (values spread over
    (-1, 1), some near saturation), and policy_conv2 scaled so that the position-dependent part of the logits (each logit
    minus its mean over the positions) has standard deviation 1.  A fresh net's value is nearly constant and its logits
    barely depend on the position, so a comparison against it cannot see the heads."""
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    net = ChessNet(blocks=blocks).eval()
    if calibrated:
        with torch.no_grad():
            for _, bn in net.conv_bn_pairs():
                bn.weight.copy_(torch.rand(bn.num_features, generator=g) * 1.5 + 0.5)
                bn.bias.copy_(torch.randn(bn.num_features, generator=g) * 0.3)
            _calibrate_chess_net(net, chess_calibration_encodings())
        return net
    if randomize_bn:
        with torch.no_grad():
            for _, bn in net.conv_bn_pairs():
                bn.running_mean.copy_(torch.randn(bn.num_features, generator=g) * 0.1)
                bn.running_var.copy_(torch.rand(bn.num_features, generator=g) * 0.5 + 0.75)
                bn.weight.copy_(torch.rand(bn.num_features, generator=g) * 0.5 + 0.75)
                bn.bias.copy_(torch.randn(bn.num_features, generator=g) * 0.1)
    return net


def chess_calibration_encodings(n=64, seed=97):
    """Encodings of n fixed positions: the position after a random playout of 0..99 plies (oracle rules, seeded)."""
    from . import pychess
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        g = pychess.Game()
        for _ in range(int(rng.integers(0, 100))):
            lm = g.legal_moves()
            if g.status() != 0 or not lm:
                break
            g.make_move(int(lm[rng.integers(len(lm))]))
        if g.status() == 0:
            out.append(g.encode())
    return np.stack(out)


def _calibrate_chess_net(net, enc):
    def bn_from(conv, bn, x):
        u = conv(x)
        bn.running_mean.copy_(u.mean((0, 2, 3)))
        bn.running_var.copy_(u.var((0, 2, 3)))
        return bn(u)
    x = torch.from_numpy(np.ascontiguousarray(enc, dtype=np.float32))
    x = torch.relu(bn_from(net.stem, net.stem_bn, x))
    for b in net.blocks:
        x = torch.relu(x + bn_from(b.conv2, b.bn2, torch.relu(bn_from(b.conv1, b.bn1, x))))
    u = net.vconv(x)
    m, s = u.mean(), u.std()
    net.vconv.weight.div_(s)
    net.vconv.bias.sub_(m).div_(s)
    z = net.fc2(torch.relu(net.fc1(torch.relu(net.vconv(x)).flatten(1))))
    m, s = z.mean(), z.std() / 0.8
    net.fc2.weight.div_(s)
    net.fc2.bias.sub_(m).div_(s)
    lg = net.p2(torch.relu(net.p1(x))).flatten(1)
    net.p2.weight.div_((lg - lg.mean(0)).std())


def chess_logit_deviation(logits):
    """Standard deviation of the position-dependent part of the logits: each logit minus its mean over the positions."""
    lg = np.asarray(logits, np.float64)
    return float((lg - lg.mean(0)).std())


def chess_to_safetensors_explicit(net) -> bytes:
    out = []
    for i, (conv, bn) in enumerate(net.conv_bn_pairs()):
        out += [("conv%d.weight" % i, conv.weight), ("conv%d.bias" % i, conv.bias), ("bn%d.weight" % i, bn.weight),
                ("bn%d.bias" % i, bn.bias), ("bn%d.running_mean" % i, bn.running_mean), ("bn%d.running_var" % i, bn.running_var)]
    for name, m in (("policy_conv1", net.p1), ("policy_conv2", net.p2), ("value_conv", net.vconv), ("value_fc1", net.fc1), ("value_fc2", net.fc2)):
        out += [(name + ".weight", m.weight), (name + ".bias", m.bias)]
    return _write_safetensors([(n, t.detach().numpy()) for n, t in out])


def chess_to_safetensors_tch(net, shuffle_seed=None) -> bytes:
    """tch VarStore names with every layer on the root path (model/chess.rs:55-71): creation order torso, policy head, value head."""
    created = []
    def wb(m):
        created.extend([("bias", m.bias), ("weight", m.weight)])
    for c, b in net.conv_bn_pairs():
        wb(c)
        for k in ("weight", "bias", "running_mean", "running_var"):
            created.append((k, getattr(b, k)))
    for m in (net.p1, net.p2, net.vconv, net.fc1, net.fc2):
        wb(m)
    named, seen = [], set()
    for base, t in created:
        name = base if base not in seen else "%s__%d" % (base, len(named))
        seen.add(base)
        named.append((name, t.detach().numpy()))
    if shuffle_seed is not None:
        rng = np.random.default_rng(shuffle_seed)
        named = [named[i] for i in rng.permutation(len(named))]
    return _write_safetensors(named)


def chess_forward(net, enc):
    """-> (softmax over the 4,672 cells, values, raw logits)."""
    with torch.no_grad():
        x = torch.from_numpy(np.ascontiguousarray(enc, dtype=np.float32))
        p, v = net(x)
        return torch.softmax(p, -1).numpy(), v.reshape(-1).numpy(), p.numpy()


def load_chess_tch_safetensors(blob: bytes):
    """Builds the torch chess net from a tch-style checkpoint (creation-order names)."""
    hlen = struct.unpack("<Q", blob[:8])[0]
    header = json.loads(blob[8:8 + hlen])
    data = blob[8 + hlen:]
    items = []
    for name, meta in header.items():
        if name == "__metadata__":
            continue
        base, _, idx = name.partition("__")
        arr = np.frombuffer(data[meta["data_offsets"][0]:meta["data_offsets"][1]], dtype=np.float32).reshape(meta["shape"])
        items.append((int(idx) if idx else -1, base, arr))
    items.sort(key=lambda t: t[0])
    net = ChessNet().eval()
    it = iter(items)

    def take(n):
        got = {}
        for _ in range(n):
            _, base, arr = next(it)
            got[base] = torch.from_numpy(arr.copy())
        return got
    with torch.no_grad():
        def fill_wb(m):
            g = take(2); m.weight.copy_(g["weight"]); m.bias.copy_(g["bias"])
        for c, b in net.conv_bn_pairs():
            fill_wb(c)
            g = take(4); b.weight.copy_(g["weight"]); b.bias.copy_(g["bias"]); b.running_mean.copy_(g["running_mean"]); b.running_var.copy_(g["running_var"])
        for m in (net.p1, net.p2, net.vconv, net.fc1, net.fc2):
            fill_wb(m)
    return net
