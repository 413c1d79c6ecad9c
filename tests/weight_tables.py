"""(name, tensor) lists of the test nets in each naming scheme the weight readers accept, and safetensors files of them.

The lists are what a learner hands to load_weights_device: a Python learner's module tensors, or tch's
VarStore::variables(), whose names are those var_store.save writes.  Written with write_safetensors in F32 they are the
bytes oracle/torch_net.py's writers produce (checked in test_device_weights.py), so a device table and a checkpoint of
the same list hold the same tensors under the same names.
"""
import json
import struct

import numpy as np
import torch

from oracle import torch_net


def _tch_names(created):
    """tch de-duplication on one path: the first variable of a name keeps it, later ones get "__{variables so far}"."""
    named, seen = [], set()
    for base, t in created:
        named.append((base if base not in seen else "%s__%d" % (base, len(named)), t))
        seen.add(base)
    return named


def _shuffled(named, shuffle_seed):
    if shuffle_seed is None:
        return named
    rng = np.random.default_rng(shuffle_seed)
    return [named[i] for i in rng.permutation(len(named))]


def named_explicit(net):
    out = []
    for i, (conv, bn) in enumerate(net.conv_bn_pairs()):
        out += [("conv%d.weight" % i, conv.weight), ("conv%d.bias" % i, conv.bias), ("bn%d.weight" % i, bn.weight),
                ("bn%d.bias" % i, bn.bias), ("bn%d.running_mean" % i, bn.running_mean), ("bn%d.running_var" % i, bn.running_var)]
    return out + [("policy_fc.weight", net.pfc.weight), ("policy_fc.bias", net.pfc.bias),
                  ("value_fc.weight", net.vfc.weight), ("value_fc.bias", net.vfc.bias)]


def named_tch(net, bn_order=("weight", "bias", "running_mean", "running_var"), shuffle_seed=None):
    created = []
    for c, b in net.conv_bn_pairs()[:-2]:
        created += [("bias", c.bias), ("weight", c.weight)] + [(k, getattr(b, k)) for k in bn_order]
    for c, b, l in ((net.pconv, net.pbn, net.pfc), (net.vconv, net.vbn, net.vfc)):
        created += [("bias", c.bias), ("weight", c.weight)] + [(k, getattr(b, k)) for k in bn_order] + [("bias", l.bias), ("weight", l.weight)]
    return _shuffled(_tch_names(created), shuffle_seed)


def chess_named_explicit(net):
    out = []
    for i, (conv, bn) in enumerate(net.conv_bn_pairs()):
        out += [("conv%d.weight" % i, conv.weight), ("conv%d.bias" % i, conv.bias), ("bn%d.weight" % i, bn.weight),
                ("bn%d.bias" % i, bn.bias), ("bn%d.running_mean" % i, bn.running_mean), ("bn%d.running_var" % i, bn.running_var)]
    for name, m in (("policy_conv1", net.p1), ("policy_conv2", net.p2), ("value_conv", net.vconv), ("value_fc1", net.fc1), ("value_fc2", net.fc2)):
        out += [(name + ".weight", m.weight), (name + ".bias", m.bias)]
    return out


def chess_named_tch(net, shuffle_seed=None):
    created = []
    for c, b in net.conv_bn_pairs():
        created += [("bias", c.bias), ("weight", c.weight)] + [(k, getattr(b, k)) for k in ("weight", "bias", "running_mean", "running_var")]
    for m in (net.p1, net.p2, net.vconv, net.fc1, net.fc2):
        created += [("bias", m.bias), ("weight", m.weight)]
    return _shuffled(_tch_names(created), shuffle_seed)


SCHEMES = {
    "explicit": named_explicit,
    "tch": named_tch,
    "tch_shuffled": lambda net: named_tch(net, shuffle_seed=5),
    "tch_bn_reordered": lambda net: named_tch(net, bn_order=("running_mean", "running_var", "weight", "bias")),
}
CHESS_SCHEMES = {"explicit": chess_named_explicit, "tch": chess_named_tch, "tch_shuffled": lambda net: chess_named_tch(net, shuffle_seed=3)}

_ST = {torch.float32: "F32", torch.bfloat16: "BF16", torch.float64: "F64", torch.float16: "F16"}


def write_safetensors(named, dtype=torch.float32):
    """A safetensors file of the list, every tensor cast to `dtype`; in F32 the bytes of torch_net._write_safetensors."""
    if dtype == torch.float32:
        return torch_net._write_safetensors([(n, t.detach().cpu().numpy()) for n, t in named])
    header, off, chunks = {}, 0, []
    for name, t in named:
        b = t.detach().cpu().to(dtype).contiguous().view(torch.uint8).numpy().tobytes()
        header[name] = {"dtype": _ST[dtype], "shape": list(t.shape), "data_offsets": [off, off + len(b)]}
        off += len(b)
        chunks.append(b)
    hj = json.dumps(header, separators=(",", ":")).encode()
    hj += b" " * ((8 - len(hj) % 8) % 8)
    return struct.pack("<Q", len(hj)) + hj + b"".join(chunks)


def on_device(named, device=0, dtype=torch.float32):
    """The list with every tensor copied to cuda:device in `dtype` (fresh contiguous tensors)."""
    return [(n, t.detach().to(device=torch.device("cuda", device), dtype=dtype).contiguous()) for n, t in named]
