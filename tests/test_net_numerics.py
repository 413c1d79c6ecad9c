"""The chess 10x256 network (csrc/chess_net.cu) against a bf16-faithful float64 reference (tests/chess_net_ref.py) at the
batch sizes the persistent tile loop of k_conv distinguishes, up to the 4,096 positions of the benchmark's engine.

Why not torch fp32: bf16 operands through 21 convolutions move a logit by a sizeable part of its position-dependent
spread (on a fresh net, whose logits barely depend on the position, by most of it), so a bound against fp32 has to be
loose enough to accept a kernel that gets a head wrong.  The reference rounds where the device rounds; what is left is the f32
accumulation order of the tensor cores and the bf16 roundings it flips.

Two nets: make_chess_net(seed=0) (fresh: value nearly constant, logits barely position-dependent) and
make_chess_net(seed=0, calibrated=True) (trained-like torso, live heads).  Logits are compared as |Δlogit| over the
position-dependent spread of that logit (its standard deviation over the 4,096 positions), values as |Δv|.
The bf16 roundings the accumulation order flips are themselves carried through the torso, so the reference is only
about 1.5 x closer to the kernel than torch fp32 in the worst logit; per position (the RMS over its logits) the kernel is
within 3 % of a spread.  Measured on a B200 at 1,000 W (maxima over the 4,096 positions, the same at every batch size
from 263 on; profiles/r07_net_error.txt has the distribution per size):
  calibrated: max |Δlogit| / spread 0.133, per-position RMS 0.030, max |Δv| 0.121 (torch fp32: 0.195 and 0.108)
  seed 0:     max |Δlogit| / spread 0.342, per-position RMS 0.044, max |Δv| 6.4e-4 (torch fp32: 0.397 and 8.6e-4)
"""
import numpy as np
import pytest
import torch

import selfplay_b200 as S
import chess_net_ref as R
from oracle import torch_net
from test_chess import export_all
from test_chess_search import net_positions

G = 4096
NETS = {"calibrated": dict(seed=0, calibrated=True), "seed0": dict(seed=0)}
# (max |Δlogit| / spread, max per-position RMS of |Δlogit| / spread, max |Δv|): about 1.5 x the measured maxima above
BOUNDS = {"calibrated": (0.2, 0.045, 0.18), "seed0": (0.5, 0.065, 1e-3)}


# ---- the tile loop of k_conv (chess_net.cu) ------------------------------------------------------------------------
def tiles_for(n):
    """chess_net.cu::tiles_for: an M tile is 16 board rows, a position 9 (8 + the zero row it shares with the next)."""
    return (9 * n + 15) // 16


def conv_pairs(max_positions, sms):
    """CTA pairs of launch_conv: one per two SMs, no more than the pair-tiles of the activation set's capacity."""
    return min(sms // 2, (tiles_for(max_positions) + 1) // 2)


def max_pass(n, pairs):
    """The largest `it` of k_conv's loop at n positions: pair p runs pair-tiles p, p + pairs, ... of ceil(tiles / 2)."""
    return ((tiles_for(n) + 1) // 2 - 1) // pairs


def batch_sizes(pairs):
    """1, 2, the largest n at which every pair runs exactly one tile, the first n of `it` = 1 (with an odd tile count: the
    dummy tile) and of `it` = 2 (the accumulator barrier's parity flips), 1,000 and the full engine."""
    first = [next(n for n in range(1, G + 1) if max_pass(n, pairs) >= it) for it in (1, 2)]
    return [1, 2, first[0] - 1, first[0], first[1], 1000, G - 1, G]


def errors(lg, v, ref_lg, ref_v, spread):
    """-> (max |Δlogit| / spread, the largest root-mean-square of |Δlogit| / spread over one position's logits, max |Δv|)."""
    r = (lg - ref_lg) / spread
    return float(np.abs(r).max()), float(np.sqrt((r * r).mean(1)).max()), float(np.abs(v - ref_v).max())


def accepts(err, name):
    return all(e <= b for e, b in zip(err, BOUNDS[name]))


# ---- CPU -----------------------------------------------------------------------------------------------------------

def test_bf16_rounding_matches_f2bf():
    """chess_net.cu::f2bf: nearest, ties to even, inf / NaN truncated; the tensor helper must agree bit for bit."""
    cases = {
        0x3F800000: 0x3F80,   # 1.0
        0x3F808000: 0x3F80,   # 1 + 2^-8: tie, even stays
        0x3F818000: 0x3F82,   # 1 + 3 * 2^-8: tie, odd rounds up
        0x3F808001: 0x3F81,   # just above the tie
        0x3F807FFF: 0x3F80,   # just below the tie
        0xBF818000: 0xBF82,   # negative tie
        0x7F7F0000: 0x7F7F,   # the largest bf16
        0x7F7F7FFF: 0x7F7F,   # below the tie above it
        0x7F7F8000: 0x7F80,   # the tie above the largest bf16 rounds to inf
        0xFF7F8000: 0xFF80,
        0x7F800000: 0x7F80,   # inf
        0x7FC00001: 0x7FC0,   # NaN: truncated
        0x00008000: 0x0000,   # subnormal tie, even
        0x00018000: 0x0002,   # subnormal tie, odd
        0x80000000: 0x8000,   # -0
        0x3DCCCCCD: 0x3DCD,   # 0.1
        0x3C23D70A: 0x3C24,   # 0.01 (plane 17 at fifty = 1)
    }
    bits = np.array(list(cases), np.uint32)
    got = R.bf16_round(torch.from_numpy(bits.view(np.float32).copy())).numpy().view(np.uint32) >> 16
    for b, g in zip(bits, got):
        assert R.f2bf_bits(b) == cases[int(b)], hex(b)
        assert int(g) == cases[int(b)], hex(b)
    # random finite patterns: the tensor helper, the scalar restatement and torch's own rounding agree
    rng = np.random.default_rng(0)
    r = rng.integers(0, 1 << 32, 20000, dtype=np.uint64).astype(np.uint32)
    r = r[(r & 0x7F800000) != 0x7F800000]
    got = R.bf16_round(torch.from_numpy(r.view(np.float32).copy())).numpy().view(np.uint32) >> 16
    assert (got == np.array([R.f2bf_bits(x) for x in r], np.uint32)).all()
    torch_bf = torch.from_numpy(r.view(np.float32).copy()).to(torch.bfloat16).to(torch.float32).numpy().view(np.uint32) >> 16
    assert (got == torch_bf).all()


@pytest.mark.parametrize("name", list(NETS))
def test_reference_without_rounding_equals_torch_fp32(name):
    """Layouts, BatchNorm folding and the wiring of both heads: with every rounding point off the reference is the torch net."""
    net = torch_net.make_chess_net(**NETS[name])
    enc = np.stack([g.encode() for g in net_positions()])
    _, v32, lg32 = torch_net.chess_forward(net, enc)
    lg, v = R.ChessNetRef(net, rounding=False).forward(enc)
    # measured: 6.7e-7 of the logit scale, |Δv| 2.3e-5 (tanh of the calibrated net's fc2 near saturation)
    assert np.abs(lg - lg32).max() <= 1e-5 * np.abs(lg32).max()
    assert np.abs(v - v32).max() <= 2e-4
    lgb, vb = R.ChessNetRef(net).forward(enc)
    assert np.abs(lgb - lg).max() > 0 and np.abs(vb - v).max() > 0           # and the rounding points are really there


def test_calibrated_chess_net_has_live_heads():
    """On positions the calibration did not see: values spread over (-1, 1) without piling up at ±1, and logits whose
    position-dependent part keeps at least half of its calibration spread."""
    net = torch_net.make_chess_net(seed=0, calibrated=True)
    _, _, lg_cal = torch_net.chess_forward(net, torch_net.chess_calibration_encodings())
    calib_dev = torch_net.chess_logit_deviation(lg_cal)
    assert abs(calib_dev - 1.0) < 1e-3
    enc = np.stack([g.encode() for g in net_positions()])
    lg, v = R.ChessNetRef(net).forward(enc)
    assert v.std() >= 0.3, v.std()
    assert (np.abs(v) > 0.95).mean() < 0.25
    assert torch_net.chess_logit_deviation(lg) >= 0.5 * calib_dev


# ---- GPU -----------------------------------------------------------------------------------------------------------

def distinct_positions(e, n, seed=5):
    """net_positions() (repetitions, high counters) and the benchmark's synthetic roots, every encoding distinct: a
    duplicate is moved on by random plies until it is new.  -> (states, history) of n positions."""
    from selfplay_b200.synth import synthetic_chess_roots_device
    st0, h0 = export_all(net_positions())
    st1, h1 = synthetic_chess_roots_device(e, n)
    st, hist = np.concatenate([st0, st1]), np.concatenate([h0, h1])
    rng = np.random.default_rng(seed)
    while True:
        enc = e.encode(st, hist)
        seen, dup = set(), []
        for i in range(len(st)):
            k = enc[i].tobytes()
            if k in seen:
                dup.append(i)
            seen.add(k)
        if not dup:
            return st[:n], hist[:n]
        dup = np.array(dup)
        moves, counts, _, _, _ = e.legal_moves(st[dup], hist[dup])
        pick = moves[np.arange(len(dup)), rng.integers(0, counts)]
        nxt, h2, err = e.next_states(st[dup], hist[dup], pick)
        assert not err.any()
        ongoing = e.legal_moves(nxt, h2)[3] == 0
        st[dup[ongoing]], hist[dup[ongoing]] = nxt[ongoing], h2[ongoing]


@pytest.fixture(scope="module")
def engine():
    with S.ChessEngine(num_games=G, evaluator=S.EVAL_NET) as e:
        yield e


@pytest.fixture(scope="module")
def positions(engine):
    st, hist = distinct_positions(engine, G)
    enc = engine.encode(st, hist)
    keys = [enc[i].tobytes() for i in range(G)]
    assert len(set(keys)) == G
    return st, hist, enc


_cache = {}


def net_case(name, engine, positions):
    """-> dict(net, blob, ref logits / values of all positions, per-logit spread, device outputs at the full batch);
    leaves `name`'s weights loaded in `engine`."""
    st, hist, enc = positions
    if name not in _cache:
        net = torch_net.make_chess_net(**NETS[name])
        ref_lg, ref_v = R.ChessNetRef(net, device="cuda").forward(enc)
        spread = ref_lg.std(0)
        assert spread.min() > 0
        _cache[name] = dict(net=net, blob=torch_net.chess_to_safetensors_explicit(net), ref_lg=ref_lg, ref_v=ref_v, spread=spread)
    c = _cache[name]
    engine.load_weights(c["blob"])
    if "v" not in c:
        _, c["v"], c["lg"] = engine.predict(st, hist, want_logits=True)
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NETS))
def test_chess_net_matches_bf16_reference_at_every_tile_loop_regime(name, engine, positions):
    """predict at the batch sizes that change k_conv's tile loop, against the reference; and every size gives every
    position exactly the numbers the full batch gives it."""
    st, hist, _ = positions
    c = net_case(name, engine, positions)
    pairs = conv_pairs(G, torch.cuda.get_device_properties(0).multi_processor_count)
    sizes = batch_sizes(pairs)
    assert [max_pass(n, pairs) for n in sizes[2:5]] == [0, 1, 2] and tiles_for(sizes[3]) % 2 == 1
    rows = []
    for n in sizes:
        _, v, lg = engine.predict(st[:n], hist[:n], want_logits=True)
        err = errors(lg, v, c["ref_lg"][:n], c["ref_v"][:n], c["spread"])
        rows.append((n, max_pass(n, pairs)) + err)
        assert np.array_equal(lg, c["lg"][:n]) and np.array_equal(v, c["v"][:n]), n
    print("\n%s: %d CTA pairs" % (name, pairs))
    for r in rows:
        print("  n %4d  it <= %2d  max|dlogit|/spread %.3e  position RMS %.3e  max|dv| %.3e" % r)
    for r in rows:
        assert accepts(r[2:], name), r


@pytest.mark.gpu
def test_chess_net_is_batch_invariant_bit_for_bit(engine, positions):
    """A position's outputs do not depend on where it sits in the batch: a roll by 7 changes every position's row offset in
    its tile (9 b mod 16), its CTA pair and its pass of the tile loop; and an engine of 64 games (36 CTAs) gives the numbers
    the 4,096-game engine (148 CTAs) gives."""
    st, hist, _ = positions
    c = net_case("calibrated", engine, positions)
    for n in (1000, G):
        _, v, lg = engine.predict(np.roll(st[:n], 7), np.roll(hist[:n], 7, axis=0), want_logits=True)
        assert np.array_equal(lg, np.roll(c["lg"][:n], 7, axis=0)) and np.array_equal(v, np.roll(c["v"][:n], 7)), n
    with S.ChessEngine(num_games=64, evaluator=S.EVAL_NET) as small:
        small.load_weights(c["blob"])
        for n in (1, 21, 64):
            _, v, lg = small.predict(st[:n], hist[:n], want_logits=True)
            assert np.array_equal(lg, c["lg"][:n]) and np.array_equal(v, c["v"][:n]), n


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, S.FLAG_LOCKSTEP], ids=["two-halves", "lockstep"])
def test_chess_search_roots_take_predict_values_and_priors(flags, engine, positions):
    """4,096 trees, one simulation: every root is the leaf, evaluated by the search's own batches (two halves of 2,048 on the
    two activation sets, or one batch of 4,096).  backup (chess_tree.cuh) gives the leaf +v, so a root's value_sum is the
    value predict gives that root, bit for bit; its children's priors are the softmax of predict's logits over the legal
    moves: measured max relative error 1.2e-6 on the B200 where the prior is a normal float, bound 1e-4."""
    st, hist, _ = positions
    c = net_case("calibrated", engine, positions)
    with S.ChessEngine(num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
        e.load_weights(c["blob"])
        e.reset_games(st, hist)
        e.search(1)
        for i in range(G):
            d = e.node_stats(i, 0)
            assert d["visit_count"] == 1 and d["value_sum"] == float(c["v"][i]), i
        worst = 0.0
        for i in list(range(0, G, 7)) + [G // 2 - 1, G // 2, G - 1]:     # both halves, every row offset in a tile
            mvs, _, ids = e.root_children(i)
            lg = c["lg"][i, [S.chess.policy_index(int(st[i]["side"]), m) for m in mvs]].astype(np.float64)
            want = np.exp(lg - lg.max())
            want /= want.sum()
            got = np.array([e.node_stats(i, k)["prior"] for k in ids])
            # below f32's normal range the device's priors are denormal or flushed to zero
            assert (np.abs(got - want) <= 1e-4 * want + 2e-38).all(), i
            normal = want >= 2e-38
            worst = max(worst, float((np.abs(got - want)[normal] / want[normal]).max()))
    print("\nflags %d: max relative error of the priors in f32's normal range %.3e" % (flags, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(NETS))
def test_comparison_rejects_a_perturbed_reference(name, engine, positions):
    """The comparison accepts the reference and rejects each of: every value replaced by one constant; the centre tap of
    output channels of one residual conv zeroed (one channel is within the noise: measured on the calibrated net max
    |Δlogit| / spread 0.18, per-position RMS 0.038, |Δv| 0.083 against the real 0.133 / 0.029 / 0.10; the test reports the
    smallest number of channels caught); one position's outputs taken from its batch neighbour; the value head's vcell of
    one cell dropped."""
    n = 527
    st, hist, enc = positions
    c = net_case(name, engine, positions)
    lg, v = c["lg"][:n], c["v"][:n]
    ref_lg, ref_v = c["ref_lg"][:n], c["ref_v"][:n]
    real = errors(lg, v, ref_lg, ref_v, c["spread"])
    assert accepts(real, name), real
    found = {}
    const_v = np.full_like(ref_v, (ref_v.max() + ref_v.min()) / 2)
    found["values -> one constant"] = errors(lg, v, ref_lg, const_v, c["spread"])
    if name == "seed0":
        # test_chess_network_matches_torch_fp32 accepts a constant value for this net: its check against torch fp32 on its
        # own positions, with the constant halfway between their smallest and largest value
        _, v32, _ = torch_net.chess_forward(c["net"], np.stack([g.encode() for g in net_positions()]))
        assert np.allclose(np.full_like(v32, (v32.max() + v32.min()) / 2), v32, rtol=1e-2, atol=1e-2)
    # the centre tap of output channels 0 .. k-1 of a residual conv in the middle of the torso zeroed: the smallest k caught
    for taps in (1, 2, 4, 8, 16, 32, 64, 128, 256):
        ref = R.ChessNetRef(c["net"], device="cuda")
        w, b = ref.convs[10]
        w = w.clone()
        w[:taps, :, 1, 1] = 0
        ref.convs[10] = (w, b)
        err = errors(lg, v, *ref.forward(enc[:n]), c["spread"])
        if not accepts(err, name):
            break
    found["conv 10: centre tap of %d channel(s) zeroed" % taps] = err
    k = n // 2
    nb_lg, nb_v = ref_lg.copy(), ref_v.copy()
    nb_lg[k], nb_v[k] = ref_lg[k + 1], ref_v[k + 1]
    found["position %d from its neighbour" % k] = errors(lg, v, nb_lg, nb_v, c["spread"])
    ref = R.ChessNetRef(c["net"], device="cuda")
    with torch.no_grad():
        x, last = ref.torso(enc[:n])
        vc = ref.vcell(last)
        cell = int(torch.relu(vc + ref.vb).mean(0).argmax())              # the most active cell
        vc[:, cell] = 0
        found["vcell %d dropped" % cell] = errors(lg, v, ref_lg, ref.value(vc).cpu().numpy(), c["spread"])
    print("\n%s: real %.3e / %.3e / %.3e" % ((name,) + real))
    for k2, e2 in found.items():
        print("  %-40s max|dlogit|/spread %.3e  position RMS %.3e  max|dv| %.3e" % ((k2,) + e2))
    for k2, e2 in found.items():
        assert not accepts(e2, name), (k2, e2)
