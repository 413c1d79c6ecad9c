"""The Connect4 / tic-tac-toe evaluator kernels (k_eval_umma, the product path, and the SIMT cross-check k_eval_simt)
against a bf16-faithful float64 reference (tests/small_net_ref.py), at every batch shape the static work split of
k_eval_umma distinguishes, on three nets and on positions that reach the pad column and pad row of the kernel's layout.

Why not torch fp32 (test_gpu_evaluator.py): bf16 rounding alone moves the logits by 0.6 .. 1.3 % of their scale, most of
that check's 1 % budget, so it accepts kernels that get a channel of a residual conv wrong or leave the head activations
unrounded (test_fp32_check_accepts_what_this_comparison_rejects); and the value of a fresh or trained-like net hardly
depends on the position (standard deviation 0.02), so a value head wrong in a position-dependent way is invisible.  The
reference rounds where the device rounds; what is left is the f32 accumulation order and the bf16 roundings it flips.

Nets (all seed 2): fresh (make_net), trained-like (trained_like=True: larger heads, random BatchNorm statistics) and
calibrated (calibrated=True: BatchNorm statistics of its own activations, live value head, logits of unit spread).
Logits are compared as |Δlogit| over the position-dependent spread of that logit (its standard deviation over the
positions), values as |Δv|, and for the calibrated net the masked softmax as |Δp|.  Positions: tic-tac-toe, all 4,520
reachable ongoing positions; Connect4, 19,000 positions: edge positions (empty board, full columns 0 and 6, the first
row of a board in the kernel's layout filled, nearly full boards) followed by random playouts.
Measured on a B200 at 1,000 W over every position in one call (every batch size gives every position the same numbers,
so these are the maxima over all sizes too), the larger of the two kernels (profiles/r10_eval_error.txt has them per
kernel and batch size); max |Δlogit| / spread, per-position RMS max and median, max |Δv|, max |Δp|:
  c4 fresh          0.0417  0.0219  5.6e-7  1.2e-3
  c4 trained-like   0.109   0.0527  1.2e-6  1.7e-3
  c4 calibrated     0.0407  0.0188  1.8e-7  0.0213  8.4e-3
  ttt fresh         0.0278  0.0152  3.2e-7  5.3e-4
  ttt trained-like  0.0936  0.0470  9.1e-7  1.3e-4
  ttt calibrated    0.0305  0.0143  1.1e-7  0.0190  9.4e-3
The maxima are bf16 roundings that the f32 accumulation order flips and the torso carries to the outputs: 10 layers of
64 channels, so they stay below chess's 0.13 of spread.  Most positions see no flip at all, so the median per-position
RMS sits at the f32 summation error of the Linear heads; an error every position carries shows there even when it hides
under the maxima.  Leaving the head activations unrounded (what k_eval_simt did before it stored them as bf16) moves the
maxima by less than this noise floor on every net (c4 calibrated: 0.034 / 0.016 / |Δv| 0.018), but the median by
2.4e-3 .. 1.9e-2, four orders of magnitude above its bound.
"""
import numpy as np
import pytest
import torch

import selfplay_b200 as S
import small_net_ref as R
from helpers import random_states
from oracle import pyoracle as O, torch_net
from test_gpu_evaluator import check_against_fp32

GAMES = {"c4": S.GAME_C4, "ttt": S.GAME_TTT}
NETS = {"fresh": dict(seed=2), "trained-like": dict(seed=2, trained_like=True), "calibrated": dict(seed=2, calibrated=True)}
KERNELS = {"tcgen05": 0, "simt": S.FLAG_EVAL_SIMT}
C4_POSITIONS = 19000
# (max |Δlogit| / spread, max and median per-position RMS of |Δlogit| / spread, max |Δv|, max |Δp| or None): about
# 1.5 x the measured maxima above, one bound per (game, net) for both kernels
BOUNDS = {
    ("c4", "fresh"): (0.063, 0.033, 8.4e-7, 1.8e-3, None),
    ("c4", "trained-like"): (0.16, 0.079, 1.8e-6, 2.5e-3, None),
    ("c4", "calibrated"): (0.061, 0.028, 2.7e-7, 0.032, 0.013),
    ("ttt", "fresh"): (0.042, 0.023, 4.8e-7, 7.9e-4, None),
    ("ttt", "trained-like"): (0.14, 0.071, 1.4e-6, 2.0e-4, None),
    ("ttt", "calibrated"): (0.046, 0.021, 1.7e-7, 0.028, 0.014),
}


# ---- the static work split of k_eval_umma (evaluator_umma.cu) ---------------------------------------------------------
def boards_per_batch(game):
    """Geo<G>::NB: four 128-row tiles of boards of 7 x 8 rows (Connect4) or 4 x 4 rows (tic-tac-toe)."""
    return 4 * 128 // (56 if game == S.GAME_C4 else 16)


def batches(n, sms, game):
    """The batch sizes of a call of n positions: min(sms, n) CTAs, CTA k takes positions [n k / ncta, n (k + 1) / ncta)
    and runs them in batches of NB boards, the last one short."""
    nb, ncta = boards_per_batch(game), min(sms, n)
    out = []
    for cta in range(ncta):
        b, e = n * cta // ncta, n * (cta + 1) // ncta
        out += [min(nb, e - b0) for b0 in range(b, e, nb)]
    return out


def batch_sizes(game, sms):
    """1, 2 and sms - 1 (one board per CTA); sms (t + 1/2) for odd t (CTAs of t and t + 1 boards: every short batch of
    1 .. NB boards, hence every tail of the Linear heads' 3-board loop and every last tile of a short batch); sms NB and
    the sizes on either side; the benchmark's 4,096 trees; 19,000 (about 128 boards per CTA, many full batches)."""
    nb = boards_per_batch(game)
    return [1, 2, sms - 1] + [sms * t + sms // 2 for t in range(1, nb, 2)] + [sms * nb - 1, sms * nb, sms * nb + 1, 4096, 19000]


def check_batch_sizes(game, sms):
    nb = boards_per_batch(game)
    sizes = batch_sizes(game, sms)
    seen = set()
    for n in sizes:
        seen |= set(batches(n, sms, game))
    assert seen == set(range(1, nb + 1))
    assert all(set(batches(n, sms, game)) == {1} for n in sizes if n < sms)
    assert set(batches(sms * nb, sms, game)) == {nb} and 1 in batches(sms * nb + 1, sms, game)
    return sizes


# ---- positions -------------------------------------------------------------------------------------------------------
def play(game, moves):
    s = O.State()
    for a in moves:
        s = O.next_state(game, s, a)
        assert s is not None and s.status == O.ONGOING, moves
    return s


def ttt_positions():
    """Every reachable ongoing tic-tac-toe position, in breadth-first order (5,478 reachable, 4,520 ongoing)."""
    seen, frontier, out = {O.State().key()}, [O.State()], []
    n_all = 1
    while frontier:
        out += frontier
        nxt = []
        for s in frontier:
            for a in O.valid_actions(O.GAME_TTT, s):
                t = O.next_state(O.GAME_TTT, s, a)
                if t.key() not in seen:
                    seen.add(t.key())
                    n_all += 1
                    if t.status == O.ONGOING:
                        nxt.append(t)
        frontier = nxt
    assert n_all == 5478 and len(out) == 4520
    return out


def c4_edge_positions(nearly_full=24, seed=17):
    """The empty board, full column 0, full column 6, both, row 0 filled (the first row of a board in the kernel's layout,
    next to the previous board's pad row), and boards of 40 and 41 stones without a winner (row 5, next to the pad
    row, nearly filled; one or two legal moves)."""
    out = [play(O.GAME_C4, m) for m in ([], [0] * 6, [6] * 6, [0] * 6 + [6] * 6, list(range(7)), list(range(7)) + [0] * 5)]
    rng = np.random.default_rng(seed)
    while len(out) < 6 + nearly_full:
        s, target = O.State(), 40 + len(out) % 2
        while s is not None and s.num_actions_played < target:
            safe = [t for t in (O.next_state(O.GAME_C4, s, a) for a in O.valid_actions(O.GAME_C4, s)) if t.status == O.ONGOING]
            s = safe[rng.integers(len(safe))] if safe else None
        if s is not None:
            out.append(s)
    return out


def positions(game):
    if game == S.GAME_TTT:
        return ttt_positions()
    edges = c4_edge_positions()
    return edges + random_states(game, C4_POSITIONS - len(edges), seed=23, include_terminal=False)


def legal_masks(game, states):
    m = np.zeros((len(states), O.NUM_ACTIONS[game]), bool)
    for i, s in enumerate(states):
        m[i, O.valid_actions(game, s)] = True
    return m


def masked_softmax(logits, mask):
    p = R.softmax(logits) * mask
    return p / p.sum(1, keepdims=True)


# ---- metrics ---------------------------------------------------------------------------------------------------------
def metrics(c, lg, v, pol, ref_lg=None, ref_v=None, idx=None):
    """-> (max |Δlogit| / spread; the largest and the median root-mean-square of |Δlogit| / spread over one position's
    logits; max |Δv|; max |Δp| of the masked softmax)."""
    idx = np.arange(len(lg)) if idx is None else idx
    ref_lg = c["ref_lg"][idx] if ref_lg is None else ref_lg
    ref_v = c["ref_v"][idx] if ref_v is None else ref_v
    r = (lg - ref_lg) / c["spread"]
    rms = np.sqrt((r * r).mean(1))
    dp = np.abs(pol - masked_softmax(ref_lg, c["mask"][idx])).max()
    return float(np.abs(r).max()), float(rms.max()), float(np.median(rms)), float(np.abs(v - ref_v).max()), float(dp)


def accepts(err, game_name, net_name):
    b = BOUNDS[(game_name, net_name)]
    return all(e <= x for e, x in zip(err, b) if x is not None)


# ---- CPU -------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("game", list(GAMES))
def test_batch_sizes_reach_every_batch_shape(game):
    """The sizes the GPU tests use, on a 148-SM B200 and on a part with fewer SMs, give every short batch."""
    for sms in (148, 132):
        check_batch_sizes(GAMES[game], sms)


@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("game", list(GAMES))
def test_reference_without_rounding_equals_torch_fp32(game, net):
    """BatchNorm folding, the fused head conv's channel order, the Linear heads' flat index and the value's tanh: with every
    rounding point off the reference is the torch net."""
    g = GAMES[game]
    tn = torch_net.make_net(g, **NETS[net])
    states = random_states(g, 300, seed=5, include_terminal=False)
    enc = np.stack([O.encode(g, s) for s in states])
    _, v32, lg32 = torch_net.forward_probs(tn, enc)
    lg, v = R.SmallNetRef(tn, rounding=False).forward(enc)
    # measured: at most 8.6e-7 of the logit scale, |Δv| at most 3.1e-6 (the calibrated net's live value)
    assert np.abs(lg - lg32).max() <= 1e-5 * np.abs(lg32).max()
    assert np.abs(v - v32).max() <= 3e-5
    lgb, vb = R.SmallNetRef(tn).forward(enc)
    assert np.abs(lgb - lg).max() > 0 and np.abs(vb - v).max() > 0          # and the rounding points are really there


@pytest.mark.parametrize("game", list(GAMES))
def test_calibrated_net_has_live_heads(game):
    """On positions the calibration did not see: values spread over (-1, 1) without piling up at ±1, and logits whose
    position-dependent part keeps at least half of its calibration spread."""
    g = GAMES[game]
    net = torch_net.make_net(g, **NETS["calibrated"])
    _, _, lg_cal = torch_net.forward_probs(net, torch_net.calibration_encodings(g))
    assert np.allclose(lg_cal.std(0, ddof=1), 1.0, atol=1e-3)              # torch_net scales by the unbiased estimate
    held_out = random_states(g, 2000, seed=29, include_terminal=False)
    lg, v = R.SmallNetRef(net).forward(np.stack([O.encode(g, s) for s in held_out]))
    assert v.std() >= 0.45, v.std()
    assert (np.abs(v) > 0.95).mean() < 0.1
    assert ((lg - lg.mean(0)).std(0) >= 0.5).all()
    for other in ("fresh", "trained-like"):                                    # what the other nets' values look like
        _, v_other = R.SmallNetRef(torch_net.make_net(g, **NETS[other])).forward(np.stack([O.encode(g, s) for s in held_out]))
        assert v_other.std() < 0.05


def perturbed(net, what, device="cpu"):
    """The reference with one error a kernel could make: the bias of channel 5 of conv 5 (the second conv of the second
    residual block) missing, the centre tap of that channel zeroed, or the head activations left unrounded."""
    ref = R.SmallNetRef(net, device=device)
    if what == "head unrounded":
        ref.round_head = False
        return ref
    w, b = ref.convs[5]
    w, b = w.clone(), b.clone()
    if what == "bias missing":
        b[5] = 0
    else:
        w[5, :, 1, 1] = 0
    ref.convs[5] = (w, b)
    return ref


def fp32_check_accepts(game, net, states, lg, v, trained_like):
    """test_gpu_evaluator.py's comparison against torch fp32, with (lg, v) standing in for the kernel's outputs."""
    pol = np.stack([O.mask_invalid_actions(game, s, p) for s, p in zip(states, R.softmax(lg).astype(np.float32))])
    try:
        check_against_fp32(game, net, states, pol, v.astype(np.float32), lg.astype(np.float32), trained_like)
    except AssertionError:
        return False
    return True


FP32_ACCEPTS = {"fresh": ("bias missing", "centre tap zeroed", "head unrounded"),
                "trained-like": ("bias missing", "centre tap zeroed", "head unrounded")}


@pytest.mark.parametrize("net", list(FP32_ACCEPTS))
def test_fp32_check_accepts_what_this_comparison_rejects(net):
    """Connect4, 2,000 random positions of test_tcgen05_evaluator_matches_torch (seed 2): the fp32 check of
    test_gpu_evaluator.py accepts the bf16 reference standing in for the kernel, and accepts it with each error of
    perturbed(); test_comparison_rejects_a_perturbed_reference shows that the comparison of this file rejects them.
    Channel 5 of conv 5 is one whose missing bias and zeroed centre tap the fp32 check accepts on both nets (of channels
    0 .. 5 of conv 5 it accepts the missing bias of channels 1 and 5 on the fresh net, of 3, 4 and 5 on the trained-like
    net).  Measured, as max |Δlogit| / spread, per-position RMS, |Δv| against the unperturbed reference:
      fresh:        bias missing 0.077 / 0.037 / 2e-3, centre tap zeroed 0.121 / 0.060 / 4e-3, head unrounded 0.041 / 0.020 / 1.3e-3
      trained-like: bias missing 0.225 / 0.118 / 3e-3, centre tap zeroed 0.301 / 0.173 / 3e-3, head unrounded 0.075 / 0.038 / 1.9e-3
    As a control, it rejects the stand-in with the logits of actions 0 and 1 swapped."""
    g, tl = S.GAME_C4, net == "trained-like"
    tn = torch_net.make_net(g, **NETS[net])
    states = random_states(g, 2000, seed=3, include_terminal=False)
    enc = np.stack([O.encode(g, s) for s in states])
    lg, v = R.SmallNetRef(tn).forward(enc)
    assert fp32_check_accepts(g, tn, states, lg, v, tl)
    for what in FP32_ACCEPTS[net]:
        assert fp32_check_accepts(g, tn, states, *perturbed(tn, what).forward(enc), tl), what
    assert not fp32_check_accepts(g, tn, states, lg[:, [1, 0, 2, 3, 4, 5, 6]], v, tl)


# ---- GPU -------------------------------------------------------------------------------------------------------------
_cache = {}


def case(game_name, net_name):
    """-> dict(net, blob, states, mask, reference logits / values on every position, per-logit spread)."""
    key = (game_name, net_name)
    if key not in _cache:
        g = GAMES[game_name]
        if game_name not in _cache:
            st = positions(g)
            _cache[game_name] = dict(states=O.states_array(st), enc=np.stack([O.encode(g, s) for s in st]), mask=legal_masks(g, st))
        pos = _cache[game_name]
        net = torch_net.make_net(g, **NETS[net_name])
        ref_lg, ref_v = R.SmallNetRef(net, device="cuda").forward(pos["enc"])
        spread = ref_lg.std(0)
        assert spread.min() > 0
        _cache[key] = dict(pos, net=net, blob=torch_net.to_safetensors_tch(net), ref_lg=ref_lg, ref_v=ref_v, spread=spread)
    return _cache[key]


def predict_all(c, game_name, kernel):
    """The kernel's outputs on every position in one call (cached)."""
    if kernel not in c:
        with S.Engine(game=GAMES[game_name], num_games=4, evaluator=S.EVAL_NET, flags=KERNELS[kernel]) as e:
            e.load_weights(c["blob"])
            c[kernel] = e.predict(c["states"], want_logits=True)
    return c[kernel]


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("game", list(GAMES))
def test_evaluator_matches_bf16_reference_at_every_batch_shape(game, net, kernel):
    """One call over every position against the reference; and every size of batch_sizes() (positions repeated cyclically
    past the end of the set) gives every position exactly the numbers that call gives it, so the bounds hold at every
    size (the rows printed for the sizes are subsets; a median over a call of one or two positions is no median)."""
    g = GAMES[game]
    c = case(game, net)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    sizes = check_batch_sizes(g, sms)
    pol_all, v_all, lg_all = predict_all(c, game, kernel)
    rows = [(len(v_all),) + metrics(c, lg_all, v_all, pol_all)]
    with S.Engine(game=g, num_games=4, evaluator=S.EVAL_NET, flags=KERNELS[kernel]) as e:
        e.load_weights(c["blob"])
        for n in sizes:
            idx = np.arange(n) % len(c["states"])
            pol, v, lg = e.predict(c["states"][idx], want_logits=True)
            rows.append((n,) + metrics(c, lg, v, pol, idx=idx))
            assert np.array_equal(lg, lg_all[idx]) and np.array_equal(v, v_all[idx]) and np.array_equal(pol, pol_all[idx]), n
    print("\n%s %s %s (%d SMs)" % (game, net, kernel, sms))
    for r in rows:
        print("  n %5d  max|dlogit|/spread %.3e  position RMS max %.3e median %.3e  max|dv| %.3e  max|dp| %.3e" % r)
    assert accepts(rows[0][1:], game, net), rows[0]


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, S.FLAG_LOCKSTEP], ids=["async", "lockstep"])
@pytest.mark.parametrize("game", list(GAMES))
def test_search_roots_take_predict_priors_and_values_bit_for_bit(game, flags):
    """4,096 trees (the benchmark's engine), one simulation on the calibrated net: every root is the leaf, evaluated by the
    search's own batches (the asynchronous pipeline's leaf ring, or the lock-step pipeline's static list).  Every root
    child's prior is predict's masked policy for its action, bit for bit, and the root's value_sum is predict's value
    with the sign backup gives the leaf (+v)."""
    G = 4096
    c = case(game, "calibrated")
    roots = c["states"][:G]
    with S.Engine(game=GAMES[game], num_games=G, evaluator=S.EVAL_NET, flags=flags) as e:
        e.load_weights(c["blob"])
        pol, v = e.predict(roots)
        e.reset_games(roots)
        e.search(1)
        a, _, ids, n = e.root_children_all()
        for slot in range(G):
            root = e.node_stats(slot, 0)
            assert root["visit_count"] == 1 and root["value_sum"] == float(v[slot]), slot
            assert n[slot] == c["mask"][slot].sum() == root["n_children"], slot
            for j in range(int(n[slot])):
                assert e.node_stats(slot, int(ids[slot, j]))["prior"] == float(pol[slot, a[slot, j]]), (slot, j)


@pytest.mark.gpu
@pytest.mark.parametrize("net", list(NETS))
@pytest.mark.parametrize("game", list(GAMES))
def test_comparison_rejects_a_perturbed_reference(game, net):
    """The tcgen05 kernel's outputs on every position against the reference accepted, and against each perturbed
    reference rejected: perturbed()'s three errors (the ones the fp32 check accepts), one position's outputs taken
    from its neighbour, and the most active value channel of the head conv dropped.  Measured on the B200 of the
    bounds: the missing bias and the zeroed centre tap exceed every max-type bound (c4 trained-like, the closest: max
    |Δlogit| / spread 0.227 and 0.324 against 0.16) and every median bound by four orders of magnitude; the unrounded
    heads stay under the max-type bounds on every net, within the noise floor, and are caught by the median alone
    (1.8e-2 c4 trained-like, 2.4e-3 ttt calibrated); the neighbour by max |Δlogit| / spread (1.2 .. 2.6), the dropped
    value channel by |Δv| (0.13 .. 1.9)."""
    g = GAMES[game]
    c = case(game, net)
    pol, v, lg = predict_all(c, game, "tcgen05")
    real = metrics(c, lg, v, pol)
    found = {}
    for what in ("bias missing", "centre tap zeroed", "head unrounded"):
        found[what] = metrics(c, lg, v, pol, *perturbed(c["net"], what, device="cuda").forward(c["enc"]))
    k = len(v) // 2
    while np.array_equal(c["enc"][k], c["enc"][k + 1]):
        k += 1
    nb_lg, nb_v = c["ref_lg"].copy(), c["ref_v"].copy()
    nb_lg[k], nb_v[k] = c["ref_lg"][k + 1], c["ref_v"][k + 1]
    found["position %d from its neighbour" % k] = metrics(c, lg, v, pol, nb_lg, nb_v)
    ref = R.SmallNetRef(c["net"], device="cuda")
    with torch.no_grad():
        h = torch.cat([ref.head(ref.torso(c["enc"][i:i + 4096])) for i in range(0, len(v), 4096)])
        ch = ref.policy_ch + int(h[:, ref.policy_ch:].mean((0, 2, 3)).argmax())
        h[:, ch] = 0
        d_lg, z = ref.linear(h)
        found["value channel %d dropped" % (ch - ref.policy_ch)] = metrics(c, lg, v, pol, d_lg.cpu().numpy(), torch.tanh(z).cpu().numpy())
    print("\n%s %s: real %.3e / %.3e / %.3e / %.3e / %.3e" % ((game, net) + real))
    for k2, e2 in found.items():
        print("  %-32s max|dlogit|/spread %.3e  position RMS max %.3e median %.3e  max|dv| %.3e  max|dp| %.3e" % ((k2,) + e2))
    assert accepts(real, game, net), real
    for k2, e2 in found.items():
        assert not accepts(e2, game, net), (k2, e2)
