"""Every trunk kernel against the bf16-emulating oracle BIT FOR BIT, on nets whose arithmetic is exact.

The kernels and `orc.forward(emulate_bf16=True)` round at the same points (bf16 inputs and weights, fp32 accumulation,
bias (+ skip) -> ReLU -> bf16 round-to-nearest-even after every conv) and differ only in the order of their fp32
accumulations.  On a random net that order flips bf16 roundings, so the other forward tests need tolerances, and a
bug smaller than them - or one that every kernel shares - passes.  Here the nets are built so that every fp32
accumulation is EXACT, and then the order cannot matter:

  * every weight and bias of a layer is a small integer m (|m| <= 2, mostly 0) times a power of two, and every input
    value is a multiple of a known power of two; so all the terms of a layer's sums (activation x weight, bias, skip)
    are multiples of one grid g, and bf16 rounding and ReLU keep a multiple of g a multiple of g;
  * the sum of the absolute terms of every output element of every layer - the trunk convs, the policy and value
    convs, FC1 and FC2 - is below 2^22 g (checked in float64 on the very inputs the tests feed), so every partial sum
    in any order is an fp32 number, with two bits to spare for a tensor core that aligns its products and truncates.

Then the dense logits of every kernel must equal the oracle's bit for bit; win and draw go through expf and a
division on exact inputs and must agree within a few ulp.  The per-layer powers of two keep the values in realistic
ranges (logit rms ~ 1-3, pre-sigmoid values within +-8); they do not change the bound, which is relative to g.

The CPU part checks the premise: on these nets the oracle equals an independent float64 forward bit for bit, and on a
random-init net it does not.  The generator also asserts that the tests are not vacuous (every conv layer has weights in
every output channel, tap and 16-channel K block; 20-80 % of the activations are non-zero; bf16 rounding and exact
ties happen; the value head is alive)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import helpers

BOUND = 2.0 ** 22       # sum |terms| / grid must stay below this at every output element
BASE = 24               # distinct inputs per input path; larger batches tile them
FIRST_SCALAR = 82       # channels from here on enter the stem twice (hi + twin lo, DESIGN.md §6.8)

# name -> (channels, blocks, in_channels, conv density, weight seed, input seed)
# The sum of absolute terms per grid step grows by a roughly constant factor per layer (about 1.5-2 at these densities,
# see the generator's stats), on top of what the inputs start with.  The shallow nets spend most of the 2^22 on inputs
# with fine grids and up to 12 significant bits (both halves of the twin channels); the deep nets have 21 conv layers
# and coarse inputs.  The conv densities scale as 1 / channels, so that every output reads about as many terms.
NETS = {
    "128x2": (128, 2, 86, 0.002, 1, 11),
    "128x10": (128, 10, 86, 0.001, 2, 12),
    "192x2": (192, 2, 86, 0.0013, 3, 13),
    "192x10": (192, 10, 86, 0.00067, 4, 14),
    "256x2": (256, 2, 86, 0.001, 5, 15),
    "256x10": (256, 10, 86, 0.0005, 6, 16),
    "128x2c93": (128, 2, 93, 0.002, 7, 17),
    "256x2c93": (256, 2, 93, 0.001, 8, 18),
}


# ---- float64 restatement ------------------------------------------------------------------------------------------
def bf16(x):
    """Round-to-nearest-even to 8 significant bits, in float64 (exact: no double rounding through fp32)."""
    x = np.asarray(x, dtype=np.float64)
    m, e = np.frexp(x)
    return np.ldexp(np.round(m * 256.0), e - 8)   # np.round: half to even


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64))


def stem_input(planes, in_channels):
    """The stem's input as the kernels and the oracle see it: bf16 of every plane, then for every plane from channel 82
    on a twin carrying bf16 of what that rounding lost (fp32 arithmetic: v - bf16(v) is exact)."""
    x = np.asarray(planes, dtype=np.float64).reshape(-1, in_channels, 81)
    hi = bf16(x)
    if in_channels <= FIRST_SCALAR:
        return hi
    lo = bf16(x[:, FIRST_SCALAR:] - hi[:, FIRST_SCALAR:])
    return np.concatenate([hi, lo], axis=1)


def stem_weights(w, in_channels):
    """The stem weights extended by the twins' copies of the scalar planes' weights."""
    return np.concatenate([w, w[:, FIRST_SCALAR:]], axis=1) if in_channels > FIRST_SCALAR else w


def conv(a, w, b=None, pad=1):
    """a [n][cin][81], w [cout][cin][k][k] -> [n][cout][81], float64 (exact on the nets here)."""
    y = F.conv2d(_t(a).reshape(a.shape[0], -1, 9, 9), _t(w), None if b is None else _t(b), padding=pad)
    return y.reshape(a.shape[0], w.shape[0], 81).numpy()


def forward64(desc, blob, planes):
    """Independent float64 forward of the canonical net with the bf16 rounding points of the kernels: torch conv2d in
    float64, bf16 after each trunk conv's bias (+ skip) and ReLU, value conv / FC1 / FC2 and the logits unrounded."""
    w = helpers.split_blob(desc, np.asarray(blob, dtype=np.float64))
    IN = desc.in_channels
    x = bf16(np.maximum(conv(stem_input(planes, IN), stem_weights(w["stem_w"], IN), w["stem_b"]), 0))
    for (w1, b1, w2, b2) in w["blocks"]:
        t = bf16(np.maximum(conv(x, w1, b1), 0))
        x = bf16(np.maximum(conv(t, w2, b2) + x, 0))
    pol = conv(x, w["pol_w"][:, :, None, None], w["pol_b"], pad=0).reshape(-1, 27 * 81)
    v = np.maximum(conv(x, w["val_w"][None, :, None, None], w["val_b"], pad=0)[:, 0], 0)
    h = np.maximum(v @ w["fc1_w"].T + w["fc1_b"], 0)
    o = h @ w["fc2_w"].T + w["fc2_b"]
    return pol, o


# ---- the generator ------------------------------------------------------------------------------------------------
def _pow2(x):
    return 2.0 ** np.round(np.log2(x))


def _is_multiple(x, g):
    q = np.asarray(x, dtype=np.float64) / g
    return bool(np.all(q == np.round(q)))


def row_grids(x):
    """Per input row (position), the coarsest power of two that all its values are multiples of, shaped [n][1][1].
    Rows are independent, so each may have its own grid: a row of large integer fill values and a row of fine
    fractions need not share the fine one."""
    g = np.ones(x.shape[0])
    for i in range(x.shape[0]):
        while not _is_multiple(x[i], g[i]):
            g[i] /= 2
    return g[:, None, None]


class _Gen:
    """Draws the integer weights of one net and records, layer by layer, the grid, the bound and the statistics."""

    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.layers = []   # per trunk layer: dict of stats

    def ints(self, shape, density, nonzero=False):
        """Integers in {-2..2}: non-zero with probability `density` (or always), |m| = 2 for a quarter of those."""
        mag = np.where(self.rng.random(shape) < 0.25, 2.0, 1.0) * np.where(self.rng.random(shape) < 0.5, -1.0, 1.0)
        return mag if nonzero else np.where(self.rng.random(shape) < density, mag, 0.0)

    def conv_ints(self, cout, cin, density):
        m = self.ints((cout, cin, 3, 3), density)
        for co in range(cout):   # every output channel gets at least one weight
            if not m[co].any():
                m[co, self.rng.integers(cin), self.rng.integers(3), self.rng.integers(3)] = self.ints((), 0, True)
        return m

    @staticmethod
    def scale(y, target=1.0):
        """The power of two s that brings the rms of y near `target`."""
        r = float(np.sqrt(np.mean(y * y)))
        return _pow2(target / r) if r > 0 else 1.0

    def check(self, what, bound, g):
        """bound [n][...] = sum of |terms| per output element, g [n][1][1] = the row's grid."""
        ratio = float((bound.reshape(bound.shape[0], -1) / g.reshape(-1, 1)).max())
        assert ratio < BOUND, f"{what}: sum |terms| / grid = {ratio:.3g} >= 2^22"
        assert g.min() > 2.0 ** -100, f"{what}: grid {g.min()} too fine"
        return ratio

    def trunk_layer(self, a, g_in, m, skip=None, g_skip=None):
        """One conv layer on activations `a` (grid g_in), with the skip `skip` (grid g_skip) if given: returns (out, grid,
        weights, bias).  A residual layer's biases are <= 0, so that the residual stream does not only grow."""
        y0 = conv(a, m)
        s = self.scale(y0)
        w = m * s
        g = g_in * s if skip is None else np.minimum(g_in * s, g_skip)
        mb = self.ints((m.shape[0],), 0.5)
        if skip is not None:
            mb = -np.abs(mb)
        unit = max(_pow2(0.5), g.max())             # bias of order 0.5, on every row's grid
        b = mb * unit
        pre = y0 * s + b[None, :, None] + (0 if skip is None else skip)
        bound = conv(np.abs(a), np.abs(w)) + np.abs(b)[None, :, None] + (0 if skip is None else np.abs(skip))
        ratio = self.check(f"layer {len(self.layers)}", bound, g)
        relu = np.maximum(pre, 0)
        out = bf16(relu)
        assert _is_multiple(out, g)
        # statistics: non-zero share, roundings, exact ties (the dropped part is exactly half an ulp of the result)
        mant, _ = np.frexp(relu)
        frac = mant * 256.0 - np.floor(mant * 256.0)
        self.layers.append({"nonzero": float(np.mean(out != 0)), "rounded": int(np.sum(out != relu)),
                            "ties": int(np.sum((frac == 0.5) & (relu != 0))), "ratio": ratio})
        return out, g, w, b


def exact_blob(desc, seed, planes, density, stem_density=0.02):
    """A canonical blob (helpers.split_blob layout) on which the fp32 forward of `planes` is exact, and its statistics.
    planes: [n][in_channels][81] fp32, the inputs the tests will feed (both input paths)."""
    C, IN, NB, H = desc.channels, desc.in_channels, desc.blocks, desc.value_hidden
    x_in = stem_input(planes, IN)
    g0 = row_grids(x_in)
    gen = _Gen(seed)
    parts = []
    m = gen.conv_ints(C, IN, stem_density)
    x, g, w, b = gen.trunk_layer(x_in, g0, stem_weights(m, IN))
    parts += [w[:, :IN], b]
    for _ in range(NB):
        t, gt, w1, b1 = gen.trunk_layer(x, g, gen.conv_ints(C, C, density))
        x, g, w2, b2 = gen.trunk_layer(t, gt, gen.conv_ints(C, C, density), skip=x, g_skip=g)
        parts += [w1, b1, w2, b2]
    stats = {"layers": gen.layers, "grid0": g0.ravel()}
    # policy conv 1x1: every plane reads ~6 channels and has a non-zero bias
    mp = gen.ints((27, C), 6.0 / C)
    yp = conv(x, mp[:, :, None, None], pad=0)
    sp = gen.scale(yp, target=2.0)
    gp = g * sp
    bp = gen.ints((27,), 0, nonzero=True) * max(_pow2(0.5), gp.max())
    wp = mp * sp
    stats["policy_ratio"] = gen.check("policy", conv(x, np.abs(wp)[:, :, None, None], np.abs(bp), pad=0), gp)
    parts += [wp, bp]
    # value conv 1x1 -> 1: a few channels; ReLU, unrounded (the kernels keep the plane in fp32)
    mv = gen.ints((C,), 2.0 / C)
    yv = conv(x, mv[None, :, None, None], pad=0)[:, 0]
    sv = gen.scale(yv)
    gv = g * sv
    uv = max(_pow2(0.25), gv.max())
    bv = np.array([-np.round(np.median(yv * sv) / uv) * uv or uv])   # about half of the squares live, never 0
    wv = mv * sv
    gv = gv[:, 0]                                   # [n][1]: the value plane and FC1 / FC2 are [n][k]
    stats["value_ratio"] = gen.check("value conv", conv(x, np.abs(wv)[None, :, None, None], np.abs(bv), pad=0)[:, 0], gv)
    v = np.maximum(yv * sv + bv, 0)
    parts += [wv, bv]
    # FC1: every hidden unit reads a few squares.  The first and the last unit (where a loop bound goes wrong) read one
    # square that varies over the inputs, with a positive weight and a bias >= 0: they are live on every draw.
    m1 = gen.ints((H, 81), 1.5 / 81)
    varying = np.nonzero(np.ptp(v, axis=0) > 0)[0]
    assert varying.size > 0, "dead value plane"
    edge = [0, H - 1]
    m1[edge] = 0
    m1[edge, gen.rng.choice(varying, size=2)] = np.abs(gen.ints((2,), 0, nonzero=True))
    y1 = v @ m1.T
    s1 = gen.scale(y1)
    g1 = gv * s1
    b1 = gen.ints((H,), 0.5) * max(_pow2(0.25), g1.max())
    b1[edge] = np.abs(b1[edge])
    w1 = m1 * s1
    stats["fc1_ratio"] = gen.check("FC1", np.abs(v) @ np.abs(w1).T + np.abs(b1), g1)
    hid = np.maximum(v @ w1.T + b1, 0)
    parts += [w1, b1]
    # FC2: the two edge units and two more live ones per output (hidden units that vary over the inputs); scaled so
    # the pre-sigmoid values spread over a few units, centred
    live = np.setdiff1d(np.nonzero(np.ptp(hid, axis=0) > 0)[0], edge)
    assert np.ptp(hid[:, edge], axis=0).all() and live.size >= 2, "dead value head"
    m2 = np.zeros((2, H))
    for k in range(2):
        pick = np.concatenate([edge, gen.rng.choice(live, size=2, replace=False)])
        m2[k, pick] = gen.ints((pick.size,), 0, nonzero=True)
    y2 = hid @ m2.T
    s2 = np.array([gen.scale(y2[:, k] - y2[:, k].mean(), target=1.5) for k in range(2)])
    s2 = float(s2.min())
    g2 = g1 * s2
    w2 = m2 * s2
    u2 = max(_pow2(0.25), g2.max())
    b2 = -np.round(y2.mean(0) * s2 / u2) * u2
    stats["fc2_ratio"] = gen.check("FC2", np.abs(hid) @ np.abs(w2).T + np.abs(b2), g2)
    parts += [w2, b2]
    stats["pre_sigmoid"] = z = hid @ w2.T + b2
    assert np.abs(z).max() < 8, "pre-sigmoid values out of range"
    assert (np.ptp(1 / (1 + np.exp(-z)), axis=0) > 1e-2).all(), "dead value head"   # DESIGN.md §4
    blob = np.concatenate([np.ravel(p) for p in parts]).astype(np.float32)
    assert np.array_equal(blob.astype(np.float64), np.concatenate([np.ravel(p) for p in parts])), "blob not fp32-exact"
    return blob, stats


# ---- inputs on the grid -------------------------------------------------------------------------------------------
def bitboard_inputs(synth, in_channels, seed, wide):
    """BASE inputs as FeatureBitboards: synth's fuzz (random masks, rotation, garbage bits) with dyadic fill values.
    The 0/1-like planes get small dyadic values; the scalar planes get values with more than 8 significant bits, so
    both halves of their twin are non-zero (`wide`; shallow nets).  Deep nets get small integers: the grid of a row
    scales the bound of every layer, and 21 layers leave no room for a fine one."""
    fb = synth.random_feature_bitboards(BASE * in_channels, seed=seed).reshape(BASE, in_channels)
    rng = np.random.default_rng(seed)
    ns = in_channels - FIRST_SCALAR
    if wide:
        val = rng.choice(np.array([1.0, 1.0, 1.0, 0.5, 1.5, 2.0, 0.25]), size=(BASE, in_channels))
        val[:, FIRST_SCALAR:] = rng.integers(257, 4096, size=(BASE, ns)) / 256.0
    else:
        val = rng.choice(np.array([1.0, 1.0, 1.0, 2.0]), size=(BASE, in_channels))
        val[:, FIRST_SCALAR:] = rng.integers(0, 8, size=(BASE, ns))
    bits = val.astype(np.float32).view(np.uint32).astype(np.uint64)
    fb["hi"] = (fb["hi"] & np.uint64(0xFFFFFFFF)) | (bits << np.uint64(32))
    return np.ascontiguousarray(fb.reshape(-1))


def position_inputs(synth, seed, wide):
    """BASE packed positions whose scalar planes are dyadic: max_ply a power of two (or 1), so ply / max_ply is exact,
    and dyadic draw values.  In the shallow nets' inputs (`wide`) a third of the positions carry integer draw values
    from 257 to 1023 with low bits set (both halves of the twin non-zero); they have max_ply = 1, so that their grid stays
    1.  The deep nets' inputs have max_ply 1 or 2 and small integer draw values (see bitboard_inputs)."""
    pos = synth.random_positions(BASE, seed=seed)
    rng = np.random.default_rng(seed)
    big = np.arange(BASE) % 3 == 0
    mp = np.where(big, 1, rng.choice(np.array([2, 4, 8, 256]) if wide else np.array([1, 2]), size=BASE))
    pos["max_ply"] = mp
    pos["ply"] = rng.integers(0, 1 << 16, size=BASE) % mp
    for key in ("black_draw_value", "white_draw_value"):
        v = rng.integers(0, 16, size=BASE) / 8.0 if wide else rng.integers(0, 4, size=BASE) * 1.0
        if wide:
            v[big] = rng.integers(257, 1024, size=int(big.sum()))
        pos[key] = v.astype(np.float32)
    return pos


# ---- fixtures -----------------------------------------------------------------------------------------------------
_NETS = {}


def exact_net(nb, synth, orc, name):
    """(desc, blob, stats, inputs) of NETS[name], built once per session.  inputs: {"fb": bitboards, "pos": positions or
    None, "planes": the oracle's planes of both}.  A draw that fails the bound is re-drawn with the next weight seed."""
    if name not in _NETS:
        C, NB, IN, density, wseed, iseed = NETS[name]
        desc = nb.net_desc(C, NB, in_channels=IN)
        wide = NB <= 2
        fb = bitboard_inputs(synth, IN, iseed, wide)
        planes = orc.expand(fb, BASE, IN)
        pos = None
        if IN == 86:
            pos = position_inputs(synth, iseed, wide)
            planes = np.concatenate([planes, orc.expand(orc.pack(pos), BASE)])
        for seed in range(wseed, wseed + 8):
            try:
                blob, stats = exact_blob(desc, seed, planes, density)
                break
            except AssertionError as e:
                err = e
        else:
            raise AssertionError(f"{name}: no weight seed satisfies the bound: {err}")
        _NETS[name] = (desc, blob, stats, {"fb": fb, "pos": pos, "planes": planes})
    return _NETS[name]


# ---- CPU: the premise, and that the tests are not vacuous -----------------------------------------------------------
@pytest.mark.parametrize("name", list(NETS))
def test_generator_is_exact_and_not_vacuous(nb, synth, orc, name):
    desc, blob, stats, inp = exact_net(nb, synth, orc, name)
    w = helpers.split_blob(desc, blob)
    convs = [w["stem_w"]] + [c for blk in w["blocks"] for c in (blk[0], blk[2])]
    for i, c in enumerate(convs):
        nz = c != 0
        assert nz.any(axis=(1, 2, 3)).all(), f"conv {i}: an output channel without weights"
        assert nz.any(axis=(0, 1)).all(), f"conv {i}: a tap without weights"
        kb = nz.any(axis=(0, 2, 3))
        assert all(kb[k:k + 16].any() for k in range(0, c.shape[1], 16)), f"conv {i}: a 16-channel K block without weights"
    assert (w["pol_b"] != 0).all() and w["val_b"][0] != 0
    assert (w["fc2_w"][:, [0, desc.value_hidden - 1]] != 0).all()              # FC2 reads the first and last hidden unit
    for i, layer in enumerate(stats["layers"]):
        assert 0.2 <= layer["nonzero"] <= 0.8, (i, layer)
    assert sum(layer["rounded"] > 0 for layer in stats["layers"]) >= 3        # bf16 rounding really happens
    assert sum(layer["ties"] for layer in stats["layers"]) > 0                 # ... exact ties included
    assert np.abs(stats["pre_sigmoid"]).max() < 8
    _, win, draw = orc.forward(desc, blob, inp["planes"], emulate_bf16=True)
    assert np.ptp(win) > 1e-2 and np.ptp(draw) > 1e-2, "dead value head"
    # the twins carry something wherever the inputs have more than 8 significant bits
    if NETS[name][1] <= 2 and desc.in_channels > FIRST_SCALAR:
        assert (stem_input(inp["planes"], desc.in_channels)[:, desc.in_channels:] != 0).any()


@pytest.mark.parametrize("name", list(NETS))
def test_oracle_equals_float64_forward_bit_for_bit(nb, synth, orc, name):
    """The premise: the oracle (fp32, its own accumulation order) equals a float64 torch forward (another order) bit for
    bit on the exact nets - logits; win / draw within the ulps of expf."""
    desc, blob, _, inp = exact_net(nb, synth, orc, name)
    pb, wb, db = orc.forward(desc, blob, inp["planes"], emulate_bf16=True)
    pol, o = forward64(desc, blob, inp["planes"])
    assert np.array_equal(pb.astype(np.float64), pol)
    for got, z in ((wb, o[:, 0]), (db, o[:, 1])):
        assert ulps(got, (1.0 / (1.0 + np.exp(-z))).astype(np.float32)).max() <= 4


def test_random_net_is_not_exact(nb, synth, orc):
    """Negative control: on a random-init net the accumulation order shows, so the equality above is not automatic."""
    desc = nb.net_desc(128, 2)
    blob = nb.random_blob(desc, 1234)
    planes = orc.expand(orc.pack(synth.random_positions(8, seed=3)), 8)
    pb, _, _ = orc.forward(desc, blob, planes, emulate_bf16=True)
    pol, _ = forward64(desc, blob, planes)
    assert not np.array_equal(pb.astype(np.float64), pol)


def ulps(a, b):
    """Distance in units in the last place between float32 arrays of one sign."""
    return np.abs(np.asarray(a, np.float32).view(np.int32).astype(np.int64) - np.asarray(b, np.float32).view(np.int32))


# ---- GPU: every trunk kernel against the oracle, bit for bit ------------------------------------------------------
SIZES = (1, 3, 5, 601)   # idle slots in the last group / pair / quad, and a second pass on every kernel
# DECODE_PROBS is held to the float64 softmax of the oracle's logits (bit-exact inputs of the softmax).  The kernel's fp32
# softmax of a row of m <= 593 moves - expf (2 ulp), a sum of <= 19 terms per lane and a 5-level butterfly, a reciprocal
# and a product - is within about 33 u of it (u = 2^-24); the limit doubles that.  orc.decode at the rtol 1e-6 of
# test_decode_matches_oracle is not the yardstick here: its serial fp32 sum differs from the kernel's order alone by up to
# 1.6e-6 on 593-move rows of these nets, where the probabilities are too large for that test's atol to absorb it.
TOL_PROBS_REL = 2.0 ** -18

# kernel -> (NSB_TRUNK128, NSB_TRUNK256, slots, diag, trunk_kernel_name (the fused kernels' exactly, else its prefix), nets)
# The *_1slot rows are the kernel choices of one-slot 128-channel contexts: the duo and quad kernels forced, and unforced,
# where each batch runs on trunk_fused_kernel<128> or trunk_duo_kernel (two weight streams, chosen by batch size).
KERNELS = {
    "classic": ("classic", None, 1, False, "trunk_fused_kernel<128>", ["128x2", "128x10", "128x2c93"]),
    "duo": (None, None, 2, False, "trunk_duo_kernel", ["128x2", "128x10"]),
    "quad": (None, None, 4, False, "trunk_quad_kernel", ["128x2", "128x10", "128x2c93"]),
    "duo_1slot": ("duo", None, 1, False, "trunk_duo_kernel", ["128x2", "128x10"]),
    "quad_1slot": ("quad", None, 1, False, "trunk_quad_kernel", ["128x2", "128x10"]),
    "auto_1slot": (None, None, 1, False,
                   "trunk_fused_kernel<128> (trunk_duo_kernel for batches where two CTAs per SM are faster)", ["128x2", "128x10"]),
    "pair": (None, None, 1, False, "trunk_pair_kernel", ["256x2", "256x10", "192x2", "192x10", "256x2c93"]),
    "single256": (None, "single", 1, True, "trunk_fused_kernel<256>", ["256x2", "256x10"]),
}
CASES = [(k, n) for k, v in KERNELS.items() for n in v[5]]


def _tile(a, n, per_row):
    """Row i of the batch is distinct input i % BASE."""
    idx = np.arange(n) % BASE
    return np.ascontiguousarray(a.reshape(BASE, -1)[idx].reshape(-1) if per_row else a[idx])


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,name", CASES)
def test_kernel_equals_oracle_bit_for_bit(nb, synth, orc, monkeypatch, kernel, name):
    t128, t256, slots, diag, kname, _ = KERNELS[kernel]
    desc, blob, _, inp = exact_net(nb, synth, orc, name)
    for var, val in (("NSB_TRUNK128", t128), ("NSB_TRUNK256", t256)):
        if val:
            monkeypatch.setenv(var, val)
        else:
            monkeypatch.delenv(var, raising=False)
    op, ow, od = orc.forward(desc, blob, inp["planes"], emulate_bf16=True)
    paths = [("bitboards", 0)] + ([("positions", BASE)] if inp["pos"] is not None else [])
    nmax = max(SIZES)
    off, idx = synth.random_legal_moves(nmax, seed=len(name), edge_rows=True)
    with nb.Context(desc, batch_max=nmax, slots=slots, blob=blob, diag=diag) as ctx:
        name_ = ctx.trunk_kernel_name()
        assert name_ == kname if kname.startswith("trunk_fused") else name_.startswith(kname), name_
        for path, r0 in paths:
            for n in SIZES:
                rows = r0 + np.arange(n) % BASE
                wp, ww, wd = op[rows], ow[rows], od[rows]
                o, ix = off[:n + 1], idx[:int(off[n])]
                policy = np.zeros((n, nb.POLICY_SIZE), dtype=np.float32)
                win, draw = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
                legal = {m: np.zeros(int(o[-1]), dtype=np.float32) for m in (nb.DECODE_LOGITS, nb.DECODE_PROBS)}
                w2, d2 = np.zeros(n, dtype=np.float32), np.zeros(n, dtype=np.float32)
                slot = n % slots
                if path == "bitboards":
                    fb = _tile(inp["fb"], n, True)
                    ctx.eval_async(slot, fb, n, policy, win, draw)
                    ctx.await_(slot)
                    for m in legal:
                        ctx.eval_decode_async(slot, fb, n, o, ix, m, legal[m], w2, d2, None)
                        ctx.await_(slot)
                else:
                    pos = _tile(inp["pos"], n, False)
                    ctx.eval_positions_async(slot, pos, n, policy, win, draw)
                    ctx.await_(slot)
                    for m in legal:
                        ctx.eval_positions_decode_async(slot, pos, n, o, ix, m, legal[m], w2, d2, None)
                        ctx.await_(slot)
                where = (kernel, name, path, n)
                bad = np.nonzero((policy.view(np.uint32) != wp.view(np.uint32)).any(axis=1))[0]
                assert bad.size == 0, (where, "rows with logits != oracle", bad[:8],
                                       int((policy != wp).sum()), float(np.abs(policy - wp).max()))
                assert ulps(win, ww).max() <= 4 and ulps(draw, wd).max() <= 4, (where, ulps(win, ww).max(), ulps(draw, wd).max())
                assert np.array_equal(w2, win) and np.array_equal(d2, draw), where   # the decode launches' value head
                want_logits, _ = orc.decode(wp, ww, wd, o, ix, nb.DECODE_LOGITS)
                assert np.array_equal(legal[nb.DECODE_LOGITS].view(np.uint32), want_logits.view(np.uint32)), where
                want_probs = helpers.softmax_rows(wp, o, ix)
                assert np.allclose(legal[nb.DECODE_PROBS], want_probs, rtol=TOL_PROBS_REL, atol=1e-30), where
