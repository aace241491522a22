"""Deterministic, integer-only synthetic luma frames and int8 models (SURVEY.md section 8d).

The reference ships neither YUV sequences nor trained int8 weights (inference/kernel.cu:7-10
points at the author's D: drive), only the per-QP blu/mul/shift triples.  Everything here is
derived from one 64-bit seed with a splitmix64-style hash of (seed, stream, a, b, c) so the same
frames / weights can be rebuilt anywhere (numpy here, C++ in csrc/qv_synth.hpp).
"""
from __future__ import annotations

import numpy as np

from .formats import LAYERS, Model, SHIPPED_QPARAMS

_GOLD = np.uint64(0x9E3779B97F4A7C15)
_M1 = np.uint64(0xBF58476D1CE4E5B9)
_M2 = np.uint64(0x94D049BB133111EB)


def _mix(z):
    z = (z ^ (z >> np.uint64(30))) * _M1
    z = (z ^ (z >> np.uint64(27))) * _M2
    return z ^ (z >> np.uint64(31))


def hash5(seed, stream, a, b, c):
    """h(seed, stream, a, b, c) -> uint64 (broadcasts over numpy arrays)."""
    with np.errstate(over="ignore"):
        k = _mix(np.uint64(seed) + _GOLD * np.uint64(stream + 1))
        k = _mix(k + _GOLD * (np.asarray(a).astype(np.uint64) + np.uint64(1)))
        k = _mix(k + _GOLD * (np.asarray(b).astype(np.uint64) + np.uint64(1)))
        k = _mix(k + _GOLD * (np.asarray(c).astype(np.uint64) + np.uint64(1)))
    return k


def make_frames(seed: int, frames: int, h: int, w: int, first_frame: int = 0, rows=None):
    """Returns (anchor, ori) u8 [frames,h,w].  anchor = blocky 16x16 content + 5-bit noise
    (what an intra-coded frame looks like to the net); ori = anchor + small noise so that the
    'before net' PSNR is finite.  rows = (y0, y1): only those rows of the h-row frames (a strip's share)."""
    f = (np.arange(frames, dtype=np.uint64) + np.uint64(first_frame))[:, None, None]
    y = (np.arange(h, dtype=np.uint64) if rows is None else np.arange(rows[0], rows[1], dtype=np.uint64))[None, :, None]
    x = np.arange(w, dtype=np.uint64)[None, None, :]
    base = (hash5(seed, 0, f, y >> np.uint64(4), x >> np.uint64(4)) & np.uint64(0xFF)).astype(np.int32)
    noise = (hash5(seed, 1, f, y, x) & np.uint64(0x1F)).astype(np.int32) - 16
    anchor = np.clip(base + noise, 0, 255)
    d = (hash5(seed, 2, f, y, x) & np.uint64(7)).astype(np.int32) - 3
    ori = np.clip(anchor + d, 0, 255)
    return anchor.astype(np.uint8), ori.astype(np.uint8)


def make_uniform_frames(seed: int, frames: int, h: int, w: int):
    f = np.arange(frames, dtype=np.uint64)[:, None, None]
    y = np.arange(h, dtype=np.uint64)[None, :, None]
    x = np.arange(w, dtype=np.uint64)[None, None, :]
    return (hash5(seed, 3, f, y, x) & np.uint64(0xFF)).astype(np.uint8)


# Per-layer weight / bias amplitudes, calibrated once against the oracle on 416x240 synthetic
# frames so that hidden activations have roughly 30-70 % zeros and a few % saturated to 127 and
# the C4 residual spans about +-8 (see tests/test_synth.py for the recorded statistics).
# Bound kept by construction: 128*sum|w| + |b| < 2^24 per output channel (SURVEY fact 7).
WEIGHT_AMPL = {
    # (weight amplitude A, bias amplitude B[, bias offset b0]) : w in [-A,A], b in b0 + [-B,B]
    # QP22's shipped C4 pair is the stale mul=5, shift=24 (SURVEY fact 9): the residual is non-zero
    # only for |u4| > 1.68e6, so its C4 bias is centred on that threshold to exercise the path.
    22: ((20, 1500), (5, 1500), (4, 2000), (12, 6000), (7, 1500), (127, 60_000, 1_690_000)),
    27: ((40, 3000), (8, 2500), (10, 5000), (6, 2500), (8, 2000), (24, 4000)),
    32: ((48, 4000), (12, 4000), (8, 4000), (6, 2500), (6, 1500), (24, 4000)),
    37: ((52, 4000), (12, 4000), (8, 4000), (11, 5000), (10, 2500), (12, 6000)),
}


def make_model(seed: int, qp: int, ampl=None) -> Model:
    """Synthetic int8 model carrying the SHIPPED blu/mul/shift for `qp`."""
    ampl = ampl or WEIGHT_AMPL[qp]
    m = Model()
    for l, (cin, cout, k) in enumerate(LAYERS):
        A, B = ampl[l][0], ampl[l][1]
        b0 = ampl[l][2] if len(ampl[l]) > 2 else 0
        kk = np.arange(cout, dtype=np.uint64)[:, None, None]
        cc = np.arange(cin, dtype=np.uint64)[None, :, None]
        tt = np.arange(k * k, dtype=np.uint64)[None, None, :]
        hw = hash5(seed, 10 + l, kk, cc, tt)
        w = (hw % np.uint64(2 * A + 1)).astype(np.int64) - A
        # a sprinkling of exact zeros and of full-scale taps, like a trained, pruned filter bank
        sel = (hw >> np.uint64(40)) & np.uint64(15)
        w = np.where(sel == 0, 0, w)
        w = np.clip(w, -128, 127).astype(np.int8).reshape(cout, cin, k, k)
        hb = hash5(seed, 20 + l, np.arange(cout, dtype=np.uint64), 0, 0)
        b = ((hb % np.uint64(2 * B + 1)).astype(np.int64) - B + b0).astype(np.int32)
        bound = 128 * np.abs(w.astype(np.int64)).reshape(cout, -1).sum(1) + np.abs(b.astype(np.int64))
        assert int(bound.max()) < (1 << 24), (l, int(bound.max()))
        m.w.append(w)
        m.b.append(b)
        m.qparams.append(tuple(SHIPPED_QPARAMS[qp][l]))
    m.check()
    return m


# ---- edge models: the corners of the admissible model space ---------------------------------------------------------
# qv_load_static_para accepts every model with 128*sum|w| + |b| < 2^24 per output channel and 0 <= blu < 2^24, mul > 0,
# 1 <= shift <= 30 per layer, and promises the reference's results bit for bit on all of them.  The calibrated models above
# use a few percent of that space; these generators reach its edges.  Every one is built layer by layer against a small
# calibration frame so that what it claims to exercise (saturation, zeros, intermediate values, wraps) really happens.
#   full_scale         taps from {-128, 127, small, 0}, every output channel at exactly 128*sum|w| + |b| = 2^24 - 1
#   saturated_padding  hidden biases above blu: every in-image activation is 127, every out-of-image one must stay 0
#   dead_layers        C2_2, C3_1 and C3_2 output 0 everywhere: u4 == the C4 bias, the frame is clamp(x + t)
#   quant_rows         a seeded sweep of hidden requantiser rows; the variant decides which rows pass the fast path's
#                      precondition: "fast" (all five, shifts 1..24 over seeds 0..4), "generic" (none) or
#                      "one_generic" (exactly layer seed % 5 fails)
#   c4_wrap            C4 rows with mul near 2^31: u4 * mul wraps int32 and x + t leaves the range of a short
# The variant "generic" of the other families replaces the five hidden rows by rows that fail the precondition, so that the
# same model runs through the fused kernels' generic requantiser.
EDGE_FAMILIES = ("full_scale", "saturated_padding", "dead_layers", "quant_rows", "c4_wrap")
ENVELOPE = (1 << 24) - 1
HIDDEN = (0, 1, 2, 3, 4)                       # C1, C2_1, C2_2, C3_1, C3_2
GENERIC_KINDS = ("big_shift", "not_127", "wrap_neg")


def fast_row_ok(blu: int, mul: int, shift: int) -> bool:
    """The precondition of the fused kernel's fast requantiser (qv_fused.cu, build_host_image: mkq)."""
    rb = (1 << (shift - 1)) // mul
    top = (blu + rb) * mul
    return shift <= 24 and mul < (1 << shift) and top < (1 << 31) and (top >> shift) == 127 and blu + rb < (1 << 30)


def _fast_row(T: int, shift: int):
    """A row that satisfies fast_row_ok with blu as close to T as the shift allows."""
    mul = int(min(max(round(127.5 * (1 << shift) / max(T, 1)), 1), (1 << shift) - 1))
    rb = (1 << (shift - 1)) // mul
    lo = -(-(127 << shift) // mul) - rb
    hi = -(-(128 << shift) // mul) - 1 - rb
    blu = int(min(max(T, lo, 0), hi, ENVELOPE))
    assert fast_row_ok(blu, mul, shift), (T, blu, mul, shift)
    return blu, mul, shift


def _generic_row(kind: str, T: int, rng):
    """A row with blu = T that fails fast_row_ok: shift 25..30 ("big_shift"), BLU(blu) ~ 100 ("not_127") or a BLU(blu) of
    ~200, which the (char) store wraps to a negative activation ("wrap_neg")."""
    T = int(min(max(T, 64), ENVELOPE))
    if kind == "big_shift":
        shift = int(rng.integers(25, 31))
        mul = max(1, ((1 << 31) - 1) // (2 * T + 2))
        return T, mul, shift
    shift = int(min(max(int(np.log2(T)) - 3 + int(rng.integers(0, 3)), 1), 22))      # mul of 12 .. 100
    top = 100 if kind == "not_127" else 200
    mul = int(max(round(top * (1 << shift) / T), 1))
    row = (T, mul, shift)
    assert mul >= 1 and not fast_row_ok(*row), (kind, row)
    return row


def _conv_acc(a: np.ndarray, w: np.ndarray) -> np.ndarray:
    """int64 cross-correlation with zero padding (k-1)/2; a [C,H,W], w [K,C,k,k] -> [K,H,W]."""
    K, C, k, _ = w.shape
    p = (k - 1) // 2
    _, H, W = a.shape
    ap = np.pad(a.astype(np.int64), ((0, 0), (p, p), (p, p)))
    cols = np.stack([ap[:, r:r + H, s:s + W] for r in range(k) for s in range(k)], axis=1).reshape(C * k * k, H * W)
    return (w.astype(np.int64).reshape(K, C * k * k) @ cols).reshape(K, H, W)


def _blu(u: np.ndarray, blu: int, mul: int, shift: int) -> np.ndarray:
    """The hidden-layer requantiser of the reference (inference/mat.cu:262-303), for calibration only."""
    rb = (1 << (shift - 1)) // mul
    prod = ((u + rb) * mul) & 0xFFFFFFFF
    prod = np.where(prod >= 1 << 31, prod - (1 << 32), prod)
    q = (prod >> shift) & 0xFF
    q = np.where(q >= 128, q - 256, q)
    return np.where(u > blu, 127, np.where(u < 0, 0, q))


def _full_bias(w: np.ndarray, sign: np.ndarray) -> np.ndarray:
    """Biases that put every output channel exactly at the envelope edge: 128*sum|w| + |b| = 2^24 - 1."""
    s = np.abs(w.astype(np.int64)).reshape(w.shape[0], -1).sum(1)
    assert (128 * s <= ENVELOPE).all()
    return (sign * (ENVELOPE - 128 * s)).astype(np.int32)


def _full_scale_weights(rng, l: int) -> np.ndarray:
    cin, cout, k = LAYERS[l]
    n = cin * k * k
    # per channel a share p of -128 and of 127 taps (C2_2's 1600 taps cannot all be full scale inside the envelope): the
    # channels' biases, and with them the positive u, spread over the top of the envelope
    p = rng.uniform(0.03, 0.15 if l == 2 else 0.45, size=(cout, 1))
    r = rng.random((cout, n))
    cat = np.where(r < p, 0, np.where(r < 2 * p, 1, np.where(r < 0.5 + p, 2, 3)))
    small = rng.integers(1, 9, size=(cout, n)) * rng.choice([-1, 1], size=(cout, n))
    w = np.select([cat == 0, cat == 1, cat == 2], [-128, 127, small], 0).astype(np.int64)
    for c in range(cout):                          # trim until the channel fits the envelope
        while 128 * np.abs(w[c]).sum() > ENVELOPE:
            w[c, rng.integers(0, n)] = 0
    if l in (1, 3, 4):                             # all-full-scale filters: all 127 and all -128
        w[0] = 127
        w[1] = -128
    return w.reshape(cout, cin, k, k).astype(np.int8)


def _scaled_weights(rng, l: int, a_in: np.ndarray, target: float) -> np.ndarray:
    """Random weights whose accumulators on a_in spread about `target` (as far as int8 weights allow)."""
    cin, cout, k = LAYERS[l]
    w127 = rng.integers(-127, 128, size=(cout, cin, k, k))
    w127 = np.where(rng.random(w127.shape) < 0.1, 0, w127)
    sd = float(_conv_acc(a_in, w127).std()) or 1.0
    a = min(max(target / sd, 1.0 / 127), 1.0)
    return np.clip(np.rint(w127 * a), -127, 127).astype(np.int8)


def _c4_row(rng, u4: np.ndarray):
    """A C4 row that keeps t = (u4 * mul + 2^(shift-1)) >> shift in the tens for most pixels, without wraps."""
    sd = max(float(u4.std()), 1.0)
    lo = max(1, int(np.ceil(np.log2(max(sd / 40, 1)))))
    shift = int(rng.integers(lo, min(lo + 12, 30) + 1))
    mul = max(1, int(round(40 * (1 << shift) / sd)))
    while mul > 1 and int(np.abs(u4).max()) * mul >= (1 << 30):
        mul //= 2
    return 0, mul, shift


def make_edge_model(seed: int, family: str, variant: str = "fast", calib=None) -> Model:
    """A seeded model of one of EDGE_FAMILIES, inside the envelope.  variant: "fast" | "generic" (| "one_generic" for
    quant_rows), see the table above.  `calib` (u8 [H,W]) is the frame the activations are calibrated on."""
    assert family in EDGE_FAMILIES and variant in ("fast", "generic", "one_generic"), (family, variant)
    assert variant != "one_generic" or family == "quant_rows"
    rng = np.random.default_rng([seed, EDGE_FAMILIES.index(family), ("fast", "generic", "one_generic").index(variant)])
    x = make_uniform_frames(seed, 1, 24, 48)[0] if calib is None else calib
    xp = x.astype(np.int64)[None] - 128
    m = Model()
    m.w, m.b, m.qparams = [None] * 6, [None] * 6, [None] * 6
    kinds = {}                                     # hidden layer -> "fast" | one of GENERIC_KINDS
    for j, l in enumerate(HIDDEN):
        if variant == "fast" or (variant == "one_generic" and l != seed % 5):
            kinds[l] = "fast"
        else:
            kinds[l] = GENERIC_KINDS[(j + seed) % 3]
    shifts = {l: (5 * seed + j) % 24 + 1 for j, l in enumerate(HIDDEN)}          # quant_rows: the shift sweep

    def row_for(l, T):
        if kinds[l] != "fast":
            return _generic_row(kinds[l], T, rng)
        if family == "quant_rows":
            return _fast_row(T, shifts[l])
        ok = [s for s in range(1, 25) if 1 <= round(127.5 * (1 << s) / max(T, 1)) < (1 << s)]
        exact = [s for s in ok if _fast_row(T, s)[0] == T]                # shifts fine enough to put blu at T
        return _fast_row(T, int(rng.choice(exact or ok)))

    def hidden(l, a_in):
        cin, cout, k = LAYERS[l]
        if family == "full_scale":
            w = _full_scale_weights(rng, l)
            sign = np.where(rng.random(cout) < (0.6 if l == 0 else 0.5), 1, -1)
            if l in (1, 3, 4):
                sign[0] = 1
            b = _full_bias(w, sign)
            u = _conv_acc(a_in, w) + b[:, None, None]
            # blu at the 60th percentile of the positive u: saturated, zero and intermediate activations in every layer
            row = row_for(l, int(np.quantile(u[u > 0], 0.6)) if (u > 0).any() else 1 << 20)
        else:
            T = int(2 ** rng.uniform(9, 20))
            if family == "quant_rows" and kinds[l] == "fast":
                T = min(T, 100 << shifts[l])
            if family == "dead_layers":                       # room for a bias below -128 * sum|w|
                T = min(T, 1 << 12)
            row = row_for(l, T)
            T = row[0]
            w = _scaled_weights(rng, l, a_in, T)
            s = np.abs(w.astype(np.int64)).reshape(cout, -1).sum(1)
            if family == "saturated_padding":              # |acc| <= 128 * sum|w|: u > blu for every input
                b = (T + 1 + 128 * s + rng.integers(0, 1000, cout)).astype(np.int32)
            elif family == "dead_layers" and l in (2, 3, 4):  # u < 0 for every input
                b = (-(128 * s + 1) - rng.integers(0, 1000, cout)).astype(np.int32)
            else:
                b = rng.integers(-T // 2, T // 2 + 1, cout).astype(np.int32)
            u = _conv_acc(a_in, w) + b[:, None, None]
        m.w[l], m.b[l], m.qparams[l] = w, b, tuple(int(v) for v in row)
        return _blu(u, *row)

    a1 = hidden(0, xp)
    a2 = np.concatenate([hidden(1, a1), hidden(2, a1)])
    a3 = np.concatenate([hidden(3, a2), hidden(4, a2)])
    # ---- C4 ----
    cin, cout, k = LAYERS[5]
    if family == "full_scale":
        w4 = _full_scale_weights(rng, 5)
        b4 = _full_bias(w4, np.array([1 if rng.random() < 0.5 else -1]))
        # |b4| >= 2^24 - 1 - 128 * 432 * 128 puts u4 far from 0; an odd mul near 2^31 and shift 24 make t a hash of u4
        # in [-128, 127] instead, so that every bit of u4 shows in the frame
        q4 = (0, int(rng.integers(1 << 29, 1 << 30)) * 2 + 1, 24)
    elif family == "c4_wrap":
        w4 = rng.integers(-127, 128, size=(1, cin, k, k)).astype(np.int8)
        w4.reshape(-1)[rng.integers(0, cin * k * k)] = -128
        b4 = np.zeros(1, np.int32)
        # mul = 2^31 - 1 - 2j: for even u4 the product wraps to about -u4 (t small: interior values and both clamps), for
        # odd u4 to about -u4 - 2^31 (t near -2^(31-shift): x + t leaves the short range and the (short) wraps it back)
        q4 = (0, (1 << 31) - 1 - 2 * int(rng.integers(0, 64)), int(rng.integers(13, 17)))
    else:
        w4 = np.clip(rng.integers(-24, 25, size=(1, cin, k, k)), -127, 127).astype(np.int8)
        u4 = _conv_acc(a3, w4)[0]
        if family == "saturated_padding":           # a3 is 127 inside the image: centre the interior's u4 on 0
            b4 = np.array([-int(u4[u4.shape[0] // 2, u4.shape[1] // 2]) + int(rng.integers(-3000, 3001))], np.int32)
            q4 = _c4_row(rng, u4 + int(b4[0]))
        elif family == "dead_layers":               # u4 == b4 everywhere: t = +-(40..120)
            q4 = (0, 1, 12)
            t = int(rng.integers(40, 121)) * (1 if seed % 2 == 0 else -1)
            b4 = np.array([t << 12], np.int32)
        else:
            b4 = rng.integers(-2000, 2001, 1).astype(np.int32)
            q4 = _c4_row(rng, u4 + int(b4[0]))
    m.w[5], m.b[5], m.qparams[5] = w4, b4, tuple(int(v) for v in q4)
    for l, (w, b) in enumerate(zip(m.w, m.b)):
        bound = 128 * np.abs(w.astype(np.int64)).reshape(w.shape[0], -1).sum(1) + np.abs(b.astype(np.int64))
        assert int(bound.max()) <= ENVELOPE, (family, variant, l, int(bound.max()))
    m.check()
    return m


def edge_models():
    """(id, seed, family, variant) of every edge model the suites run."""
    out = []
    for fam in ("full_scale", "saturated_padding", "dead_layers", "c4_wrap"):
        for var in ("fast", "generic"):
            out.append(("%s-%s" % (fam, var), 7, fam, var))
    for s in range(5):
        out.append(("quant_rows-fast-%d" % s, s, "quant_rows", "fast"))
        out.append(("quant_rows-one_generic-%d" % s, s, "quant_rows", "one_generic"))
    for s in range(2):
        out.append(("quant_rows-generic-%d" % s, s, "quant_rows", "generic"))
    return out
