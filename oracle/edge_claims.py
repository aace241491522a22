"""What each edge model (qcnn_gpu_b200.host.synth.make_edge_model) claims to exercise, checked on the C oracle's taps.
TEST INFRASTRUCTURE: a parity test on an edge model only means something if the model really reaches the corner it names,
so every test that runs one also runs these checks on one of its frames."""
from __future__ import annotations

import numpy as np

from oracle import oracle_np
from qcnn_gpu_b200.host import synth

ENVELOPE = (1 << 24) - 1


def _bounds(model):
    return [128 * np.abs(w.astype(np.int64)).reshape(w.shape[0], -1).sum(1) + np.abs(b.astype(np.int64))
            for w, b in zip(model.w, model.b)]


def check_rows(model, seed, family, variant):
    """Inside the envelope, and the rows pass the fast path's precondition exactly where the variant says."""
    assert all(int(b.max()) <= ENVELOPE for b in _bounds(model))
    for l, (blu, mul, shift) in enumerate(model.qparams):
        assert mul > 0 and 1 <= shift <= 30 and (l == 5 or 0 <= blu < 1 << 24), (l, blu, mul, shift)
    fast = [synth.fast_row_ok(*q) for q in model.qparams[:5]]
    if variant == "fast":
        assert all(fast)
    elif variant == "generic":
        assert not any(fast)
    else:
        assert fast == [l != seed % 5 for l in range(5)]
    if family == "quant_rows" and variant == "fast":
        assert [q[2] for q in model.qparams[:5]] == [(5 * seed + j) % 24 + 1 for j in range(5)]
    return all(fast)


def check_claims(model, seed, family, variant, x, taps):
    """x: u8 [H,W]; taps: (rec, a1, a2, a3, u4) of the C oracle on x.  Frames of a few thousand pixels or more."""
    rec, a1, a2, a3, u4 = taps
    check_rows(model, seed, family, variant)
    layers = [a1, a2[:32], a2[32:], a3[:16], a3[16:]]           # C1, C2_1, C2_2, C3_1, C3_2
    if family == "full_scale":
        assert all((w == -128).any() for w in model.w)
        assert all((b == ENVELOPE).all() for b in _bounds(model))
        signs = np.concatenate([np.sign(b) for b in model.b])
        assert (signs > 0).any() and (signs < 0).any()
        acc = [oracle_np._conv_acc(a1, model.w[1]), oracle_np._conv_acc(a1, model.w[2]),
               oracle_np._conv_acc(a2, model.w[3]), oracle_np._conv_acc(a2, model.w[4])]
        assert max(int(np.abs(a).max()) for a in acc) >= 1 << 22
        if variant == "fast":
            for l, a in enumerate(layers):
                assert (a == 127).mean() >= 0.01 and (a == 0).mean() >= 0.01 and ((a > 0) & (a < 127)).mean() >= 0.10, l
    elif family == "saturated_padding":
        for l, a in enumerate(layers):
            assert (a == 127).all(), l
    elif family == "dead_layers":
        assert (a2[32:] == 0).all() and (a3 == 0).all()
        assert (u4 == int(model.b[5][0])).all()
        _, mul, shift = model.qparams[5]
        t = (int(model.b[5][0]) * mul + (1 << (shift - 1))) >> shift
        assert t != 0 and np.array_equal(rec, np.clip(x.astype(np.int64) + t, 0, 255))
    elif family == "c4_wrap":
        _, mul, shift = model.qparams[5]
        prod = u4.astype(np.int64) * mul + (1 << (shift - 1))
        assert ((prod >= 1 << 31) | (prod < -(1 << 31))).any()               # u4 * mul wraps int32
        p32 = prod & 0xFFFFFFFF
        t = np.where(p32 >= 1 << 31, p32 - (1 << 32), p32) >> shift
        r = x.astype(np.int64) + t
        assert (np.abs(r) > 32767).any()                                     # the (short) wraps
        r16 = ((r + 32768) & 0xFFFF) - 32768
        assert (np.clip(r16, 0, 255) != np.clip(r, 0, 255)).any()           # ... and that changes the result
        assert (rec == 0).any() and (rec == 255).any() and ((rec > 0) & (rec < 255)).any()
    # a row whose BLU(blu) lies in (127, 256) stores negative chars (in the families whose u is not forced to one side)
    wraps = [q[2] <= 24 and 127 < ((q[0] + (1 << (q[2] - 1)) // q[1]) * q[1]) >> q[2] < 256 for q in model.qparams[:5]]
    if family in ("full_scale", "quant_rows", "c4_wrap") and any(wraps):
        assert any((a < 0).any() for a in layers)
