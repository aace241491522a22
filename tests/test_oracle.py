"""Pins the C oracle (oracle/qvrcnn_oracle.c).  The reference holds no golden vectors for this
path (SURVEY 8c), so the oracle is pinned by (1) an independent torch/numpy restatement,
(2) hand-computable known-answer cases of each fixed-point formula, (3) algebraic properties,
(4) committed golden checksums, and (5) when present, recon frames produced by the unmodified
reference sources run on a B200 (tests/golden/ref_witness_*.npz, see test_ref_witness.py)."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import oracle, oracle_np
from qcnn_gpu_b200.host import formats, synth

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _om(model):
    return oracle.OracleModel(formats.write_model_vect_c(model))


@pytest.mark.parametrize("qp", [22, 27, 32, 37])
def test_c_oracle_equals_numpy_restatement(models, qp):
    m = models[qp]
    anchor, _ = synth.make_frames(0xC0FFEE, 1, 48, 80)
    rec, a1, a2, a3, u4 = _om(m).forward_taps(anchor[0])
    ref = oracle_np.forward_frame(m, anchor[0])
    for name, got in dict(rec=rec, a1=a1, a2=a2, a3=a3, u4=u4).items():
        assert np.array_equal(got, ref[name]), name
    # the synthetic weights exercise the interesting branches
    assert 0.2 < (a1 == 0).mean() < 0.8 and (a1 == 127).mean() > 0.01
    assert (rec != anchor[0]).any()


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (5, 3), (13, 13), (6, 130)])
def test_ragged_and_tiny_frames(models, shape):
    """Frames smaller than the receptive field (radius 6): every tap hits zero padding."""
    m = models[37]
    x = synth.make_uniform_frames(3, 1, *shape)[0]
    rec = _om(m).forward_blu(x[None])[0]
    assert np.array_equal(rec, oracle_np.forward_frame(m, x)["rec"])


def test_blu_known_answers():
    """BLU (inference/mat.cu:262-303) on a 1x1 image: u = w*xp + b is chosen directly.
    QP32 C1 params blu=10354 mul=6431 shift=19: rbias = (1<<18)//6431 = 40."""
    blu, mul, sh = formats.SHIPPED_QPARAMS[32][0]
    rb = (1 << (sh - 1)) // mul
    assert rb == 40

    def a1_for_u(u):
        m = synth.make_model(1, 32)
        for w in m.w: w[...] = 0
        for b in m.b: b[...] = 0
        m.b[0][0] = u
        x = np.full((1, 1), 128, np.uint8)                 # xp = 0 -> u = bias exactly
        return int(_om(m).forward_taps(x)[1][0, 0, 0])
    assert a1_for_u(-1) == 0 and a1_for_u(0) == 0                      # u<0 -> 0 ; BLU(0)=0
    assert a1_for_u(blu) == ((blu + rb) * mul) >> sh == 127            # BLU(blu)=127
    assert a1_for_u(blu + 1) == 127                                    # strict >, saturates
    assert a1_for_u(5000) == ((5000 + rb) * mul) >> sh == 61
    for u in (1, 81, 82, 163, 4999, 10353):
        assert a1_for_u(u) == ((u + rb) * mul) >> sh


def test_output_rounding_known_answers():
    """applyRes_y (inference/cnn.cu:507-523): res = (u4*mul + 2^(sh-1)) >> sh, floor shift ->
    round-half-up, also for negatives; then clamp(x + res, 0, 255)."""
    _, mul, sh = formats.SHIPPED_QPARAMS[37][5]           # 7 / 2^13
    m = synth.make_model(1, 37)
    for w in m.w: w[...] = 0
    for b in m.b: b[...] = 0
    for u4, x in ((0, 100), (585, 100), (586, 100), (-585, 100), (-586, 100), (-587, 100), (400000, 250), (-400000, 3)):
        m.b[5][0] = u4
        rec = _om(m).forward_blu(np.full((1, 1, 1), x, np.uint8))[0, 0, 0]
        res = (u4 * mul + (1 << (sh - 1))) >> sh
        assert rec == min(255, max(0, x + res)), (u4, x)
    assert (585 * 7 + 4096) >> 13 == 0 and (586 * 7 + 4096) >> 13 == 1          # .4999 / .5007
    assert (-585 * 7 + 4096) >> 13 == 0 and (-586 * 7 + 4096) >> 13 == -1       # floor shift on negatives


def test_zero_padding_is_per_layer(models):
    """Each layer zero-pads ITS OWN input (inference/cnn.cu:44-49): cropping the input and running
    the net is NOT the same as running the net and cropping, within 6 px of the crop edge, but is
    identical further inside (receptive-field radius 2+2+1+1 = 6)."""
    m = models[27]
    anchor, _ = synth.make_frames(5, 1, 40, 56)
    om = _om(m)
    full = om.forward_blu(anchor)[0]
    crop = om.forward_blu(anchor[:, 4:36, 8:48])[0]
    assert np.array_equal(crop[6:-6, 6:-6], full[4:36, 8:48][6:-6, 6:-6])
    assert not np.array_equal(crop, full[4:36, 8:48])


def test_frames_are_independent(models):
    m = models[22]
    anchor, _ = synth.make_frames(9, 3, 24, 40)
    om = _om(m)
    batch = om.forward_blu(anchor)
    for f in range(3):
        assert np.array_equal(batch[f], om.forward_blu(anchor[f:f + 1])[0])


def test_fp32_materialisation_is_exact_inside_envelope(models):
    """SURVEY fact 7: with 128*sum|w|+|b| < 2^24 the reference's fp32 `u` equals integer arithmetic."""
    for qp, m in models.items():
        for w, b in zip(m.w, m.b):
            bound = 128 * np.abs(w.astype(np.int64)).reshape(w.shape[0], -1).sum(1) + np.abs(b.astype(np.int64))
            assert bound.max() < 1 << 24


def test_golden_checksums(models):
    """Committed sha256 of the oracle's recon for config 1 (QP37 416x240) and a small frame per QP:
    any drift of the oracle itself shows up here."""
    path = os.path.join(GOLDEN, "oracle_checksums.json")
    want = json.load(open(path))
    got = {}
    anchor, _ = synth.make_frames(0xC0FFEE, 1, 240, 416)
    got["qp37_416x240"] = hashlib.sha256(_om(models[37]).forward_blu(anchor).tobytes()).hexdigest()
    small, _ = synth.make_frames(0xC0FFEE + 1, 2, 32, 48)
    for qp in (22, 27, 32, 37):
        got["qp%d_2x32x48" % qp] = hashlib.sha256(_om(models[qp]).forward_blu(small).tobytes()).hexdigest()
    assert got == want


def test_psnr_matches_reference_formula():
    anchor, ori = synth.make_frames(11, 2, 16, 32)
    p, sse = oracle.psnr(anchor, ori)
    d = anchor.astype(np.int64) - ori
    assert sse == int((d * d).sum())
    assert p == 10 * np.log10(65025.0 / (sse / anchor.size))


@pytest.mark.parametrize("mid,seed,family,variant", synth.edge_models(), ids=[e[0] for e in synth.edge_models()])
def test_c_oracle_equals_numpy_restatement_on_edge_models(mid, seed, family, variant):
    """The same cross-check on the corners of the envelope (synth.make_edge_model): -128 taps, channels at exactly
    128*sum|w| + |b| = 2^24 - 1, rows of every shift, requantiser rows that wrap, C4 rows whose product wraps int32 and
    whose residual wraps as a short.  Each model is also shown to exercise what its family names."""
    from oracle import edge_claims
    m = synth.make_edge_model(seed, family, variant)
    x = synth.make_uniform_frames(0xED6E + seed, 1, 48, 80)[0]
    taps = _om(m).forward_taps(x)
    ref = oracle_np.forward_frame(m, x)
    for name, got in zip(("rec", "a1", "a2", "a3", "u4"), taps):
        assert np.array_equal(got, ref[name]), name
    edge_claims.check_claims(m, seed, family, variant, x, taps)
