"""Parity on the corners of the admissible model space (synth.make_edge_model): -128 taps, channels at exactly
128*sum|w| + |b| = 2^24 - 1, hidden requantiser rows of every shift that pass or fail the fast path's precondition, C4 rows
whose product wraps int32 and whose residual wraps as a short -- through every entry point, bit for bit against the C oracle.
The generic families are what launch the generic-requantiser builds of the row-window and SSE kernels.  Also the boundaries
of what qv_load_static_para accepts, the SSE height limit of the fused path, and a check that the matrix launches all nine
non-profiling instantiations of the fused kernels."""
import re

import numpy as np
import pytest

from oracle import edge_claims, oracle
from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, shard, synth

pytestmark = pytest.mark.gpu

EDGE = synth.edge_models()
EDGE_IDS = [e[0] for e in EDGE]
# (frames, H, W, batch of the handle): a single pixel, tiny, ragged around the 120-pixel strip columns, more frames than
# the handle's batch
GEOMS = [(1, 1, 1, 1), (2, 7, 5, 2), (1, 33, 131, 1), (3, 61, 250, 2)]
TMA_GEOM = (2, 20, 160, 2)          # width a multiple of 16 and >= 144: the TMA input ring applies
ENVELOPE = (1 << 24) - 1


def _np_sse(x, ori):
    return ((x.astype(np.int64) - ori.astype(np.int64)) ** 2).reshape(len(ori), -1).sum(axis=1)


def _net(image, batch, h, w, impl):
    net = api.QVRCNN(0, batch, 1, h, w)
    net.load_static_para_mem(image)
    net.set_impl(impl)
    return net


def _sse_run(net, anchor, ori):
    import torch
    d_in, d_ori = torch.from_numpy(anchor).cuda(), torch.from_numpy(ori).cuda()
    d_out = torch.empty_like(d_in)
    d_sse = torch.zeros((len(anchor), 2), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    net.forward_frames_device_sse(d_in.data_ptr(), d_ori.data_ptr(), d_out.data_ptr(), len(anchor), d_sse.data_ptr())
    return d_out.cpu().numpy(), d_sse.cpu().numpy()


def _strips(image, anchor, ori, h, w, S):
    """S strips of one frame on device 0, driven on one stream in the stream-ordered layout (all loads of a frame before its
    forwards); strip_forward for every frame, then strip_forward_sse for every frame.  Returns (frames, frames, sse [K,2])."""
    import torch
    K = len(anchor)
    bounds = [shard.split(h, i, S)[0] for i in range(S)] + [h]
    nets = []
    for i in range(S):
        n = api.QVRCNN(0, 1, 1, bounds[i + 1] - bounds[i], w)
        n.load_static_para_mem(image)
        n.strip_setup(h, bounds[i], bounds[i + 1])
        nets.append(n)
    descs = [n.strip_export() for n in nets]
    for i, n in enumerate(nets):
        if i > 0:
            n.strip_attach(api.STRIP_ABOVE, descs[i - 1])
        if i + 1 < S:
            n.strip_attach(api.STRIP_BELOW, descs[i + 1])
    st = torch.cuda.Stream()
    sse = [torch.zeros((K, 2), dtype=torch.int64, device="cuda") for _ in range(S)]
    outs, keep = {}, []
    torch.cuda.synchronize()
    for step in range(2 * K):
        k, with_sse = step % K, step >= K
        for i, n in enumerate(nets):
            n.strip_load(step & 1, anchor[k, bounds[i]:bounds[i + 1]], st.cuda_stream)
        for i, n in enumerate(nets):
            with torch.cuda.stream(st):
                o = torch.empty((bounds[i + 1] - bounds[i], w), dtype=torch.uint8, device="cuda")
                r = torch.from_numpy(np.ascontiguousarray(ori[k, bounds[i]:bounds[i + 1]])).to("cuda")
            keep.append(r)
            if with_sse:
                n.strip_forward_sse(step & 1, r.data_ptr(), o.data_ptr(), sse[i][k].data_ptr(), st.cuda_stream)
            else:
                n.strip_forward(step & 1, o.data_ptr(), st.cuda_stream)
            outs[(step, i)] = o
    for n in nets:
        n.synchronize(st.cuda_stream)
    got = [np.stack([np.concatenate([outs[(s, i)].cpu().numpy() for i in range(S)]) for s in range(K * j, K * (j + 1))])
           for j in (0, 1)]
    total = sum(s.cpu().numpy() for s in sse)
    for n in nets:
        n.strip_release()
    return got[0], got[1], total


@pytest.mark.parametrize("mid,seed,family,variant", EDGE, ids=EDGE_IDS)
def test_edge_model_on_every_entry_point(mid, seed, family, variant, monkeypatch):
    import torch
    m = synth.make_edge_model(seed, family, variant)
    image = formats.write_model_vect_c(m)
    om = oracle.OracleModel(image)
    fast = edge_claims.check_rows(m, seed, family, variant)
    rng = np.random.default_rng(seed * 100 + len(mid))
    for gi, (n, h, w, batch) in enumerate(GEOMS):
        x = synth.make_uniform_frames(0xED6E + 10 * seed + gi, n, h, w)
        ori = synth.make_uniform_frames(0x0415 + 10 * seed + gi, n, h, w)
        want = om.forward_blu(x)
        where = "%s %dx%dx%d" % (mid, n, h, w)
        if h * w >= 4096:
            edge_claims.check_claims(m, seed, family, variant, x[0], om.forward_taps(x[0]))
        for impl in (api.IMPL_LAYERED, api.IMPL_FUSED):
            net = _net(image, batch, h, w, impl)
            net.load_data(x[:batch])
            net.forward_blu()
            assert np.array_equal(net.get_recon(), want[:batch]), (where, impl, "forward_blu")
            assert np.array_equal(net.forward_frames_host(x), want), (where, impl, "forward_frames_host")
            out, sse = _sse_run(net, x, ori)
            assert np.array_equal(out, want), (where, impl, "forward_frames_device_sse")
            assert np.array_equal(sse[:, 0], _np_sse(x, ori)) and np.array_equal(sse[:, 1], _np_sse(want, ori)), (where, impl)
            # a random output window of frame 0 with the rows it needs
            y0 = int(rng.integers(0, h)); y1 = int(rng.integers(y0 + 1, h + 1))
            r0, r1 = max(0, y0 - 6), min(h, y1 + 6)
            d_in = torch.from_numpy(np.ascontiguousarray(x[0, r0:r1])).cuda()
            d_out = torch.zeros((y1 - y0, w), dtype=torch.uint8, device="cuda")
            net.forward_rows_device(d_in.data_ptr(), h, r0, r1 - r0, d_out.data_ptr(), y0, y1)
            assert np.array_equal(d_out.cpu().numpy(), want[0, y0:y1]), (where, impl, "forward_rows_device", y0, y1)
            net.close()
        if h >= 18:
            S = 3 if h >= 40 else 2
            plain, with_sse, total = _strips(image, x, ori, h, w, S)
            assert np.array_equal(plain, want) and np.array_equal(with_sse, want), (where, "strips", S)
            assert np.array_equal(total, np.stack([_np_sse(x, ori), _np_sse(want, ori)], axis=1)), (where, "strip sse")
    if fast:
        n, h, w, batch = TMA_GEOM
        x = synth.make_uniform_frames(0x7A + seed, n, h, w)
        monkeypatch.setenv("QV_FUSED_TMA", "1")             # read when the model is uploaded
        net = _net(image, batch, h, w, api.IMPL_FUSED)
        assert np.array_equal(net.forward_frames_host(x), om.forward_blu(x)), (mid, "TMA input ring")
        net.close()


# ---- the envelope and the quant-row bounds -------------------------------------------------------------------------------
def _small_check(model, h=24, w=40):
    image = formats.write_model_vect_c(model)
    x = synth.make_uniform_frames(0xB0B, 2, h, w)
    want = oracle.OracleModel(image).forward_blu(x)
    for impl in (api.IMPL_LAYERED, api.IMPL_FUSED):
        net = _net(image, 2, h, w, impl)
        assert np.array_equal(net.forward_frames_host(x), want), impl
        net.close()


@pytest.mark.parametrize("layer", range(6), ids=formats.LAYER_NAMES)
def test_envelope_boundary_per_layer(models, layer):
    """One output channel at exactly 128*sum|w| + |b| = 2^24 - 1 loads and runs bit-exact on both implementations; one unit
    more is refused with QV_ERR_RANGE, by load_static_para_mem and by set_weights."""
    import copy
    m = copy.deepcopy(models[32])
    ch = 3 if layer < 5 else 0
    s = int(np.abs(m.w[layer][ch].astype(np.int64)).sum())
    sign = -1 if layer % 2 else 1
    m.b[layer][ch] = sign * (ENVELOPE - 128 * s)
    _small_check(m)
    bad = copy.deepcopy(m)
    bad.b[layer][ch] = sign * (ENVELOPE - 128 * s + 1)
    net = api.QVRCNN(0, 1, 1, 16, 16)
    with pytest.raises(api.QVError) as e:
        net.load_static_para_mem(formats.write_model_vect_c(bad))
    assert e.value.code == -4
    net.load_static_para_mem(formats.write_model_vect_c(m))
    with pytest.raises(api.QVError) as e:
        net.set_weights(layer, bad.w[layer], bad.b[layer])
    assert e.value.code == -4


@pytest.mark.parametrize("case", ["blu_2^24-1", "shift_30", "blu_2^24", "shift_31", "mul_0"])
def test_quant_row_bounds(models, case):
    """validate_qparams: blu up to 2^24 - 1 and shift up to 30 are accepted and bit-exact; blu = 2^24, shift = 31 and mul = 0
    are refused with QV_ERR_RANGE."""
    import copy
    m = copy.deepcopy(models[27])
    q = [list(t) for t in m.qparams]
    l = 3
    q[l] = {"blu_2^24-1": [ENVELOPE, 1, 17], "shift_30": [q[l][0], 1 << 16, 30], "blu_2^24": [1 << 24, 1, 17],
            "shift_31": [q[l][0], 1 << 16, 31], "mul_0": [q[l][0], 0, 14]}[case]
    m.qparams = [tuple(t) for t in q]
    if case in ("blu_2^24-1", "shift_30"):
        _small_check(m)
        return
    net = api.QVRCNN(0, 1, 1, 16, 16)
    with pytest.raises(api.QVError) as e:
        net.load_static_para_mem(formats.write_model_vect_c(m))
    assert e.value.code == -4


# ---- the SSE height limit -------------------------------------------------------------------------------------------------
def test_sse_height_boundary(models):
    """The fused kernel's SSE form keeps a 32-bit sum per output column and thread; 255^2 * H < 2^32 holds up to H = 66051,
    and taller frames are refused (QV_ERR_ARG) on the fused path.  The row plan also cuts a tall column into segments, so
    at the limit no single sum comes near 2^31 either.  At 66051 rows (anchor 0, original 255: the largest error everywhere)
    the fused SSEs equal numpy and the frame equals the layered path's; at 66052 the fused SSE call is refused while the
    plain fused forward still runs, and the layered path, whose SSE pass sums in 64 bits, takes the frame and equals numpy."""
    import torch
    image = formats.write_model_vect_c(models[32])
    w = 8
    for h in (66051, 66052):
        x = np.zeros((1, h, w), np.uint8)
        ori = np.full((1, h, w), 255, np.uint8)
        lay = _net(image, 1, h, w, api.IMPL_LAYERED)
        lout, lsse = _sse_run(lay, x, ori)
        assert np.array_equal(lsse[:, 0], _np_sse(x, ori)) and np.array_equal(lsse[:, 1], _np_sse(lout, ori)), h
        lay.close()
        fus = _net(image, 1, h, w, api.IMPL_FUSED)
        if h == 66051:
            out, sse = _sse_run(fus, x, ori)
            assert int(sse[0, 0]) == 255 * 255 * h * w
            assert np.array_equal(out, lout) and np.array_equal(sse, lsse)
        else:
            with pytest.raises(api.QVError) as e:
                _sse_run(fus, x, ori)
            assert e.value.code == -1
            d_in = torch.from_numpy(x).cuda()
            d_out = torch.empty_like(d_in)
            fus.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), 1)
            assert np.array_equal(d_out.cpu().numpy(), lout)
        fus.close()


# ---- launch coverage --------------------------------------------------------------------------------------------------------
_FUSED_BUILDS = {("k_fused", a) for a in [(1, 0, 0, 0), (0, 0, 0, 0), (1, 0, 1, 0), (0, 0, 1, 0), (1, 0, 0, 1)]} | \
                {("k_enh_sse", a) for a in [(1, 0), (0, 0), (1, 1), (0, 1)]}


def _builds(name):
    """('k_fused', (FAST, PROF, ROWS, TMA)) or ('k_enh_sse', (FAST, ROWS)) from a demangled or mangled kernel name."""
    for k in ("k_fused", "k_enh_sse"):
        m = re.search(k + r"<([^>]*)>", name)
        if m:
            args = tuple(int(a.strip() == "true") for a in m.group(1).split(","))
        else:
            m = re.search(k + r"I((?:Lb[01]E)+)E", name)
            if not m:
                continue
            args = tuple(int(b) for b in re.findall(r"Lb([01])E", m.group(1)))
        return k, args + (0,) * (4 - len(args)) if k == "k_fused" else args
    return None


def test_every_fused_instantiation_is_launched(monkeypatch):
    """One fast and one generic edge model through whole frames, a row window, the TMA input ring, the SSE form and a strip's
    SSE form: the profiler sees all nine non-profiling instantiations of the fused kernels launched."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    monkeypatch.setenv("QV_FUSED_TMA", "1")
    n, h, w, batch = TMA_GEOM
    x = synth.make_uniform_frames(0xC0DE, n, h, w)
    ori = synth.make_uniform_frames(0xC0DF, n, h, w)
    seen = set()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for mid in ("full_scale-fast", "full_scale-generic"):
            _, seed, family, variant = EDGE[EDGE_IDS.index(mid)]
            image = formats.write_model_vect_c(synth.make_edge_model(seed, family, variant))
            want = oracle.OracleModel(image).forward_blu(x)
            net = _net(image, batch, h, w, api.IMPL_FUSED)
            assert np.array_equal(net.forward_frames_host(x), want), mid          # TMA build when the model is fast
            monkeypatch.setenv("QV_FUSED_TMA", "0")
            net.load_static_para_mem(image)
            assert np.array_equal(net.forward_frames_host(x), want), mid          # whole-frame build
            monkeypatch.setenv("QV_FUSED_TMA", "1")
            out, _ = _sse_run(net, x, ori)
            assert np.array_equal(out, want), mid
            d_in = torch.from_numpy(np.ascontiguousarray(x[0])).cuda()
            d_out = torch.zeros((h, w), dtype=torch.uint8, device="cuda")
            net.forward_rows_device(d_in.data_ptr(), h, 0, h, d_out.data_ptr(), 0, h)
            assert np.array_equal(d_out.cpu().numpy(), want[0]), mid
            plain, with_sse, _ = _strips(image, x, ori, h, w, 2)
            assert np.array_equal(plain, want) and np.array_equal(with_sse, want), mid
            net.close()
        torch.cuda.synchronize()
    for e in prof.events():
        b = _builds(e.name)
        if b:
            seen.add(b)
    print("fused instantiations launched:", sorted(seen))
    assert _FUSED_BUILDS <= seen, sorted(_FUSED_BUILDS - seen)
