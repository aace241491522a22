"""Parity tests proper: the CUDA path through the C ABI vs the CPU oracle, bit for bit.
Run on the B200 box:  python -m pytest tests -m gpu -x -q"""
import hashlib
import json
import os

import numpy as np
import pytest

from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, synth

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
IMPLS = [api.IMPL_LAYERED, api.IMPL_FUSED]
IMPL_NAME = {api.IMPL_LAYERED: "layered", api.IMPL_FUSED: "fused"}


def _oracle(model):
    from oracle import oracle
    return oracle.OracleModel(formats.write_model_vect_c(model))


def _net(model, batch, h, w, impl, tmp_path=None):
    net = api.QVRCNN(0, batch, 1, h, w)
    net.load_static_para_mem(formats.write_model_vect_c(model))
    net.set_impl(impl)
    return net


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
@pytest.mark.parametrize("qp", [22, 27, 32, 37])
def test_config1_416x240_bit_exact(models, qp, impl, tmp_path):
    """BASELINE config 1 geometry (one 416x240 frame) for all four QP parameter sets, through the
    reference's own call sequence: load_static_para(file) -> load_data -> forward_blu -> x_rec."""
    m = models[qp]
    anchor, ori = synth.make_frames(0xC0FFEE, 1, 240, 416)
    path = tmp_path / ("qvrcnn_nchw_vect_c_8bit_qfp_%d.data" % qp)
    path.write_bytes(formats.write_model_vect_c(m))
    net = api.QVRCNN(0, 1, 1, 240, 416)
    net.load_static_para(str(path))
    net.set_impl(impl)
    net.load_data(anchor)
    net.forward_blu()
    rec = net.get_recon()
    want = _oracle(m).forward_blu(anchor)
    assert np.array_equal(rec, want), "mismatching pixels: %d" % int((rec != want).sum())
    assert (rec != anchor).any()
    if qp == 37:
        gold = json.load(open(os.path.join(GOLDEN, "oracle_checksums.json")))["qp37_416x240"]
        assert hashlib.sha256(rec.tobytes()).hexdigest() == gold
    # identical frames => identical PSNR report
    d = api.VRCNNData(1, 240, 416)
    d.ori[:] = ori
    from oracle import oracle
    assert d.psnr(rec) == oracle.psnr(want, ori)[0]


@pytest.mark.parametrize("qp", [22, 27, 32, 37])
def test_layered_activations_match_oracle(models, qp):
    """Per-layer parity: a1 / a2 / a3 (C1.v, Conc1.conc, Conc2.conc) vs the oracle's taps."""
    m = models[qp]
    anchor, _ = synth.make_frames(0xC0FFEE + 2, 1, 72, 104)
    net = _net(m, 1, 72, 104, api.IMPL_LAYERED)
    net.load_data(anchor)
    net.forward_blu()
    rec, a1, a2, a3, _ = _oracle(m).forward_taps(anchor[0])
    assert np.array_equal(net.get_activation(1), a1)
    assert np.array_equal(net.get_activation(2), a2)
    assert np.array_equal(net.get_activation(3), a3)
    assert np.array_equal(net.get_recon()[0], rec)


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
@pytest.mark.parametrize("shape", [(1, 1), (1, 9), (7, 5), (13, 13), (33, 31), (8, 257), (130, 20), (61, 123)])
def test_ragged_and_tiny_frames(models, impl, shape):
    """Frames smaller than one tile / not multiples of any tile size / thinner than the halo."""
    m = models[32]
    h, w = shape
    x = synth.make_uniform_frames(17, 2, h, w)
    net = _net(m, 2, h, w, api.IMPL_LAYERED)
    net.set_impl(impl)
    net.load_data(x)
    net.forward_blu()
    assert np.array_equal(net.get_recon(), _oracle(m).forward_blu(x))


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
@pytest.mark.parametrize("value", [0, 128, 255])
def test_constant_frames(models, impl, value):
    m = models[27]
    x = np.full((1, 40, 72), value, np.uint8)
    net = _net(m, 1, 40, 72, api.IMPL_LAYERED)
    net.set_impl(impl)
    net.load_data(x)
    net.forward_blu()
    assert np.array_equal(net.get_recon(), _oracle(m).forward_blu(x))


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
def test_config2_8x832x480_all_qps(models, impl):
    """BASELINE config 2: 8-frame 832x480 sequence, all four QP sets; oracle on frames 0 and 7,
    the other frames through frame-independence (batch result == per-frame result)."""
    anchor, _ = synth.make_frames(0xC0FFEE + 3, 8, 480, 832)
    for qp in (22, 27, 32, 37):
        m = models[qp]
        net = _net(m, 8, 480, 832, api.IMPL_LAYERED)
        net.set_impl(impl)
        out = net.forward_frames_host(anchor)
        om = _oracle(m)
        assert np.array_equal(out[0], om.forward_blu(anchor[0:1])[0])
        assert np.array_equal(out[7], om.forward_blu(anchor[7:8])[0])
        one = _net(m, 1, 480, 832, impl)
        for f in (3, 5):
            one.load_data(anchor[f])
            one.forward_blu()
            assert np.array_equal(one.get_recon()[0], out[f])
        net.close(); one.close()


def test_fused_equals_layered_1080p(models):
    """Full-size property check (BASELINE config 3 geometry, 6 of the 64 frames): two independently
    written CUDA implementations agree bit for bit, and frame 0 also matches the oracle."""
    m = models[32]
    anchor, _ = synth.make_frames(0xC0FFEE + 4, 6, 1080, 1920)
    a = _net(m, 6, 1080, 1920, api.IMPL_LAYERED)
    out_l = a.forward_frames_host(anchor)
    a.set_impl(api.IMPL_FUSED)
    out_f = a.forward_frames_host(anchor)
    assert np.array_equal(out_l, out_f)
    assert np.array_equal(out_f[0], _oracle(m).forward_blu(anchor[0:1])[0])


def test_config3_all_64_distinct_frames(models):
    """BASELINE config 3 at full size with 64 DISTINCT frames (the bench tiles 8): the two independently written CUDA
    implementations agree on every one of them, the oracle pins three, and every frame differs from its input."""
    m = models[32]
    anchor, _ = synth.make_frames(0xC0FFEE + 40, 64, 1080, 1920)
    net = _net(m, 8, 1080, 1920, api.IMPL_LAYERED)
    out_l = net.forward_frames_host(anchor)
    net.set_impl(api.IMPL_FUSED)
    out_f = net.forward_frames_host(anchor)
    assert np.array_equal(out_l, out_f)
    pick = [0, 37, 63]
    assert np.array_equal(out_f[pick], _oracle(m).forward_blu(anchor[pick]))
    assert all((out_f[i] != anchor[i]).any() for i in range(64))
    assert len({hashlib.sha256(out_f[i].tobytes()).hexdigest() for i in range(64)}) == 64


def test_hwcn_model_file_loads_to_the_same_network(models, tmp_path):
    """qv_load_static_para_hwcn (the TF-side HWCN dump, input of model_qfp_HWCN2NCHW_VECT_C, inference/qvrcnn.cu:535-585)
    gives the same network as the converted NCHW_VECT_C file: on the reference's own converter golden and on a fresh model,
    both CUDA paths."""
    g = np.load(os.path.join(GOLDEN, "ref_converter_qp32.npz"))
    fin = tmp_path / "hwcn.data"
    fin.write_bytes(g["hwcn"].tobytes())
    anchor, _ = synth.make_frames(0xC0FFEE + 41, 2, 90, 200)
    a = api.QVRCNN(0, 2, 1, 90, 200)
    a.load_static_para_hwcn(str(fin))
    b = api.QVRCNN(0, 2, 1, 90, 200)
    b.load_static_para_mem(g["vect_c"].tobytes())               # what the REFERENCE's converter wrote
    want = _oracle(formats.read_model_vect_c(g["vect_c"].tobytes())).forward_blu(anchor)
    for impl in IMPLS:
        a.set_impl(impl); b.set_impl(impl)
        assert np.array_equal(a.forward_frames_host(anchor), want)
        assert np.array_equal(b.forward_frames_host(anchor), want)
    assert a.quant_params().tolist() == b.quant_params().tolist()
    with pytest.raises(api.QVError):
        a.load_static_para_hwcn(str(tmp_path / "missing.data"))
    short = tmp_path / "short.data"
    short.write_bytes(g["hwcn"].tobytes()[:-1])
    with pytest.raises(api.QVError):
        a.load_static_para_hwcn(str(short))


def test_two_threads_load_and_run_two_handles_concurrently(models):
    """include/qvrcnn_b200.h: "distinct handles may be used from distinct threads" -- including the model upload (the
    operand table in constant memory is written once per device under a lock; `qcnn_gpu --gpus N` is this pattern)."""
    import threading
    imgs = {qp: formats.write_model_vect_c(models[qp]) for qp in (22, 37)}
    frames = {22: synth.make_frames(0xC0FFEE + 42, 3, 120, 250)[0], 37: synth.make_frames(0xC0FFEE + 43, 3, 120, 250)[0]}
    got, errs = {}, []
    gate = threading.Barrier(2)

    def work(qp):
        try:
            for rep in range(3):
                gate.wait(timeout=60)
                net = api.QVRCNN(0, 3, 1, 120, 250)
                net.load_static_para_mem(imgs[qp])
                got[(qp, rep)] = net.forward_frames_host(frames[qp])
                net.close()
        except Exception as e:            # noqa: BLE001
            errs.append(repr(e))
    th = [threading.Thread(target=work, args=(qp,)) for qp in (22, 37)]
    [t.start() for t in th]
    [t.join(timeout=300) for t in th]
    assert not errs, errs
    for qp in (22, 37):
        want = _oracle(models[qp]).forward_blu(frames[qp])
        for rep in range(3):
            assert np.array_equal(got[(qp, rep)], want), (qp, rep)


def test_random_geometries_fused_equals_layered_and_oracle(models):
    """Seeded sweep over ragged geometries: 48 random (frames, height, width, QP) -- widths around the 120-pixel strip columns,
    heights around the row-segment cuts -- fused == layered bit for bit, the small ones also == oracle; and for each a random
    row window through qv_forward_rows_device (the row-window instantiation of the fused kernel) == the same rows of the
    whole-frame result."""
    import torch
    rng = np.random.default_rng(20261018)
    net_cache = {}
    for case in range(48):
        qp = int(rng.choice([22, 27, 32, 37]))
        n = int(rng.integers(1, 4))
        h = int(rng.choice([rng.integers(1, 40), rng.integers(40, 300)]))
        w = int(rng.choice([rng.integers(1, 130), 120 * rng.integers(1, 4) + rng.integers(-3, 4), rng.integers(130, 500)]))
        w = max(w, 1)
        x = synth.make_uniform_frames(1000 + case, n, h, w) if case % 3 == 0 else synth.make_frames(2000 + case, n, h, w)[0]
        net = api.QVRCNN(0, n, 1, h, w)
        net.load_static_para_mem(formats.write_model_vect_c(models[qp]))
        net.set_impl(api.IMPL_LAYERED)
        out_l = net.forward_frames_host(x)
        net.set_impl(api.IMPL_FUSED)
        out_f = net.forward_frames_host(x)
        assert np.array_equal(out_l, out_f), (case, qp, n, h, w, int((out_l != out_f).sum()))
        if n * h * w <= 40000:
            assert np.array_equal(out_f, _oracle(models[qp]).forward_blu(x)), (case, qp, n, h, w)
        # a random output window [y0, y1) with the rows it needs
        y0 = int(rng.integers(0, h)); y1 = int(rng.integers(y0 + 1, h + 1))
        r0, r1 = max(0, y0 - 6), min(h, y1 + 6)
        d_in = torch.from_numpy(np.ascontiguousarray(x[0, r0:r1])).cuda()
        d_out = torch.zeros((y1 - y0, w), dtype=torch.uint8, device="cuda")
        net.forward_rows_device(d_in.data_ptr(), h, r0, r1 - r0, d_out.data_ptr(), y0, y1)
        assert np.array_equal(d_out.cpu().numpy(), out_f[0, y0:y1]), (case, "window", h, w, y0, y1)
        net.close()


def test_full_size_properties_4k_and_8k(models):
    """BASELINE configs 4 and 5 at their real frame sizes, through properties that need no CPU oracle run:
    (a) 3840x2160, QP 27: frames are independent -- a frame inside a batch of 3 equals the same frame processed alone,
        a permuted batch gives the permuted output, and the two CUDA implementations agree;
    (b) 7680x4320, QP 22: fused == layered on the whole frame, and a 1300x2100 window with a 6-pixel margin reproduces
        the frame's interior (the net is a stencil of radius 6: SURVEY 8e);
    (c) the oracle pins one 64-row band of the 4K frame (rows 1000..1063 with their halo)."""
    m4, m8 = models[27], models[22]
    # (a)
    h, w = 2160, 3840
    anchor, _ = synth.make_frames(0xC0FFEE + 9, 3, h, w)
    net = _net(m4, 3, h, w, api.IMPL_LAYERED)
    out_l = net.forward_frames_host(anchor)
    net.set_impl(api.IMPL_FUSED)
    out_f = net.forward_frames_host(anchor)
    assert np.array_equal(out_l, out_f)
    perm = anchor[[2, 0, 1]]
    assert np.array_equal(net.forward_frames_host(perm), out_f[[2, 0, 1]])
    one = _net(m4, 1, h, w, api.IMPL_FUSED)
    assert np.array_equal(one.forward_frames_host(anchor[1:2])[0], out_f[1])
    # (c) oracle on a band: rows 994..1069 as a frame; its rows 6..69 are exact for the 4K frame's rows 1000..1063
    band = np.ascontiguousarray(anchor[0:1, 994:1070, :])
    want = _oracle(m4).forward_blu(band)[0][6:70]
    assert np.array_equal(out_f[0][1000:1064], want)
    del net, one
    # (b)
    h, w = 4320, 7680
    anchor, _ = synth.make_frames(0xC0FFEE + 10, 1, h, w)
    net = _net(m8, 1, h, w, api.IMPL_LAYERED)
    out_l = net.forward_frames_host(anchor)
    net.set_impl(api.IMPL_FUSED)
    out_f = net.forward_frames_host(anchor)
    assert np.array_equal(out_l, out_f)
    y0, x0, hh, ww = 1501, 2999, 1300, 2100
    win = np.ascontiguousarray(anchor[:, y0:y0 + hh, x0:x0 + ww])
    wnet = _net(m8, 1, hh, ww, api.IMPL_FUSED)
    out_w = wnet.forward_frames_host(win)[0]
    assert np.array_equal(out_w[6:-6, 6:-6], out_f[0][y0 + 6:y0 + hh - 6, x0 + 6:x0 + ww - 6])


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
def test_rows_mode_strips_equal_whole_frame(models, impl):
    """Spatial partition (BASELINE config 5 in miniature): a frame cut into 3 horizontal strips with
    6-row input halos reproduces the whole-frame result bit for bit."""
    import torch
    m = models[22]
    h, w = 150, 200
    anchor, _ = synth.make_frames(0xC0FFEE + 5, 1, h, w)
    net = _net(m, 1, h, w, api.IMPL_LAYERED)
    net.set_impl(impl)
    net.load_data(anchor)
    net.forward_blu()
    whole = net.get_recon()[0]
    d_in = torch.from_numpy(anchor[0]).cuda()
    d_out = torch.zeros_like(d_in)
    bounds = [0, 47, 101, h]
    for i in range(3):
        y0, y1 = bounds[i], bounds[i + 1]
        r0, r1 = max(0, y0 - 6), min(h, y1 + 6)
        net.forward_rows_device(d_in.data_ptr() + r0 * w, h, r0, r1 - r0, d_out.data_ptr() + y0 * w, y0, y1)
    torch.cuda.synchronize()
    assert np.array_equal(d_out.cpu().numpy(), whole)
    with pytest.raises(api.QVError):      # fewer than 6 halo rows on an interior edge is refused
        net.forward_rows_device(d_in.data_ptr() + 45 * w, h, 45, 60, d_out.data_ptr() + 47 * w, 47, 101)


def test_device_entry_and_sse(models):
    """qv_forward_frames_device on torch-owned device memory + on-device exact SSE == host PSNR."""
    import torch
    m = models[37]
    anchor, ori = synth.make_frames(0xC0FFEE + 6, 3, 64, 96)
    net = _net(m, 2, 64, 96, api.IMPL_AUTO)          # n_frames (3) > batch (2): chunked
    d_in = torch.from_numpy(anchor).cuda()
    d_ori = torch.from_numpy(ori).cuda()
    d_out = torch.empty_like(d_in)
    acc = torch.zeros(1, dtype=torch.int64, device="cuda")
    st = api.stream_arg(torch.cuda.current_stream().cuda_stream)     # torch's legacy default stream, named explicitly
    net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), 3, st)
    api.sse_device(d_out.data_ptr(), d_ori.data_ptr(), d_in.numel(), acc.data_ptr(), st)
    torch.cuda.synchronize()
    rec = d_out.cpu().numpy()
    want = _oracle(m).forward_blu(anchor)
    assert np.array_equal(rec, want)
    p, sse = formats.psnr(want, ori)
    assert int(acc.item()) == sse
    assert api.psnr_from_sse(int(acc.item()), rec.size) == pytest.approx(p, abs=1e-12)
    assert net.launch_count() > 0


@pytest.mark.parametrize("entry", ["frames", "frames_sse", "rows"])
def test_layered_calls_on_several_streams_are_ordered(models, entry):
    """A layered handle's calls share its activation scratch, whatever stream they run on: two asynchronous calls with
    different inputs on two streams, then a third on a caller stream directly followed by qv_get_activation (which runs on
    the handle's own stream), with no synchronisation in between -- every output, SSE and activation is the oracle's."""
    import torch
    m = models[27]
    om = _oracle(m)
    h, w = 120, 208
    net = _net(m, 2, h, w, api.IMPL_LAYERED)
    sse = lambda x, ori: ((x.astype(np.int64) - ori) ** 2).reshape(len(x), -1).sum(axis=1)
    calls = []
    for i in range(3):
        if entry == "rows":
            # rows [40, 160) of a 200-row image, run as a window; its rows [46, 154) are exact
            img = synth.make_frames(0xC0FFEE + 50 + i, 1, 200, w)[0]
            d_in = torch.from_numpy(np.ascontiguousarray(img[0, 40:160])).cuda()
            d_out = torch.zeros((108, w), dtype=torch.uint8, device="cuda")
            calls.append(dict(d_in=d_in, d_out=d_out, want=om.forward_blu(img)[0, 46:154], taps=img[0, 40:160]))
        else:
            x, ori = synth.make_frames(0xC0FFEE + 50 + i, 2, h, w)
            want = om.forward_blu(x)
            calls.append(dict(d_in=torch.from_numpy(x).cuda(), d_ori=torch.from_numpy(ori).cuda(),
                              d_out=torch.zeros((2, h, w), dtype=torch.uint8, device="cuda"),
                              d_sse=torch.zeros(4, dtype=torch.int64, device="cuda"), want=want, taps=x[0],
                              sse=np.stack([sse(x, ori), sse(want, ori)], axis=1).reshape(-1)))

    def run(c, stream):
        if entry == "rows":
            net.forward_rows_device(c["d_in"].data_ptr(), 200, 40, 120, c["d_out"].data_ptr(), 46, 154, stream.cuda_stream)
        elif entry == "frames":
            net.forward_frames_device(c["d_in"].data_ptr(), c["d_out"].data_ptr(), 2, stream.cuda_stream)
        else:
            net.forward_frames_device_sse(c["d_in"].data_ptr(), c["d_ori"].data_ptr(), c["d_out"].data_ptr(), 2,
                                          c["d_sse"].data_ptr(), stream.cuda_stream)

    torch.cuda.synchronize()                  # the inputs are on the device before any call
    a, b = torch.cuda.Stream(), torch.cuda.Stream()
    run(calls[0], a)
    run(calls[1], b)
    run(calls[2], a)
    acts = [net.get_activation(k) for k in (1, 2, 3)]
    torch.cuda.synchronize()
    for i, c in enumerate(calls):
        assert np.array_equal(c["d_out"].cpu().numpy(), c["want"]), (entry, i)
        if entry == "frames_sse":
            assert c["d_sse"].cpu().numpy().tolist() == c["sse"].tolist(), i
    _, a1, a2, a3, _ = om.forward_taps(calls[2]["taps"])
    for k, want in enumerate((a1, a2, a3)):
        assert np.array_equal(acts[k], want), (entry, k + 1)
    assert net.launch_count() == 3 * (10 if entry == "frames_sse" else 6)


def test_layered_scratch_errors(models):
    """qv_get_activation before any layered forward, and a row window of more pixels than batch x H x W."""
    import torch
    net = _net(models[27], 1, 40, 64, api.IMPL_LAYERED)
    with pytest.raises(api.QVError) as e:
        net.get_activation(1)
    assert e.value.code == -5
    assert str(e.value) == "qvrcnn_b200 error -5: qv_get_activation: the layered path has not run on this handle"
    d_in = torch.zeros((41, 64), dtype=torch.uint8, device="cuda")
    d_out = torch.zeros_like(d_in)
    with pytest.raises(api.QVError) as e:
        net.forward_rows_device(d_in.data_ptr(), 41, 0, 41, d_out.data_ptr(), 0, 41)
    assert e.value.code == -1
    assert str(e.value) == "qvrcnn_b200 error -1: qv_forward_rows_device: window larger than the handle's geometry"


def test_error_behaviour(models, tmp_path):
    net = api.QVRCNN(0, 1, 1, 16, 16)
    with pytest.raises(api.QVError) as e:           # forward before load
        net.forward_blu()
    assert e.value.code == -5
    with pytest.raises(api.QVError) as e:           # the reference prints "cannot open model file." and exits
        net.load_static_para(str(tmp_path / "missing.data"))
    assert e.value.code == -2 and "cannot open model file" in str(e.value)
    bad = tmp_path / "short.data"
    bad.write_bytes(b"\0" * 100)
    with pytest.raises(api.QVError):
        net.load_static_para(str(bad))
    with pytest.raises(api.QVError):
        api.QVRCNN(0, 1, 3, 16, 16)                  # luma only
    # outside the exact-integer envelope (SURVEY fact 7) -> refused, not silently different
    m = synth.make_model(1, 32)
    m.w[2][...] = 127
    with pytest.raises(api.QVError) as e:
        net.load_static_para_mem(formats.write_model_vect_c(m))
    assert e.value.code == -4


def test_kernel_failure_is_reported(models, monkeypatch):
    """A CTA of the fused kernel that detects a problem (here: forced, the operand-table check) must surface as an
    error code of the call that synchronises -- never as a silently wrong frame.  (The switch is read when the model
    is uploaded, not on the launch path.)"""
    image = formats.write_model_vect_c(models[32])
    net = _net(models[32], 1, 64, 250, api.IMPL_LAYERED)
    net.set_impl(api.IMPL_FUSED)
    x = np.full((1, 64, 250), 77, np.uint8)
    net.load_data(x)
    monkeypatch.setenv("QV_FUSED_TEST_FAIL", "1")
    net.load_static_para_mem(image)
    with pytest.raises(api.QVError, match="operand table"):
        net.forward_blu()
    # the asynchronous entry point cannot report it; qv_synchronize on the caller's stream does
    import torch
    d_in = torch.from_numpy(x).cuda()
    d_out = torch.empty_like(d_in)
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), 1, st.cuda_stream)
    with pytest.raises(api.QVError, match="operand table"):
        net.synchronize(st.cuda_stream)
    monkeypatch.delenv("QV_FUSED_TEST_FAIL")
    net.load_static_para_mem(image)
    net.forward_blu()                                   # the report was consumed; the handle keeps working
    assert np.array_equal(net.get_recon(), _oracle(models[32]).forward_blu(x))


@pytest.mark.parametrize("shape", [(3, 40, 416), (2, 33, 144), (1, 70, 1920), (2, 21, 250)])
def test_tma_input_ring_is_bit_identical(models, monkeypatch, shape):
    """QV_FUSED_TMA=1 (read when the model is uploaded): the input ring filled by cp.async.bulk.tensor.2d -- boxes that start
    16-byte aligned, out-of-image columns patched to 128, out-of-image rows filled by hand -- gives the same frames; a width
    that is not a multiple of 16 cannot be described by a tensor map and silently takes the plain ring."""
    n, h, w = shape
    image = formats.write_model_vect_c(models[27])
    x, _ = synth.make_frames(0xC0FFEE + 44, n, h, w)
    a = api.QVRCNN(0, n, 1, h, w)
    a.load_static_para_mem(image)
    a.set_impl(api.IMPL_FUSED)
    want = a.forward_frames_host(x)
    monkeypatch.setenv("QV_FUSED_TMA", "1")
    b = api.QVRCNN(0, n, 1, h, w)
    b.load_static_para_mem(image)
    b.set_impl(api.IMPL_FUSED)
    assert np.array_equal(b.forward_frames_host(x), want)
    assert np.array_equal(want[:1], _oracle(models[27]).forward_blu(x[:1]))


def test_quant_param_file_plus_set_weights(models, tmp_path):
    """The shipped artefact is the per-QP scale file; weights come separately (SURVEY fact 6)."""
    m = models[27]
    q = tmp_path / "quant_params27.data"
    formats.write_quant_params_pickle(str(q), formats.qparams_rows_from_table(27))
    anchor, _ = synth.make_frames(3, 1, 32, 48)
    net = api.QVRCNN(0, 1, 1, 32, 48)
    net.load_quant_params(str(q))
    for l in range(6):
        net.set_weights(l, m.w[l], m.b[l])
    assert net.quant_params().tolist() == [list(t) for t in formats.SHIPPED_QPARAMS[27]]
    net.load_data(anchor)
    net.forward_blu()
    assert np.array_equal(net.get_recon(), _oracle(m).forward_blu(anchor))


@pytest.mark.parametrize("impl", IMPLS, ids=lambda i: IMPL_NAME[i])
@pytest.mark.parametrize("case", ["not_127_at_blu", "wraps_to_negative", "big_shift"])
def test_generic_requant_parameters(models, impl, case):
    """Quant params for which BLU(blu) != 127 (the fast epilogue's precondition fails): the kernels must fall
    back to the reference's literal formula, including the (char) wrap of results above 127
    (inference/mat.cu:291 stores into xwtype=char), which makes hidden activations negative."""
    import copy
    m = copy.deepcopy(models[32])
    q = [list(t) for t in m.qparams]
    if case == "not_127_at_blu":
        q[0] = [5000, 100, 12]            # (5000+20)*100 >> 12 = 122
        q[3] = [7000, 281, 14]            # 120
    elif case == "wraps_to_negative":
        q[1] = [8000, 100, 12]            # 195 -> (char) -61
        q[2] = [9000, 99, 12]             # 217 -> (char) -39
    else:
        q[4] = [4526, 115 << 14, 26]      # shift > 24: outside the fast path's packing trick, same scale
    m.qparams = [tuple(t) for t in q]
    anchor, _ = synth.make_frames(0xC0FFEE + 9, 2, 70, 131)
    net = _net(m, 2, 70, 131, api.IMPL_LAYERED)
    net.set_impl(impl)
    net.load_data(anchor)
    net.forward_blu()
    want = _oracle(m).forward_blu(anchor)
    assert np.array_equal(net.get_recon(), want)
    if case == "wraps_to_negative":
        a2 = _oracle(m).forward_taps(anchor[0])[2]
        assert (a2 < 0).any()             # the case really exercises signed hidden activations
