"""Streaming a YUV sequence through the strip partition (qv_strip_stream_yuv_pf, `qcnn_gpu --strips S --stream`): every strip
handle reads its own rows of each frame from the anchor / original files and writes its own rows of the reconstruction.
Checked against the frame-sharded stream (qv_stream_yuv_pf on a whole-frame handle), numpy's SSEs and the C oracle; a frame
range in the middle of a file, strips split over calls, every refused argument, a reconstruction file that cannot be
written, the CLI against its in-memory and frame-sharded modes, and host memory that does not grow with the sequence."""
import ctypes as C
import os
import re
import subprocess
import sys
import threading

import numpy as np
import pytest

from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, shard, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "qcnn_gpu_b200", "qcnn_gpu")
FRAMES = 7                     # > 2 input slots and > 3 ring entries: both are reused


def _ndev():
    import torch
    return torch.cuda.device_count()


def _np_sse(x, ori):
    return ((x.astype(np.int64) - ori.astype(np.int64)) ** 2).reshape(len(ori), -1).sum(axis=1)


def _write_yuv(path, luma, seed):
    """luma [n, h, w] plus random NON-zero chroma bytes, so that reading or writing the wrong plane shows"""
    n, h, w = luma.shape
    chroma = np.random.default_rng(seed).integers(1, 256, size=(n, h * w // 2), dtype=np.uint8)
    np.concatenate([luma.reshape(n, h * w), chroma], axis=1).tofile(str(path))


def _luma(path, n, h, w):
    raw = np.fromfile(str(path), np.uint8).reshape(n, h * w * 3 // 2)
    return raw[:, :h * w].reshape(n, h, w), raw[:, h * w:]


def _bounds(h, S):
    return [shard.split(h, i, S)[0] for i in range(S)] + [h]


@pytest.fixture
def handles():
    """Creates handles and destroys them after the test, so that a failed test leaves no strip registered on a device."""
    made = []

    def make(dev, rows, w, image, batch=1):
        n = api.QVRCNN(dev, batch, 1, rows, w)
        n.load_static_para_mem(image)
        made.append(n)
        return n
    yield make
    for n in made:
        n.close()


def _strips(make, image, h, w, bounds, devices):
    nets = [make(devices[i], bounds[i + 1] - bounds[i], w, image) for i in range(len(bounds) - 1)]
    for i, n in enumerate(nets):
        n.strip_setup(h, bounds[i], bounds[i + 1])
    descs = [n.strip_export() for n in nets]
    for i, n in enumerate(nets):
        if i > 0:
            n.strip_attach(api.STRIP_ABOVE, descs[i - 1])
        if i + 1 < len(nets):
            n.strip_attach(api.STRIP_BELOW, descs[i + 1])
    return nets


@pytest.fixture(scope="module")
def images(models):
    """A QP model (fast requantiser) and an edge model on the generic requantiser (k_enh_sse<false, true>,
    k_fused<false, false, true>)."""
    _, seed, family, variant = [e for e in synth.edge_models() if e[0] == "full_scale-generic"][0]
    return {"qp27": formats.write_model_vect_c(models[27]),
            "full_scale-generic": formats.write_model_vect_c(synth.make_edge_model(seed, family, variant))}


def _sequence(tmp_path, h, w, n, seed):
    anchor, ori = synth.make_frames(seed, n, h, w)
    _write_yuv(tmp_path / "anchor.yuv", anchor, seed + 1)
    _write_yuv(tmp_path / "ori.yuv", ori, seed + 2)
    return anchor, ori


@pytest.mark.parametrize("S", [1, 2, 3])
@pytest.mark.parametrize("geom", [(61, 250), (120, 208)], ids=["61x250", "120x208"])
@pytest.mark.parametrize("model", ["qp27", "full_scale-generic"])
def test_equals_frame_sharded_stream(tmp_path, images, handles, model, geom, S):
    from oracle import oracle
    h, w = geom
    image = images[model]
    anchor, ori = _sequence(tmp_path, h, w, FRAMES, 0xC0FFEE + 51 + h)
    whole = api.QVRCNN(0, 3, 1, h, w)
    whole.load_static_para_mem(image)
    want_b, want_a = whole.stream_yuv_pf(str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), str(tmp_path / "whole.yuv"), 0, FRAMES)
    whole.close()
    nets = _strips(handles, image, h, w, _bounds(h, S), [0] * S)
    b, a = api.strip_stream_yuv_pf(nets, str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), str(tmp_path / "strips.yuv"), 0, FRAMES)
    assert (tmp_path / "strips.yuv").read_bytes() == (tmp_path / "whole.yuv").read_bytes()
    luma, chroma = _luma(tmp_path / "strips.yuv", FRAMES, h, w)
    assert not chroma.any()
    assert b.dtype == np.int64 and a.dtype == np.int64 and len(b) == len(a) == FRAMES
    assert np.array_equal(b, want_b) and np.array_equal(a, want_a)
    assert np.array_equal(b, _np_sse(anchor, ori)) and np.array_equal(a, _np_sse(luma, ori))
    if h == 61:
        assert np.array_equal(luma, oracle.OracleModel(image).forward_blu(anchor))


def test_a_range_in_the_middle(tmp_path, images, handles):
    h, w, n = 61, 250, 8
    anchor, ori = _sequence(tmp_path, h, w, n, 0xC0FFEE + 52)
    nets = _strips(handles, images["qp27"], h, w, _bounds(h, 2), [0, 0])
    whole = api.QVRCNN(0, 1, 1, h, w)
    whole.load_static_para_mem(images["qp27"])
    want = whole.forward_frames_host(anchor)
    whole.close()
    fsz = h * w * 3 // 2
    for with_ori in (True, False):
        rec = tmp_path / ("recon_%d.yuv" % with_ori)
        rec.write_bytes(b"\xab" * (n * fsz))
        b, a = api.strip_stream_yuv_pf(nets, str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv") if with_ori else None, str(rec), 3, 2)
        raw = np.fromfile(str(rec), np.uint8).reshape(n, fsz)
        assert (raw[[0, 1, 2, 5, 6, 7]] == 0xAB).all()
        assert np.array_equal(raw[3:5, :h * w].reshape(2, h, w), want[3:5]) and not raw[3:5, h * w:].any()
        if with_ori:
            assert np.array_equal(b, _np_sse(anchor[3:5], ori[3:5])) and np.array_equal(a, _np_sse(want[3:5], ori[3:5]))
        else:
            assert not b.any() and not a.any()
    assert (tmp_path / "recon_1.yuv").read_bytes() == (tmp_path / "recon_0.yuv").read_bytes()


def test_strips_split_over_calls_on_one_device_are_refused(tmp_path, images, handles):
    h, w = 40, 64
    nets = _strips(handles, images["qp27"], h, w, _bounds(h, 2), [0, 0])
    with pytest.raises(api.QVError) as e:          # the anchor does not exist either: no file is opened before the check
        api.strip_stream_yuv_pf(nets[:1], str(tmp_path / "missing.yuv"), None, str(tmp_path / "recon.yuv"), 0, 1)
    assert e.value.code == -5, e.value
    assert "not in this call" in str(e.value)
    assert not (tmp_path / "recon.yuv").exists()


def test_strips_split_over_calls_on_two_devices(tmp_path, images, handles):
    if _ndev() < 2:
        pytest.skip("needs 2 devices")
    h, w, n = 120, 208, FRAMES
    anchor, ori = _sequence(tmp_path, h, w, n, 0xC0FFEE + 53)
    files = [str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv")]
    nets = _strips(handles, images["qp27"], h, w, _bounds(h, 2), [0, 1])
    one_b, one_a = api.strip_stream_yuv_pf(nets, *files, str(tmp_path / "one_call.yuv"), 0, n)
    got = [None, None]

    def run(i):
        try:
            got[i] = api.strip_stream_yuv_pf([nets[i]], *files, str(tmp_path / "two_calls.yuv"), 0, n)
        except Exception as ex:                    # re-raised below, in the test's thread
            got[i] = ex
    th = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    for r in got:
        assert not isinstance(r, Exception), r
    assert (tmp_path / "two_calls.yuv").read_bytes() == (tmp_path / "one_call.yuv").read_bytes()
    assert np.array_equal(got[0][0] + got[1][0], one_b) and np.array_equal(got[0][1] + got[1][1], one_a)
    luma, _ = _luma(tmp_path / "one_call.yuv", n, h, w)
    assert np.array_equal(one_b, _np_sse(anchor, ori)) and np.array_equal(one_a, _np_sse(luma, ori))
    whole = api.QVRCNN(0, 1, 1, h, w)
    whole.load_static_para_mem(images["qp27"])
    assert np.array_equal(luma, whole.forward_frames_host(anchor))
    whole.close()


def _raw_call(nets, n_nets, anchor, ori, recon, first, n, before=None, after=None):
    arr = None if nets is None else (C.c_void_p * max(len(nets), 1))(*[x._h.value for x in nets])
    enc = lambda p: os.fsencode(p) if p else None
    return api.lib().qv_strip_stream_yuv_pf(arr, n_nets, enc(anchor), enc(ori), enc(recon), first, n, before, after)


def test_errors(tmp_path, images, handles):
    image = images["qp27"]
    h, w = 40, 64
    _sequence(tmp_path, h, w, 2, 0xC0FFEE + 54)
    A, O, R = str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), str(tmp_path / "recon.yuv")
    old = bytes(range(256)) * 50
    (tmp_path / "recon.yuv").write_bytes(old)
    nets = _strips(handles, image, h, w, _bounds(h, 2), [0, 0])
    sse = np.zeros(2, np.int64)

    def refused(code, *args, **kw):
        assert _raw_call(*args, **kw) == code, api.lib().qv_last_error()
        assert (tmp_path / "recon.yuv").read_bytes() == old

    # QV_ERR_ARG
    refused(-1, None, 1, A, O, R, 0, 1)
    refused(-1, nets, 0, A, O, R, 0, 1)
    refused(-1, [nets[0], nets[1], nets[0]], 3, A, O, R, 0, 1)
    refused(-1, nets, 2, A, O, R, -1, 1)
    refused(-1, nets, 2, A, O, R, 0, -1)
    refused(-1, nets, 2, A, None, R, 0, 1, before=sse.ctypes.data)
    refused(-1, nets, 2, A, None, R, 0, 1, after=sse.ctypes.data)
    other_w = _strips(handles, image, h, w + 16, [0, h], [0])
    other_h = _strips(handles, image, h + 8, w, [0, h + 8], [0])
    refused(-1, nets + other_w, 3, A, O, R, 0, 1)
    refused(-1, nets + other_h, 3, A, O, R, 0, 1)
    tall_h = 66052                                  # the fused SSE path's height limit is 66051 rows
    tall = _strips(handles, image, tall_h, 8, _bounds(tall_h, 2), [0, 0])
    refused(-1, tall, 2, A, O, R, 0, 1)
    # QV_ERR_STATE
    no_setup = handles(0, h, w, image)
    refused(-5, [no_setup], 1, A, O, R, 0, 1)
    lonely = handles(0, 20, w, image)
    lonely.strip_setup(h, 0, 20)
    refused(-5, [lonely], 1, A, O, R, 0, 1)         # an interior edge with no neighbour attached
    other_w[0].set_impl(api.IMPL_LAYERED)
    refused(-5, other_w, 1, A, O, R, 0, 1)          # no fused path
    refused(-5, nets[:1], 1, A, O, R, 0, 1)         # the device holds strips that are not in the call
    for n in other_w + other_h + tall + [lonely]:
        n.strip_release()
    # the call succeeds once every strip of the device is in it
    assert _raw_call(nets, 2, A, O, R, 0, 2) == 0, api.lib().qv_last_error()
    done = (tmp_path / "recon.yuv").read_bytes()
    # QV_ERR_IO
    assert _raw_call(nets, 2, str(tmp_path / "missing.yuv"), O, R, 0, 1) == -2
    assert _raw_call(nets, 2, A, str(tmp_path / "missing.yuv"), R, 0, 1) == -2
    assert _raw_call(nets, 2, A, O, str(tmp_path / "no_such_dir" / "recon.yuv"), 0, 1) == -2
    assert _raw_call(nets, 2, A, O, R, 1, 2) == -2, "short read: the files hold 2 frames"
    assert "short read" in api.lib().qv_last_error().decode()
    # n_frames == 0: nothing to do, no file touched
    assert _raw_call(nets, 2, A, O, str(tmp_path / "never.yuv"), 0, 0) == 0
    assert not (tmp_path / "never.yuv").exists()
    assert _raw_call(nets, 2, A, O, R, 0, 0) == 0 and (tmp_path / "recon.yuv").read_bytes() == done


@pytest.mark.parametrize("mode", ["frames", "strips"])
def test_reconstruction_write_failure(tmp_path, images, handles, mode):
    """A reconstruction file that takes no bytes (/dev/full): the streaming call returns QV_ERR_IO instead of hanging, and the
    same handles then stream exactly as fresh ones do.  Frames: qv_stream_yuv_pf in chunks of 4 over 11 frames (3 chunks, the
    last one short); strips: 2 strips on one device, 7 frames."""
    if not os.path.exists("/dev/full"):
        pytest.skip("no /dev/full")
    h, w = 61, 250
    n = 11 if mode == "frames" else FRAMES
    _sequence(tmp_path, h, w, n, 0xC0FFEE + 57)
    A, O = str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv")
    image = images["qp27"]

    def make():
        if mode == "frames":
            nets = [handles(0, h, w, image, batch=4)]
            return nets, lambda recon: nets[0].stream_yuv_pf(A, O, recon, 0, n)
        nets = _strips(handles, image, h, w, _bounds(h, 2), [0, 0])
        return nets, lambda recon: api.strip_stream_yuv_pf(nets, A, O, recon, 0, n)
    fresh, call = make()
    want_b, want_a = call(str(tmp_path / "fresh.yuv"))
    for x in fresh:                                 # strips of one device are driven together: the fresh ones leave
        x.strip_release()
    _, call = make()
    with pytest.raises(api.QVError) as e:
        call("/dev/full")
    assert e.value.code == -2, e.value
    assert "write to the reconstruction file failed" in str(e.value)
    b, a = call(str(tmp_path / "again.yuv"))
    assert (tmp_path / "again.yuv").read_bytes() == (tmp_path / "fresh.yuv").read_bytes()
    assert np.array_equal(b, want_b) and np.array_equal(a, want_a)


# ---- the CLI ----------------------------------------------------------------------------------------------------------------
def _cli_inputs(d, h, w, frames, qp, image, seed):
    d.mkdir(exist_ok=True)
    anchor, ori = synth.make_frames(seed, frames, h, w)
    _write_yuv(d / "ori.yuv", ori, seed + 1)
    _write_yuv(d / ("anchor_Q%d.yuv" % qp), anchor, seed + 2)
    (d / ("model_%d.data" % qp)).write_bytes(image)
    return anchor, ori


def _cli(d, h, w, qp, frames, *extra):
    p = subprocess.run([CLI, "ori.yuv", "anchor_", str(h), str(w), "--model", "model_%d.data", "--qp", str(qp), "--frames", str(frames)]
                       + list(extra), cwd=d, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


@pytest.mark.parametrize("strips,gpus", [(3, 1), (2, 2)])
def test_cli_strips_stream(tmp_path, models, strips, gpus):
    """`--strips S --stream` against `--strips S` (in memory) and `--stream` (frame-sharded): same report, same per-frame
    lines, same recon_psnr.data entry, same log.txt entry (apart from date and time), byte-identical reconstruction."""
    if _ndev() < gpus:
        pytest.skip("needs %d devices" % gpus)
    qp, h, w, frames = 27, 96, 200, 5
    image = formats.write_model_vect_c(models[qp])
    runs = {}
    for name, mode in (("strips_stream", ["--strips", str(strips), "--stream"]), ("strips", ["--strips", str(strips)]), ("stream", ["--stream"])):
        d = tmp_path / name
        anchor, ori = _cli_inputs(d, h, w, frames, qp, image, 0xC0FFEE + 55)
        out = _cli(d, h, w, qp, frames, "--gpus", str(gpus), "--save-recon", "r.yuv", "--psnr-pf", *mode)
        log = [l for l in (d / "log.txt").read_text().splitlines() if not l.startswith(("QVRCNN test date:", "time:"))]
        runs[name] = (out, (d / "recon_psnr.data").read_bytes(), log, (d / "r.yuv").read_bytes())
    out, psnr_data, log, rec = runs["strips_stream"]
    assert re.search(r"throughput:.*in %d strip\(s\) on %d GPU\(s\).*streamed from and to files" % (strips, gpus), out), out
    keep = lambda s: [l for l in s.splitlines() if l.startswith(("before net:PSNR=", "after quantized net:PSNR=", "PSNR of Frame", "mean per-frame"))]
    assert len(keep(out)) == 2 + frames + 1
    for other in ("strips", "stream"):
        o_out, o_psnr, o_log, o_rec = runs[other]
        assert keep(out) == keep(o_out), other
        assert psnr_data == o_psnr and len(psnr_data) == 8, other
        assert log == o_log, other
        assert rec == o_rec, other
    from oracle import oracle
    luma, chroma = _luma(tmp_path / "strips_stream" / "r.yuv", frames, h, w)
    assert np.array_equal(luma[:2], oracle.OracleModel(image).forward_blu(anchor[:2])) and not chroma.any()


_RSS = "import resource, subprocess, sys; subprocess.run(sys.argv[1:], check=True, stdout=subprocess.DEVNULL); " \
       "print(resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss)"


def test_cli_host_memory_does_not_grow_with_the_sequence(tmp_path, models):
    """Peak resident memory of the CLI at 8 and at 40 frames of 1080p, one wrapper process per measurement (RUSAGE_CHILDREN
    keeps the largest child seen): streamed, it grows by less than one frame's three arrays; in memory, by the 32 frames'."""
    qp, h, w, frames = 32, 1080, 1920, 40
    rng = np.random.default_rng(56)
    fsz = h * w * 3 // 2
    for name in ("ori.yuv", "anchor_Q%d.yuv" % qp):
        rng.integers(0, 256, size=frames * fsz, dtype=np.uint8).tofile(str(tmp_path / name))
    (tmp_path / ("model_%d.data" % qp)).write_bytes(formats.write_model_vect_c(models[qp]))

    def peak_kb(n, *mode):
        cmd = [CLI, "ori.yuv", "anchor_", str(h), str(w), "--model", "model_%d.data", "--qp", str(qp), "--frames", str(n),
               "--strips", "3", "--save-recon", "r.yuv"] + list(mode)
        p = subprocess.run([sys.executable, "-c", _RSS] + cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout + p.stderr
        return int(p.stdout.split()[-1])
    frame_kb = 3 * h * w / 1024                     # ori + input + recon of one frame
    streamed = peak_kb(frames, "--stream") - peak_kb(8, "--stream")
    in_memory = peak_kb(frames) - peak_kb(8)
    assert streamed < frame_kb, (streamed, in_memory)
    assert in_memory > 0.8 * (frames - 8) * frame_kb, (streamed, in_memory)
