"""Per-frame SSE / PSNR from the GPU (vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112): k_enh_sse adds, per frame, the
exact sums (anchor - ori)^2 and (rec - ori)^2 in the fused kernel's output stage; the layered path gets them from a separate
pass per frame.  Every entry point is checked against numpy, the reconstruction against the plain forward and the oracle."""
import ctypes as C
import math
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest

from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, shard, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "qcnn_gpu_b200", "qcnn_gpu")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
SHAPES = [(1, 1), (1, 9), (7, 5), (13, 13), (33, 31), (8, 257), (130, 20), (61, 123)]


# ---- no GPU: what the library's SSE kernels compiled to -------------------------------------------------------------------
@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_sse_kernels_sass():
    api.lib()
    out = subprocess.run([CUOBJDUMP, "-sass", api.LIB_PATH], capture_output=True, text=True, check=True).stdout
    kernels, name = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            name = m.group(1)
            kernels[name] = []
        elif name and "/*" in line:
            kernels[name].append(line)
    sse = {k: "\n".join(v) for k, v in kernels.items() if "k_enh_sse" in k}
    assert len(sse) == 4, list(sse)                  # {FAST, generic requantiser} x {whole frames, row window}
    for k, text in sse.items():
        assert "k_fused" not in k
        assert len(re.findall(r"\bUTCIMMA\b", text)) == 27, k
        assert "A_KEEP" in text and "A_REUSE" in text, k
        assert "LDTM" in text and "UTCBAR" in text, k
        assert "UTMALDG" not in text, k                # no TMA form
        assert not re.search(r"\bLDL\b", text) and len(re.findall(r"\bSTL\b", text)) <= 3, k


# ---- GPU ------------------------------------------------------------------------------------------------------------------
def _np_sse(x, ori):
    return ((x.astype(np.int64) - ori.astype(np.int64)) ** 2).reshape(len(ori), -1).sum(axis=1)


def _net(model, batch, h, w, impl=api.IMPL_FUSED):
    net = api.QVRCNN(0, batch, 1, h, w)
    net.load_static_para_mem(formats.write_model_vect_c(model))
    net.set_impl(impl)
    return net


def _sse_run(net, anchor, ori, calls=1, stream=0):
    """forward_frames_device_sse on device copies; returns (out, sse [n, 2])"""
    import torch
    d_in, d_ori = torch.from_numpy(anchor).cuda(), torch.from_numpy(ori).cuda()
    d_out = torch.empty_like(d_in)
    d_sse = torch.zeros((len(anchor), 2), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    for _ in range(calls):
        net.forward_frames_device_sse(d_in.data_ptr(), d_ori.data_ptr(), d_out.data_ptr(), len(anchor), d_sse.data_ptr(), stream)
    if stream:
        net.synchronize(stream)
    return d_out.cpu().numpy(), d_sse.cpu().numpy()


def _plain_run(net, anchor):
    import torch
    d_in = torch.from_numpy(anchor).cuda()
    d_out = torch.empty_like(d_in)
    net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), len(anchor))
    return d_out.cpu().numpy()


def _frames(seed, n, h, w):
    a = synth.make_uniform_frames(seed, n, h, w)
    o = synth.make_uniform_frames(seed + 1, n, h, w)
    return a, o


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("qp", [22, 27, 32, 37])
def test_fused_sse_matches_numpy(models, qp, shape):
    """5 frames on a handle of batch 2 (n > batch, not a multiple of it), ragged and tiny shapes"""
    from oracle import oracle
    h, w = shape
    anchor, ori = _frames(qp * 100 + h, 5, h, w)
    net = _net(models[qp], 2, h, w)
    out, sse = _sse_run(net, anchor, ori)
    assert np.array_equal(out, _plain_run(net, anchor))
    assert np.array_equal(out[:1], oracle.OracleModel(formats.write_model_vect_c(models[qp])).forward_blu(anchor[:1]))
    assert np.array_equal(sse[:, 0], _np_sse(anchor, ori))
    assert np.array_equal(sse[:, 1], _np_sse(out, ori))


def _units(n, h, w, line):
    L = api.lib()
    L.qv_debug_fused_units.argtypes = [C.c_int] * 8 + [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
    cnt, grid = C.c_size_t(0), C.c_int(0)
    assert L.qv_debug_fused_units(148, n, h, w, 0, h, 0, line, None, C.byref(cnt), C.byref(grid)) == 0
    u = np.zeros((cnt.value, 5), np.int32)
    assert L.qv_debug_fused_units(148, n, h, w, 0, h, 0, line, u.ctypes.data, C.byref(cnt), C.byref(grid)) == 0
    return u


@pytest.mark.gpu
def test_row_line_plan_across_frames_and_layered_cross_check(models):
    """A geometry dealt out by the row line (P.linear) in which one CTA's pieces belong to different frames: the per-frame
    flush must go to the right frame.  The layered path gives the same numbers; calls add up; asynchronous calls report
    after a synchronize."""
    import torch
    n, h, w = 26, 56, 250
    u = _units(n, h, w, 1)
    assert not np.array_equal(u, _units(n, h, w, 0)), "expected the row-line plan"
    assert any(len(set(u[u[:, 0] == c][:, 1])) > 1 for c in set(u[:, 0])), "expected a CTA that spans frames"
    anchor, ori = synth.make_frames(0xC0FFEE + 41, n, h, w)
    net = _net(models[27], 8, h, w)
    out, sse = _sse_run(net, anchor, ori)
    assert np.array_equal(out, _plain_run(net, anchor))
    want = np.stack([_np_sse(anchor, ori), _np_sse(out, ori)], axis=1)
    assert np.array_equal(sse, want)
    _, twice = _sse_run(net, anchor, ori, calls=2)
    assert np.array_equal(twice, 2 * want)
    st = torch.cuda.Stream()
    _, asy = _sse_run(net, anchor, ori, stream=st.cuda_stream)
    assert np.array_equal(asy, want)
    lay = _net(models[27], 8, h, w, api.IMPL_LAYERED)
    lout, lsse = _sse_run(lay, anchor, ori)
    assert np.array_equal(lout, out) and np.array_equal(lsse, want)
    _, ltwice = _sse_run(lay, anchor, ori, calls=2)
    assert np.array_equal(ltwice, 2 * want)


@pytest.mark.gpu
@pytest.mark.parametrize("impl", [api.IMPL_FUSED, api.IMPL_LAYERED], ids=["fused", "layered"])
def test_edge_values(models, impl):
    h, w = 40, 130
    same = np.full((2, h, w), 77, np.uint8)
    net = _net(models[32], 2, h, w, impl)
    out, sse = _sse_run(net, same, same)
    assert (sse[:, 0] == 0).all() and np.array_equal(sse[:, 1], _np_sse(out, same))
    assert api.psnr_from_sse(int(sse[0, 0]), h * w) == float("inf")
    # the largest per-pixel error: all 0 against all 255 and the other way round
    lo, hi = np.zeros((1, h, w), np.uint8), np.full((1, h, w), 255, np.uint8)
    anchor, ori = np.concatenate([lo, hi]), np.concatenate([hi, lo])
    out, sse = _sse_run(net, anchor, ori)
    assert (sse[:, 0] == 255 * 255 * h * w).all()
    assert np.array_equal(sse[:, 1], _np_sse(out, ori))


@pytest.mark.gpu
def test_argument_errors(models):
    import torch
    net = _net(models[32], 1, 16, 16)
    x = torch.zeros((1, 16, 16), dtype=torch.uint8, device="cuda")
    s = torch.zeros((1, 2), dtype=torch.int64, device="cuda")
    with pytest.raises(api.QVError) as e:
        net.forward_frames_device_sse(x.data_ptr(), 0, x.data_ptr(), 1, s.data_ptr())
    assert e.value.code == -1
    with pytest.raises(api.QVError) as e:
        net.forward_frames_device_sse(x.data_ptr(), x.data_ptr(), x.data_ptr(), 1, 0)
    assert e.value.code == -1
    net.strip_setup(16, 0, 16)
    with pytest.raises(api.QVError) as e:
        net.strip_forward_sse(0, 0, x.data_ptr(), s.data_ptr())
    assert e.value.code == -1
    net.set_impl(api.IMPL_LAYERED)
    with pytest.raises(api.QVError) as e:
        net.strip_forward_sse(0, x.data_ptr(), x.data_ptr(), s.data_ptr())
    assert e.value.code == -5
    net.strip_release()
    with pytest.raises(api.QVError):
        net.stream_yuv_pf("/nonexistent/anchor.yuv", None, None, 0, 1)


def _ndev():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["two_strips", "three_strips", "one_strip_per_device"])
def test_strip_sse_adds_up_to_the_frame(models, layout):
    import torch
    qp, h, w, K = 22, 150, 250, 3
    if layout == "one_strip_per_device" and _ndev() < 2:
        pytest.skip("needs 2 devices")
    S = {"two_strips": 2, "three_strips": 3}.get(layout) or min(_ndev(), 4)
    devices = [0] * S if layout != "one_strip_per_device" else list(range(S))
    bounds = [shard.split(h, i, S)[0] for i in range(S)] + [h]
    image = formats.write_model_vect_c(models[qp])
    anchor, ori = synth.make_frames(0xC0FFEE + 42, K, h, w)
    nets = []
    for i in range(S):
        n = api.QVRCNN(devices[i], 1, 1, bounds[i + 1] - bounds[i], w)
        n.load_static_para_mem(image)
        n.strip_setup(h, bounds[i], bounds[i + 1])
        nets.append(n)
    descs = [n.strip_export() for n in nets]
    for i, n in enumerate(nets):
        if i > 0:
            n.strip_attach(api.STRIP_ABOVE, descs[i - 1])
        if i + 1 < S:
            n.strip_attach(api.STRIP_BELOW, descs[i + 1])
    streams, outs, sses, keep = {}, [[] for _ in nets], [], []
    for d in set(devices):
        with torch.cuda.device(d):
            streams[d] = torch.cuda.Stream()
    for i in range(S):
        with torch.cuda.device(devices[i]):
            sses.append(torch.zeros((K, 2), dtype=torch.int64, device="cuda"))
    for k in range(K):                            # strips that share a device: one stream, all loads of a frame first
        for i, n in enumerate(nets):
            n.strip_load(k & 1, anchor[k, bounds[i]:bounds[i + 1]], streams[devices[i]].cuda_stream)
        for i, n in enumerate(nets):
            with torch.cuda.device(devices[i]), torch.cuda.stream(streams[devices[i]]):
                o = torch.empty((bounds[i + 1] - bounds[i], w), dtype=torch.uint8, device="cuda")
                r = torch.from_numpy(ori[k, bounds[i]:bounds[i + 1]].copy()).to("cuda", non_blocking=False)
            keep.append(r)
            n.strip_forward_sse(k & 1, r.data_ptr(), o.data_ptr(), sses[i][k].data_ptr(), streams[devices[i]].cuda_stream)
            outs[i].append(o)
    for i, n in enumerate(nets):
        n.synchronize(streams[devices[i]].cuda_stream)
    got = np.stack([np.concatenate([outs[i][k].cpu().numpy() for i in range(S)]) for k in range(K)])
    total = sum(s.cpu().numpy() for s in sses)
    whole = _net(models[qp], 1, h, w)
    out, sse = _sse_run(whole, anchor, ori)
    assert np.array_equal(got, out)
    assert np.array_equal(total, sse)
    assert np.array_equal(sse, np.stack([_np_sse(anchor, ori), _np_sse(out, ori)], axis=1))
    for n in nets:
        n.strip_release()


def _write_yuv(path, luma, chroma_value):
    with open(path, "wb") as fp:
        for f in range(luma.shape[0]):
            fp.write(luma[f].tobytes())
            fp.write(bytes([chroma_value]) * (luma.shape[1] * luma.shape[2] // 2))


@pytest.mark.gpu
@pytest.mark.parametrize("impl", [api.IMPL_FUSED, api.IMPL_LAYERED], ids=["fused", "layered"])
def test_stream_yuv_pf(tmp_path, models, impl):
    qp, h, w, frames = 27, 72, 250, 11
    anchor, ori = synth.make_frames(0xC0FFEE + 43, frames, h, w)
    _write_yuv(tmp_path / "ori.yuv", ori, 0x80)
    _write_yuv(tmp_path / "anchor.yuv", anchor, 0x33)
    net = _net(models[qp], 4, h, w, impl)                 # chunks of 4: 4 + 4 + 3
    want = net.forward_frames_host(anchor)
    b, a = net.stream_yuv_pf(str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), str(tmp_path / "pf.yuv"), 0, frames)
    assert b.dtype == np.int64 and a.dtype == np.int64
    assert np.array_equal(b, _np_sse(anchor, ori)) and np.array_equal(a, _np_sse(want, ori))
    assert net.stream_yuv(str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), str(tmp_path / "pooled.yuv"), 0, frames) == (int(b.sum()), int(a.sum()))
    assert (tmp_path / "pf.yuv").read_bytes() == (tmp_path / "pooled.yuv").read_bytes()
    raw = np.frombuffer((tmp_path / "pf.yuv").read_bytes(), np.uint8).reshape(frames, h * w * 3 // 2)
    assert np.array_equal(raw[:, :h * w].reshape(frames, h, w), want)
    b2, a2 = net.stream_yuv_pf(str(tmp_path / "anchor.yuv"), str(tmp_path / "ori.yuv"), None, 5, 3)   # a range in the middle
    assert np.array_equal(b2, b[5:8]) and np.array_equal(a2, a[5:8])


def _cli(tmp_path, h, w, qp, frames, *extra):
    p = subprocess.run([CLI, "ori.yuv", "anchor_", str(h), str(w), "--model", "model_%d.data", "--qp", str(qp), "--frames", str(frames)]
                       + list(extra), cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    return p.stdout


@pytest.mark.gpu
def test_cli_psnr_pf(tmp_path, models):
    from oracle import oracle
    qp, h, w, frames = 32, 64, 112, 5
    anchor, ori = synth.make_frames(0xC0FFEE + 44, frames, h, w)
    anchor[2] = ori[2]                                    # one frame identical to its original: PSNR before = inf
    _write_yuv(tmp_path / "ori.yuv", ori, 0x80)
    _write_yuv(tmp_path / ("anchor_Q%d.yuv" % qp), anchor, 0x33)
    (tmp_path / ("model_%d.data" % qp)).write_bytes(formats.write_model_vect_c(models[qp]))
    want = oracle.OracleModel(formats.write_model_vect_c(models[qp])).forward_blu(anchor)
    n = h * w
    psnr = lambda s: 10 * math.log10(65025.0 / (float(s) / n)) if s else float("inf")      # qv_psnr_from_sse's arithmetic
    lines = ["PSNR of Frame %d:%f" % (k, psnr(s)) for k, s in enumerate(_np_sse(want, ori))]
    mean_b = np.mean([psnr(s) for s in _np_sse(anchor, ori)])
    mean_a = np.mean([psnr(s) for s in _np_sse(want, ori)])
    lines.append("mean per-frame PSNR: before net:%f after quantized net:%f" % (mean_b, mean_a))
    for mode in ([], ["--stream"], ["--strips", "2"]):
        plain = _cli(tmp_path, h, w, qp, frames, *mode)
        psnr_file = (tmp_path / "recon_psnr.data").read_bytes()
        with_pf = _cli(tmp_path, h, w, qp, frames, *(mode + ["--psnr-pf"]))
        got = [l for l in with_pf.splitlines() if l.startswith("PSNR of Frame") or l.startswith("mean per-frame")]
        assert got == lines, (mode, got, lines)
        # without the flag nothing is printed per frame, and the report itself does not depend on the flag
        assert "PSNR of Frame" not in plain
        strip = lambda s: [l for l in s.splitlines() if not l.startswith(("time:", "throughput:", "PSNR of Frame", "mean per-frame"))]
        assert strip(plain) == strip(with_pf)
        rec = (tmp_path / "recon_psnr.data").read_bytes()
        assert rec[:len(psnr_file)] == psnr_file and rec[len(psnr_file):] == psnr_file[-8:]
        (tmp_path / "recon_psnr.data").unlink()
        (tmp_path / "log.txt").unlink()


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _torchrun(nproc, extra, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), "-m", "qcnn_gpu_b200.host.multi_gpu"] + extra
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    import json
    return json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])


@pytest.mark.gpu
@pytest.mark.parametrize("nproc", [1, 2])
@pytest.mark.parametrize("mode", ["frames", "strips"])
def test_multi_gpu_per_frame(mode, nproc):
    if nproc > _ndev():
        pytest.skip("needs %d devices" % nproc)
    extra = ["--frames", "7", "--uniq", "3"] if mode == "frames" else []
    r = _torchrun(nproc, ["--mode", mode, "--qp", "27", "--height", "270", "--width", "480", "--steps", "2", "--check", "--per-frame"] + extra)
    assert r["bit_identical_to_1gpu"] is True and r["per_frame_sse_identical_to_1gpu"] is True, r
    n = 7 if mode == "frames" else 1
    assert len(r["psnr_per_frame_before"]) == n and len(r["psnr_per_frame_after"]) == n
    assert r["psnr_per_frame_mean_after"] == pytest.approx(np.mean(r["psnr_per_frame_after"]))
