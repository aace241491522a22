"""One frame over several strips with peer-mapped halo rows (qv_strip_*, SURVEY 8e-ii), bit for bit against the
whole-frame result and the oracle.

On a 1-GPU box the strips share device 0 in one process (peer = plain pointer), which runs the whole protocol (two input
slots, sequence words, acquire before reuse, halo rows read out of the neighbour's block) with the stream-level, bounded
waits.  With >= 2 devices the same tests also run one strip per GPU -- peer access in one process, CUDA IPC between
processes, over NVLink -- with the waits inside the fused kernel.  Both through the ctypes binding and through the C++
driver (`qcnn_gpu --strips`, `qcnn_gpu --gpus N`)."""
import json
import os
import re
import socket
import subprocess
import sys

import numpy as np
import pytest

from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, shard, synth

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "qcnn_gpu_b200", "qcnn_gpu")


def _ndev():
    import torch
    return torch.cuda.device_count()


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _write_yuv(path, luma, chroma_value):
    with open(path, "wb") as fp:
        for f in range(luma.shape[0]):
            fp.write(luma[f].tobytes())
            fp.write(bytes([chroma_value]) * (luma.shape[1] * luma.shape[2] // 2))


def _strip_nets(image, h, w, bounds, devices):
    nets = []
    for i in range(len(bounds) - 1):
        n = api.QVRCNN(devices[i], 1, 1, bounds[i + 1] - bounds[i], w)
        n.load_static_para_mem(image)
        n.strip_setup(h, bounds[i], bounds[i + 1])
        nets.append(n)
    descs = [n.strip_export() for n in nets]
    for i, n in enumerate(nets):
        if i > 0:
            n.strip_attach(api.STRIP_ABOVE, descs[i - 1])
        if i + 1 < len(nets):
            n.strip_attach(api.STRIP_BELOW, descs[i + 1])
    return nets


def _run_strips(nets, bounds, frames, w, devices):
    """frames [K,h,w]: K steps, slot k&1.  Strips that share a device are driven on one stream, all loads of a frame before
    its forwards (stream order is what orders them); strips on different devices have a stream each and the fused kernels
    wait for each other's rows themselves."""
    import torch
    K = frames.shape[0]
    outs = [[] for _ in nets]
    streams = {}
    for d in set(devices):
        with torch.cuda.device(d):
            streams[d] = torch.cuda.Stream()
    for k in range(K):
        for i, n in enumerate(nets):
            n.strip_load(k & 1, frames[k, bounds[i]:bounds[i + 1]], streams[devices[i]].cuda_stream)
        for i, n in enumerate(nets):
            with torch.cuda.device(devices[i]):
                o = torch.empty((bounds[i + 1] - bounds[i], w), dtype=torch.uint8, device="cuda")
            n.strip_forward(k & 1, o.data_ptr(), streams[devices[i]].cuda_stream)
            outs[i].append(o)
    for i, n in enumerate(nets):
        n.synchronize(streams[devices[i]].cuda_stream)
    return np.stack([np.concatenate([outs[i][k].cpu().numpy() for i in range(len(nets))]) for k in range(K)])


@pytest.mark.parametrize("layout", ["one_device", "one_strip_per_device"])
def test_strips_equal_whole_frame_and_oracle(models, layout):
    from oracle import oracle
    qp, h, w, K = 22, 150, 250, 5
    if layout == "one_strip_per_device" and _ndev() < 2:
        pytest.skip("needs 2 devices")
    S = 3 if layout == "one_device" else min(_ndev(), 4)
    bounds = [shard.split(h, i, S)[0] for i in range(S)] + [h]
    devices = [0] * S if layout == "one_device" else list(range(S))
    image = formats.write_model_vect_c(models[qp])
    frames, _ = synth.make_frames(0xC0FFEE + 31, K, h, w)
    nets = _strip_nets(image, h, w, bounds, devices)
    got = _run_strips(nets, bounds, frames, w, devices)
    whole = api.QVRCNN(0, 1, 1, h, w)
    whole.load_static_para_mem(image)
    want = whole.forward_frames_host(frames)
    assert np.array_equal(got, want), "strips differ from the whole frame in %d pixels" % int((got != want).sum())
    assert np.array_equal(want[:2], oracle.OracleModel(image).forward_blu(frames[:2]))
    if layout == "one_device":
        # strips that share a GPU must share the stream: a second stream is refused, not raced
        import torch
        other = torch.cuda.Stream()
        with pytest.raises(api.QVError, match="ONE caller-provided stream"):
            nets[1].strip_load(0, frames[0, bounds[1]:bounds[2]], other.cuda_stream)
    for n in nets:
        n.strip_release()


@pytest.mark.parametrize("h,w,S", [(18, 61, 3), (40, 130, 2), (97, 121, 5), (64, 8, 4)])
def test_strips_ragged_geometries(models, h, w, S):
    """Strips of exactly the halo height, heights that do not divide, widths below / just above one 120-pixel strip column:
    every split reproduces the oracle's frame (strips on one device: the stream-ordered layout)."""
    from oracle import oracle
    image = formats.write_model_vect_c(models[37])
    frames, _ = synth.make_frames(0xC0FFEE + 34, 2, h, w)
    bounds = [shard.split(h, i, S)[0] for i in range(S)] + [h]
    nets = _strip_nets(image, h, w, bounds, [0] * S)
    got = _run_strips(nets, bounds, frames, w, [0] * S)
    assert np.array_equal(got, oracle.OracleModel(image).forward_blu(frames))
    for n in nets:
        n.strip_release()


def test_strip_api_refuses_what_it_cannot_do(models):
    image = formats.write_model_vect_c(models[27])
    h, w = 40, 64
    a = api.QVRCNN(0, 1, 1, 20, w); a.load_static_para_mem(image)
    b = api.QVRCNN(0, 1, 1, 20, w); b.load_static_para_mem(image)
    with pytest.raises(api.QVError, match="qv_strip_setup"):
        a.strip_export()
    a.strip_setup(h, 0, 20)
    b.strip_setup(h, 20, 40)
    import torch
    o = torch.empty((20, w), dtype=torch.uint8, device="cuda")
    with pytest.raises(api.QVError, match="no neighbour attached"):
        a.strip_forward(0, o.data_ptr())
    a.strip_attach(api.STRIP_BELOW, b.strip_export())
    with pytest.raises(api.QVError, match="has not filled slot"):          # same GPU: loads of a frame come before its forwards
        a.strip_forward(0, o.data_ptr())
    with pytest.raises(api.QVError, match="not adjacent"):
        a.strip_attach(api.STRIP_ABOVE, b.strip_export())
    with pytest.raises(api.QVError, match="not a strip descriptor"):
        a.strip_attach(api.STRIP_BELOW, b"\0" * api.STRIP_DESC_BYTES)
    # a neighbour with fewer rows than the halo
    c = api.QVRCNN(0, 1, 1, 5, w); c.load_static_para_mem(image)
    d = api.QVRCNN(0, 1, 1, 35, w); d.load_static_para_mem(image)
    c.strip_setup(h, 0, 5)
    d.strip_setup(h, 5, 40)
    with pytest.raises(api.QVError, match="fewer than the 6-row halo"):
        d.strip_attach(api.STRIP_ABOVE, c.strip_export())
    # a single strip covering the image needs nobody
    e = api.QVRCNN(0, 1, 1, h, w); e.load_static_para_mem(image)
    e.strip_setup(h, 0, h)
    x, _ = synth.make_frames(5, 1, h, w)
    oo = torch.empty((h, w), dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    for n in (a, b, c, d):
        n.strip_release()
    e.strip_load(0, x[0], st.cuda_stream)
    e.strip_forward(0, oo.data_ptr(), st.cuda_stream)
    e.synchronize(st.cuda_stream)
    want = e.forward_frames_host(x)[0]
    assert np.array_equal(oo.cpu().numpy(), want)
    # a descriptor outlives its strip: once the strip is released, attaching its descriptor is refused
    a.strip_setup(h, 0, 20)
    b.strip_setup(h, 20, 40)
    old = b.strip_export()
    b.strip_release()
    with pytest.raises(api.QVError, match="neighbour strip was released"):
        a.strip_attach(api.STRIP_BELOW, old)
    # releasing a strip unlinks it from the strips that had it attached, also once it is set up again, until re-attached
    b.strip_setup(h, 20, 40)
    a.strip_attach(api.STRIP_BELOW, b.strip_export())
    b.strip_attach(api.STRIP_ABOVE, a.strip_export())
    a.strip_release()
    with pytest.raises(api.QVError, match="no neighbour attached"):
        b.strip_forward(0, o.data_ptr())
    a.strip_setup(h, 0, 20)
    with pytest.raises(api.QVError, match="no neighbour attached"):
        b.strip_forward(0, o.data_ptr())
    b.strip_attach(api.STRIP_ABOVE, a.strip_export())
    a.strip_attach(api.STRIP_BELOW, b.strip_export())
    ob = torch.empty((20, w), dtype=torch.uint8, device="cuda")
    a.strip_load(0, x[0][:20], st.cuda_stream)
    b.strip_load(0, x[0][20:], st.cuda_stream)
    a.strip_forward(0, o.data_ptr(), st.cuda_stream)
    b.strip_forward(0, ob.data_ptr(), st.cuda_stream)
    b.synchronize(st.cuda_stream)
    assert np.array_equal(np.vstack([o.cpu().numpy(), ob.cpu().numpy()]), want)
    # a second strip_setup of a live strip, and qv_destroy, unlink it the same way
    b.strip_setup(h, 20, 40)
    with pytest.raises(api.QVError, match="no neighbour attached"):
        a.strip_forward(0, o.data_ptr(), st.cuda_stream)
    a.strip_attach(api.STRIP_BELOW, b.strip_export())
    b.close()
    with pytest.raises(api.QVError, match="no neighbour attached"):
        a.strip_forward(0, o.data_ptr(), st.cuda_stream)


@pytest.mark.parametrize("strips,gpus", [(3, 1), (2, 2), (4, 2), (8, 8)])
def test_cli_strips(tmp_path, models, strips, gpus):
    """The C++ driver: `qcnn_gpu --strips S --gpus G` (strip i on device i mod G), several frames so that both input slots
    and the acquire-before-reuse wait are exercised; report and reconstruction file equal the oracle's."""
    from oracle import oracle
    if _ndev() < gpus:
        pytest.skip("needs %d devices" % gpus)
    qp, h, w, frames = 27, 96, 200, 4
    anchor, ori = synth.make_frames(0xC0FFEE + 32, frames, h, w)
    _write_yuv(tmp_path / "ori.yuv", ori, 0x80)
    _write_yuv(tmp_path / ("anchor_Q%d.yuv" % qp), anchor, 0x33)
    image = formats.write_model_vect_c(models[qp])
    (tmp_path / ("model_%d.data" % qp)).write_bytes(image)
    p = subprocess.run([CLI, "ori.yuv", "anchor_", str(h), str(w), "--model", "model_%d.data", "--qp", str(qp), "--frames", str(frames),
                        "--gpus", str(gpus), "--strips", str(strips), "--save-recon", "recon.yuv"],
                       cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    want = oracle.OracleModel(image).forward_blu(anchor)
    after = float(re.search(r"after quantized net:PSNR=([0-9.]+)", p.stdout).group(1))
    assert after == pytest.approx(round(oracle.psnr(want, ori)[0], 3), abs=1.1e-3)
    raw = np.frombuffer((tmp_path / "recon.yuv").read_bytes(), np.uint8).reshape(frames, h * w * 3 // 2)
    assert np.array_equal(raw[:, :h * w].reshape(frames, h, w), want)


@pytest.mark.parametrize("gpus", [2, 8])
def test_cli_frame_shards_on_several_gpus(tmp_path, models, gpus):
    """`qcnn_gpu --gpus N`: frame-sharded over N devices, one host thread per device == the oracle."""
    from oracle import oracle
    if _ndev() < gpus:
        pytest.skip("needs %d devices" % gpus)
    qp, h, w, frames = 37, 64, 112, 2 * gpus + 1
    anchor, ori = synth.make_frames(0xC0FFEE + 33, frames, h, w)
    _write_yuv(tmp_path / "ori.yuv", ori, 0x80)
    _write_yuv(tmp_path / ("anchor_Q%d.yuv" % qp), anchor, 0x33)
    image = formats.write_model_vect_c(models[qp])
    (tmp_path / ("model_%d.data" % qp)).write_bytes(image)
    p = subprocess.run([CLI, "ori.yuv", "anchor_", str(h), str(w), "--model", "model_%d.data", "--qp", str(qp), "--frames", str(frames),
                        "--gpus", str(gpus), "--save-recon", "recon.yuv"], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stdout + p.stderr
    want = oracle.OracleModel(image).forward_blu(anchor)
    raw = np.frombuffer((tmp_path / "recon.yuv").read_bytes(), np.uint8).reshape(frames, h * w * 3 // 2)
    assert np.array_equal(raw[:, :h * w].reshape(frames, h, w), want)


def _torchrun(nproc, extra, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), "-m", "qcnn_gpu_b200.host.multi_gpu"] + extra
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-4000:]
    line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
    return json.loads(line)


def test_multiprocess_strips_bit_identical():
    """One process per GPU (the bench's launch shape): the neighbours' blocks are mapped through CUDA IPC and the fused kernel
    waits for their rows itself; every step of the check uploads a different frame, alternating the input slots; rank 0
    recomputes every frame alone.  (Never several ranks on ONE GPU: kernels of different processes that wait for each
    other are not guaranteed to run at the same time -- qv_strip_attach refuses that layout.)"""
    if _ndev() < 2:
        pytest.skip("needs 2 devices")
    nproc = min(_ndev(), 8)
    r = _torchrun(nproc, ["--mode", "strips", "--qp", "22", "--height", "270", "--width", "480", "--steps", "6", "--check"])
    assert r["bit_identical_to_1gpu"] is True and r["distinct_frames_checked"] == 6, r
    assert r["n_gpus"] == nproc


def test_multiprocess_frame_shards_bit_identical():
    if _ndev() < 2:
        pytest.skip("needs 2 devices")
    nproc = min(_ndev(), 8)
    r = _torchrun(nproc, ["--mode", "frames", "--qp", "27", "--frames", str(3 * nproc + 1), "--height", "270", "--width", "480", "--steps", "2",
                          "--check", "--uniq", "2"])
    assert r["bit_identical_to_1gpu"] is True, r
