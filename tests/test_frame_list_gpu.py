"""Frames of different resolutions in one call (qv_forward_frame_list_device): every frame's output is byte-identical to
qv_forward_frames_device on a handle of that frame's geometry, its SSE pair to qv_forward_frames_device_sse, on the fused
path (k_enh_list) and on the layered path, for the HEVC test-class sizes, ragged frames, the edge-model families, lists
longer than one launch takes, permuted lists and frames at unaligned offsets of one buffer."""
import ctypes as C
import random
import re

import numpy as np
import pytest

from oracle import oracle
from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, synth

pytestmark = pytest.mark.gpu

CTC = [(240, 416), (480, 832), (720, 1280), (1080, 1920), (1600, 2560)]     # (height, width)
RAGGED = [(33, 61), (7, 121), (1, 1), (300, 5)]
SMALL = [(240, 416)] + RAGGED                                                 # also checked against the CPU oracle


def _frames(seed, hw):
    """(anchor, ori) pairs, one frame of each (height, width), from synth's seeded generator."""
    return [tuple(a[0] for a in synth.make_frames(seed + j, 1, h, w)) for j, (h, w) in enumerate(hw)]


def _mix(seed):
    hw = CTC + RAGGED
    random.Random(seed).shuffle(hw)
    return hw


def _handle(image, h, w, impl=api.IMPL_FUSED, batch=1):
    net = api.QVRCNN(0, batch, 1, h, w)
    net.load_static_para_mem(image)
    net.set_impl(impl)
    return net


def _per_geometry(image, frames, impl=api.IMPL_FUSED):
    """What qv_forward_frames_device / _sse give for every frame on a handle of its own geometry: (outputs, sse [n][2])."""
    import torch
    outs, sse, nets = [], np.zeros((len(frames), 2), np.int64), {}
    for j, (x, ori) in enumerate(frames):
        h, w = x.shape
        if (h, w) not in nets:
            nets[(h, w)] = _handle(image, h, w, impl)
        net = nets[(h, w)]
        d_in, d_ori = torch.from_numpy(x).cuda(), torch.from_numpy(ori).cuda()
        d_out = torch.empty_like(d_in)
        d_sse = torch.zeros(2, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        net.forward_frames_device(d_in.data_ptr(), d_out.data_ptr(), 1)
        plain = d_out.cpu().numpy()
        net.forward_frames_device_sse(d_in.data_ptr(), d_ori.data_ptr(), d_out.data_ptr(), 1, d_sse.data_ptr())
        assert np.array_equal(d_out.cpu().numpy(), plain)
        outs.append(plain)
        sse[j] = d_sse.cpu().numpy()
    for n in nets.values():
        n.close()
    return outs, sse


def _list_run(net, frames, with_sse=False, calls=1, stream=0):
    """One list call (or `calls` of them) over `frames` on device tensors; returns (outputs, sse or None)."""
    import torch
    ins = [torch.from_numpy(x).cuda() for x, _ in frames]
    oris = [torch.from_numpy(o).cuda() for _, o in frames]
    outs = [torch.full_like(t, 7) for t in ins]
    d_sse = torch.zeros((len(frames), 2), dtype=torch.int64, device="cuda") if with_sse else None
    torch.cuda.synchronize()
    desc = [(i, o, r) if with_sse else (i, o) for i, o, r in zip(ins, outs, oris)]
    for _ in range(calls):
        net.forward_frame_list_device(desc, d_sse, stream)
    if stream:
        net.synchronize(stream)
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in outs], (d_sse.cpu().numpy() if with_sse else None)


def _np_sse(a, ori):
    return int(((a.astype(np.int64) - ori.astype(np.int64)) ** 2).sum())


@pytest.fixture(scope="module")
def qp32(models):
    return formats.write_model_vect_c(models[32])


@pytest.fixture(scope="module")
def ctc_case(qp32):
    hw = _mix(0x7157)
    frames = _frames(0x5EED0, hw)
    return hw, frames, _per_geometry(qp32, frames)


def test_ctc_mix_matches_per_geometry_calls(qp32, ctc_case):
    hw, frames, (want, _) = ctc_case
    net = _handle(qp32, 64, 64)                     # the handle's own geometry plays no part
    before = net.launch_count()
    got, _ = _list_run(net, frames)
    assert net.launch_count() - before == 1
    for j, (h, w) in enumerate(hw):
        assert np.array_equal(got[j], want[j]), (h, w)
    ora = oracle.OracleModel(qp32)
    for j, (h, w) in enumerate(hw):
        if (h, w) in SMALL:
            assert np.array_equal(got[j], ora.forward_blu(frames[j][0][None])[0]), (h, w)
    net.close()


def test_sse_pairs_match_and_add_up(qp32, ctc_case):
    hw, frames, (want, want_sse) = ctc_case
    net = _handle(qp32, 16, 16)
    got, sse = _list_run(net, frames, with_sse=True)
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    assert np.array_equal(sse, want_sse)
    for j, (x, ori) in enumerate(frames):
        assert sse[j, 0] == _np_sse(x, ori) and sse[j, 1] == _np_sse(want[j], ori), hw[j]
    _, sse3 = _list_run(net, frames, with_sse=True, calls=3)
    assert np.array_equal(sse3, 3 * want_sse)
    net.close()


def test_layered_path_gives_the_same_bytes(qp32, ctc_case):
    hw, frames, (want, want_sse) = ctc_case
    net = _handle(qp32, 8, 8, api.IMPL_LAYERED)     # scratch for 8 x 8 pixels: the list grows it to 2560 x 1600
    got, sse = _list_run(net, frames, with_sse=True)
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    assert np.array_equal(sse, want_sse)
    got, _ = _list_run(net, frames)
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    # the handle's own geometry still runs after the growth
    x = frames[0][0][None, :8, :8].copy()
    assert np.array_equal(net.forward_frames_host(x), oracle.OracleModel(qp32).forward_blu(x))
    net.close()


def test_longer_than_one_launch(qp32):
    n = api.FRAME_LIST_LAUNCH_MAX + 40
    geoms = [(7, 5), (33, 61), (1, 1), (16, 130)]
    hw = [geoms[j % len(geoms)] for j in range(n)]
    frames = _frames(0xB16, hw)
    want, want_sse = _per_geometry(qp32, frames)
    net = _handle(qp32, 1, 1)
    before = net.launch_count()
    got, sse = _list_run(net, frames, with_sse=True)
    assert net.launch_count() - before == 2
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    assert np.array_equal(sse, want_sse)
    net.close()


def test_permuted_list_gives_every_frame_the_same_output(qp32, ctc_case):
    hw, frames, (want, _) = ctc_case
    perm = list(range(len(frames)))
    random.Random(3).shuffle(perm)
    net = _handle(qp32, 1, 1)
    got, _ = _list_run(net, [frames[p] for p in perm])
    for k, p in enumerate(perm):
        assert np.array_equal(got[k], want[p]), hw[p]
    net.close()


def test_frames_at_unaligned_offsets_of_one_buffer(qp32, ctc_case):
    import torch
    hw, frames, (want, want_sse) = ctc_case
    offs, o = [], 3
    for h, w in hw:
        offs.append(o)
        o += h * w + 5                             # odd gaps: every frame starts at another alignment
    src = torch.zeros(o, dtype=torch.uint8, device="cuda")
    ori = torch.zeros(o, dtype=torch.uint8, device="cuda")
    dst = torch.zeros(o + 1, dtype=torch.uint8, device="cuda")
    descs = (api.FrameDesc * len(hw))()
    for j, ((h, w), (x, r)) in enumerate(zip(hw, frames)):
        src[offs[j]:offs[j] + h * w] = torch.from_numpy(x.ravel()).cuda()
        ori[offs[j]:offs[j] + h * w] = torch.from_numpy(r.ravel()).cuda()
        descs[j] = api.FrameDesc(src.data_ptr() + offs[j], dst.data_ptr() + offs[j] + 1, ori.data_ptr() + offs[j], h, w)
    d_sse = torch.zeros((len(hw), 2), dtype=torch.int64, device="cuda")
    net = _handle(qp32, 1, 1)
    torch.cuda.synchronize()
    assert api.lib().qv_forward_frame_list_device(net._h, descs, len(hw), d_sse.data_ptr(), None) == 0
    out = dst.cpu().numpy()
    for j, (h, w) in enumerate(hw):
        assert np.array_equal(out[offs[j] + 1:offs[j] + 1 + h * w].reshape(h, w), want[j]), (h, w)
    assert np.array_equal(d_sse.cpu().numpy(), want_sse)
    net.close()


def test_async_on_a_torch_stream(qp32, ctc_case):
    import torch
    hw, frames, (want, want_sse) = ctc_case
    net = _handle(qp32, 1, 1)
    st = torch.cuda.Stream()
    got, sse = _list_run(net, frames, with_sse=True, stream=st.cuda_stream)
    assert api.lib().qv_synchronize(net._h, C.c_void_p(st.cuda_stream)) == 0
    assert all(np.array_equal(g, w) for g, w in zip(got, want))
    assert np.array_equal(sse, want_sse)
    net.close()


def test_argument_errors(qp32):
    import torch
    L = api.lib()
    x = torch.zeros((4, 4), dtype=torch.uint8, device="cuda")
    y = torch.zeros_like(x)
    d_sse = torch.zeros((1, 2), dtype=torch.int64, device="cuda")
    net = _handle(qp32, 1, 1)
    good = api.FrameDesc(x.data_ptr(), y.data_ptr(), None, 4, 4)

    def call(descs, n, sse=None, h=net._h):
        arr = (api.FrameDesc * max(1, len(descs)))(*descs) if descs is not None else None
        return L.qv_forward_frame_list_device(h, arr, n, sse, None)

    assert call([good], 1, h=None) == -1
    assert call(None, 1) == -1
    assert call([good], -1) == -1
    assert call([api.FrameDesc(None, y.data_ptr(), None, 4, 4)], 1) == -1
    assert call([api.FrameDesc(x.data_ptr(), None, None, 4, 4)], 1) == -1
    assert call([api.FrameDesc(x.data_ptr(), y.data_ptr(), None, 0, 4)], 1) == -1
    assert call([api.FrameDesc(x.data_ptr(), y.data_ptr(), None, 4, 0)], 1) == -1
    assert call([good], 1, d_sse.data_ptr()) == -1                                       # d_sse without d_ori
    assert call([api.FrameDesc(x.data_ptr(), y.data_ptr(), x.data_ptr(), 4, 4)], 1) == -1  # d_ori without d_sse
    tall = torch.zeros((66052, 1), dtype=torch.uint8, device="cuda")
    tall_out = torch.zeros_like(tall)
    assert call([api.FrameDesc(tall.data_ptr(), tall_out.data_ptr(), tall.data_ptr(), 66052, 1)], 1, d_sse.data_ptr()) == -1
    before = net.launch_count()
    assert call(None, 0) == 0 and call([good], 0) == 0
    assert net.launch_count() == before
    assert call([good], 1) == 0
    # the layered path takes the tall frame with its SSE
    net.set_impl(api.IMPL_LAYERED)
    assert call([api.FrameDesc(tall.data_ptr(), tall_out.data_ptr(), tall.data_ptr(), 66052, 1)], 1, d_sse.data_ptr()) == 0
    net.close()
    empty = api.QVRCNN(0, 1, 1, 4, 4)                                                    # no model loaded
    assert call([good], 1, h=empty._h) == -5
    empty.close()


def test_binding_refuses_tensors_the_kernel_cannot_read(qp32):
    """The Python wrapper passes data_ptr() on as a device address: host tensors, other dtypes and a host d_sse are refused
    before the library is called."""
    import torch
    net = _handle(qp32, 1, 1)
    x = torch.zeros((4, 4), dtype=torch.uint8, device="cuda")
    before = net.launch_count()
    for bad in ([(x.cpu(), torch.empty_like(x))], [(x, torch.empty((4, 4), dtype=torch.uint8))],
                [(x.float(), torch.empty_like(x))], [(x, torch.empty_like(x), x.cpu())]):
        with pytest.raises(ValueError):
            net.forward_frame_list_device(bad, torch.zeros((1, 2), dtype=torch.int64, device="cuda") if len(bad[0]) > 2 else None)
    with pytest.raises(ValueError):
        net.forward_frame_list_device([(x, torch.empty_like(x), x)], torch.zeros((1, 2), dtype=torch.int64))
    assert net.launch_count() == before
    net.close()


def test_activation_taps_after_a_layered_list(qp32, ctc_case):
    """After a layered list the scratch holds a list frame, not the handle's geometry: qv_get_activation refuses until the
    handle's own frames run again."""
    hw, frames, _ = ctc_case
    x = frames[0][0][None, :8, :8].copy()
    net = _handle(qp32, 8, 8, api.IMPL_LAYERED)
    net.forward_frames_host(x)
    a1 = net.get_activation(1)
    _list_run(net, frames[:3])
    with pytest.raises(api.QVError) as e:
        net.get_activation(1)
    assert e.value.code == -5
    net.forward_frames_host(x)
    assert np.array_equal(net.get_activation(1), a1)
    net.close()


def _kernel_builds(prof):
    """(FAST, SSE) of every k_enh_list build the profiler saw launched."""
    seen = set()
    for e in prof.events():
        m = re.search(r"k_enh_list<([^>]*)>", e.name)
        if m:
            seen.add(tuple(int(a.strip() == "true") for a in m.group(1).split(",")))
            continue
        m = re.search(r"k_enh_listI((?:Lb[01]E)+)E", e.name)
        if m:
            seen.add(tuple(int(b) for b in re.findall(r"Lb([01])E", m.group(1))))
    return seen


def test_edge_models_in_one_mixed_list():
    """Every edge-model family (fast and generic requantiser rows) through one mixed list, with and without SSEs, against
    per-geometry calls: all four builds of k_enh_list run."""
    from torch.profiler import ProfilerActivity, profile
    hw = [(33, 131), (1, 1), (7, 5), (61, 250), (20, 160), (2, 241)]
    frames = _frames(0xED6E, hw)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for mid, seed, family, variant in synth.edge_models():
            image = formats.write_model_vect_c(synth.make_edge_model(seed, family, variant))
            want, want_sse = _per_geometry(image, frames)
            net = _handle(image, 1, 1)
            got, _ = _list_run(net, frames)
            assert all(np.array_equal(g, w) for g, w in zip(got, want)), mid
            got, sse = _list_run(net, frames, with_sse=True)
            assert all(np.array_equal(g, w) for g, w in zip(got, want)), mid
            assert np.array_equal(sse, want_sse), mid
            net.close()
    assert _kernel_builds(prof) == {(1, 0), (0, 0), (1, 1), (0, 1)}, _kernel_builds(prof)
