"""ctypes binding of the C ABI (include/qvrcnn_b200.h) with the reference's object names.

`QVRCNN` mirrors class qvrcnn (inference/qvrcnn.cuh:25-59): same constructor arguments, same
method names (`load_static_para`, `load_data`, `forward_blu`) and the same error behaviour
translated to Python (the reference prints and exit(1)s; here a `QVError` is raised).
`VRCNNData` mirrors class vrcnn_data (inference/yuv_data.h:11-27).

There is NO CPU fallback and nothing here touches oracle/: if libqvrcnn_b200.so is missing the
import of the library fails loudly, and without a CUDA device `QVRCNN(...)` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("QVRCNN_B200_LIB", os.path.join(_PKG, "libqvrcnn_b200.so"))   # override: A/B builds only

IMPL_AUTO, IMPL_LAYERED, IMPL_FUSED = 0, 1, 2

# Every symbol include/qvrcnn_b200.h declares (tests check the built library exports them all).
ABI_SYMBOLS = (
    "qv_last_error", "qv_version", "qv_create", "qv_destroy", "qv_load_static_para",
    "qv_load_static_para_mem", "qv_load_static_para_hwcn", "qv_load_quant_params", "qv_read_quant_params",
    "qv_set_weights", "qv_get_quant_params", "qv_load_data", "qv_forward_blu", "qv_get_recon",
    "qv_forward_frames_host", "qv_stream_yuv", "qv_stream_yuv_pf", "qv_forward_frames_device", "qv_forward_frames_device_sse", "qv_forward_rows_device", "qv_device_buffers",
    "qv_sse_device", "qv_host_alloc", "qv_host_free",
    "qv_set_impl", "qv_get_impl", "qv_launch_count", "qv_get_activation",
    "qv_convert_model_hwcn_to_vect_c", "qv_yuv_read_luma", "qv_yuv_read_frame", "qv_yuv_write_recon",
    "qv_psnr", "qv_psnr_from_sse", "qv_solve_quant_params", "qv_write_quant_params_cpp", "qv_quantize_layer",
    "qv_debug_fused_tables", "qv_debug_fused_units", "qv_synchronize",
    "qv_strip_setup", "qv_strip_export", "qv_strip_attach", "qv_strip_input", "qv_strip_acquire", "qv_strip_load",
    "qv_strip_forward", "qv_strip_forward_sse", "qv_strip_stream_yuv_pf", "qv_strip_release",
)

CUDA_STREAM_LEGACY = 1      # cudaStreamLegacy: names the legacy default stream explicitly (NULL = "the handle's own stream")
STRIP_ABOVE, STRIP_BELOW = 0, 1
STRIP_DESC_BYTES = 192


def stream_arg(stream: int):
    """A cudaStream_t for the ABI from a torch `cuda_stream` integer: torch reports the legacy default stream as 0, which
    the ABI reads as "use the handle's private stream, synchronously" -- name it explicitly instead."""
    return CUDA_STREAM_LEGACY if not stream else stream


class QVError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("qvrcnn_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    """Loads libqvrcnn_b200.so (built by __graft_entry__.build() / `make -C qcnn_gpu_b200/csrc`)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no fallback implementation)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, i32, cp = C.c_void_p, C.c_int, C.c_char_p
        L.qv_last_error.restype = cp
        L.qv_version.restype = cp
        L.qv_create.argtypes = [i32, i32, i32, i32, i32, C.POINTER(vp)]
        L.qv_destroy.argtypes = [vp]
        L.qv_load_static_para.argtypes = [vp, cp]
        L.qv_load_static_para_mem.argtypes = [vp, vp, C.c_size_t]
        L.qv_load_static_para_hwcn.argtypes = [vp, cp]
        L.qv_load_quant_params.argtypes = [vp, cp]
        L.qv_read_quant_params.argtypes = [cp, vp]
        L.qv_set_weights.argtypes = [vp, i32, vp, vp]
        L.qv_get_quant_params.argtypes = [vp, vp]
        L.qv_load_data.argtypes = [vp, vp]
        L.qv_forward_blu.argtypes = [vp]
        L.qv_get_recon.argtypes = [vp, vp]
        L.qv_forward_frames_host.argtypes = [vp, vp, vp, i32]
        L.qv_forward_frames_device.argtypes = [vp, vp, vp, i32, vp]
        L.qv_forward_frames_device_sse.argtypes = [vp, vp, vp, vp, i32, vp, vp]
        L.qv_host_alloc.argtypes = [C.c_size_t]
        L.qv_host_alloc.restype = vp
        L.qv_host_free.argtypes = [vp]
        L.qv_host_free.restype = None
        L.qv_stream_yuv.argtypes = [vp, cp, cp, cp, i32, i32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.qv_stream_yuv_pf.argtypes = [vp, cp, cp, cp, i32, i32, vp, vp]
        L.qv_forward_rows_device.argtypes = [vp, vp, i32, i32, i32, vp, i32, i32, vp]
        L.qv_sse_device.argtypes = [vp, vp, C.c_size_t, vp, vp]
        L.qv_set_impl.argtypes = [vp, i32]
        L.qv_get_impl.argtypes = [vp]
        L.qv_launch_count.argtypes = [vp]
        L.qv_launch_count.restype = C.c_longlong
        L.qv_get_activation.argtypes = [vp, i32, vp]
        L.qv_convert_model_hwcn_to_vect_c.argtypes = [cp, cp]
        L.qv_yuv_read_luma.argtypes = [cp, i32, i32, i32, vp]
        L.qv_yuv_read_frame.argtypes = [cp, i32, i32, i32, vp]
        L.qv_yuv_write_recon.argtypes = [cp, vp, i32, i32, i32]
        L.qv_psnr.argtypes = [vp, vp, C.c_size_t, C.POINTER(C.c_int64)]
        L.qv_psnr.restype = C.c_double
        L.qv_psnr_from_sse.argtypes = [C.c_int64, C.c_size_t]
        L.qv_psnr_from_sse.restype = C.c_double
        L.qv_solve_quant_params.argtypes = [vp, vp, vp]
        L.qv_write_quant_params_cpp.argtypes = [cp, vp]
        L.qv_quantize_layer.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_double, C.c_double, vp, vp]
        L.qv_synchronize.argtypes = [vp, vp]
        L.qv_strip_setup.argtypes = [vp, i32, i32, i32]
        L.qv_strip_export.argtypes = [vp, vp]
        L.qv_strip_attach.argtypes = [vp, i32, vp]
        L.qv_strip_input.argtypes = [vp, i32, C.POINTER(vp)]
        L.qv_strip_acquire.argtypes = [vp, i32, vp]
        L.qv_strip_load.argtypes = [vp, i32, vp, vp]
        L.qv_strip_forward.argtypes = [vp, i32, vp, vp]
        L.qv_strip_forward_sse.argtypes = [vp, i32, vp, vp, vp, vp]
        L.qv_strip_stream_yuv_pf.argtypes = [C.POINTER(vp), i32, cp, cp, cp, i32, i32, vp, vp]
        L.qv_strip_release.argtypes = [vp]
        _lib = L
    return _lib


def _check(rc: int) -> None:
    if rc != 0:
        raise QVError(rc, lib().qv_last_error().decode("utf-8", "replace"))


def _b(path) -> bytes:
    return os.fsencode(path)


class QVRCNN:
    """qvrcnn(gpu_num, batch, channel, height, width) -- inference/qvrcnn.cu:4-29."""

    def __init__(self, gpu_num: int, batch: int, channel: int, height: int, width: int):
        self._h = C.c_void_p()
        self.batch, self.channel, self.height, self.width = batch, channel, height, width
        _check(lib().qv_create(gpu_num, batch, channel, height, width, C.byref(self._h)))

    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            lib().qv_destroy(self._h)
            self._h = C.c_void_p()

    __del__ = close

    # -- model ---------------------------------------------------------------------------
    def load_static_para(self, filename) -> int:                     # inference/qvrcnn.cu:47-63
        _check(lib().qv_load_static_para(self._h, _b(filename)))
        return 0

    def load_static_para_mem(self, image: bytes) -> int:
        _check(lib().qv_load_static_para_mem(self._h, image, len(image)))
        return 0

    def load_static_para_hwcn(self, filename) -> int:
        _check(lib().qv_load_static_para_hwcn(self._h, _b(filename)))
        return 0

    def load_quant_params(self, filename) -> int:
        _check(lib().qv_load_quant_params(self._h, _b(filename)))
        return 0

    def set_weights(self, layer: int, w_kcrs: np.ndarray, bias: np.ndarray) -> int:
        w = np.ascontiguousarray(w_kcrs, np.int8)
        b = np.ascontiguousarray(bias, np.int32)
        _check(lib().qv_set_weights(self._h, layer, w.ctypes.data, b.ctypes.data))
        return 0

    def quant_params(self) -> np.ndarray:
        q = np.zeros(18, np.int32)
        _check(lib().qv_get_quant_params(self._h, q.ctypes.data))
        return q.reshape(6, 3)

    # -- the reference's per-frame surface ------------------------------------------------
    def load_data(self, input_u8: np.ndarray) -> int:                # inference/qvrcnn.cu:64-68
        x = np.ascontiguousarray(input_u8, np.uint8)
        assert x.size == self.batch * self.height * self.width, x.shape
        _check(lib().qv_load_data(self._h, x.ctypes.data))
        return 0

    def forward_blu(self) -> int:                                    # inference/qvrcnn.cu:168-242
        _check(lib().qv_forward_blu(self._h))
        return 0

    def get_recon(self) -> np.ndarray:                               # kernel.cu:96 (I1.x_rec D2H)
        out = np.empty((self.batch, self.height, self.width), np.uint8)
        _check(lib().qv_get_recon(self._h, out.ctypes.data))
        return out

    # -- batched variants ------------------------------------------------------------------
    def forward_frames_host(self, frames_u8: np.ndarray, out: Optional[np.ndarray] = None) -> np.ndarray:
        x = np.ascontiguousarray(frames_u8, np.uint8)
        n = x.size // (self.height * self.width)
        if out is None:
            out = np.empty_like(x)
        _check(lib().qv_forward_frames_host(self._h, x.ctypes.data, out.ctypes.data, n))
        return out

    def stream_yuv(self, anchor_yuv: str, ori_yuv: Optional[str], recon_yuv: Optional[str], first_frame: int, n_frames: int):
        """Files in, file out, overlapped (qv_stream_yuv); returns (sse_before, sse_after) -- zeros without `ori_yuv`."""
        b, a = C.c_int64(0), C.c_int64(0)
        enc = lambda p: p.encode() if p else None
        _check(lib().qv_stream_yuv(self._h, enc(anchor_yuv), enc(ori_yuv), enc(recon_yuv), first_frame, n_frames,
                                   C.byref(b) if ori_yuv else None, C.byref(a) if ori_yuv else None))
        return int(b.value), int(a.value)

    def stream_yuv_pf(self, anchor_yuv: str, ori_yuv: str, recon_yuv: Optional[str], first_frame: int, n_frames: int):
        """qv_stream_yuv_pf: returns (sse_before, sse_after), two np.int64 arrays of n_frames -- the per-frame SSEs of the
        anchor and of the reconstruction against the original (vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112)."""
        before = np.zeros(max(n_frames, 0), np.int64)
        after = np.zeros(max(n_frames, 0), np.int64)
        enc = lambda p: os.fsencode(p) if p else None
        _check(lib().qv_stream_yuv_pf(self._h, enc(anchor_yuv), enc(ori_yuv), enc(recon_yuv), first_frame, n_frames,
                                      before.ctypes.data, after.ctypes.data))
        return before, after

    def forward_frames_host_ptr(self, in_ptr: int, out_ptr: int, n: int) -> None:
        _check(lib().qv_forward_frames_host(self._h, in_ptr, out_ptr, n))

    def forward_frames_device(self, d_in: int, d_out: int, n: int, stream: int = 0) -> None:
        _check(lib().qv_forward_frames_device(self._h, d_in, d_out, n, stream or None))

    def forward_frames_device_sse(self, d_in: int, d_ori: int, d_out: int, n: int, d_sse: int, stream: int = 0) -> None:
        """forward_frames_device, and per frame f the SSEs of the input / the output against d_ori ADDED to the device int64
        pair d_sse[2f], d_sse[2f + 1]."""
        _check(lib().qv_forward_frames_device_sse(self._h, d_in, d_ori, d_out, n, d_sse, stream or None))

    def forward_rows_device(self, d_in: int, img_height: int, in_row0: int, in_rows: int, d_out: int,
                            out_row0: int, out_row1: int, stream: int = 0) -> None:
        _check(lib().qv_forward_rows_device(self._h, d_in, img_height, in_row0, in_rows, d_out, out_row0,
                                            out_row1, stream or None))

    def synchronize(self, stream: int = 0) -> None:
        """Synchronises the stream (0 = the handle's own) and raises if a kernel on it reported a failure."""
        _check(lib().qv_synchronize(self._h, stream or None))

    # -- one frame over several GPUs: strips with peer-mapped halo rows (qv_strip_*) -----------
    def strip_setup(self, img_height: int, row0: int, row1: int) -> None:
        _check(lib().qv_strip_setup(self._h, img_height, row0, row1))
        self._strip_bytes = (row1 - row0) * self.width

    def strip_export(self) -> bytes:
        buf = C.create_string_buffer(STRIP_DESC_BYTES)
        _check(lib().qv_strip_export(self._h, buf))
        return buf.raw

    def strip_attach(self, side: int, desc: bytes) -> None:
        assert len(desc) == STRIP_DESC_BYTES
        _check(lib().qv_strip_attach(self._h, side, C.create_string_buffer(desc, STRIP_DESC_BYTES)))

    def strip_input(self, slot: int) -> int:
        p = C.c_void_p()
        _check(lib().qv_strip_input(self._h, slot, C.byref(p)))
        return int(p.value)

    def strip_acquire(self, slot: int, stream: int = 0) -> None:
        _check(lib().qv_strip_acquire(self._h, slot, stream or None))

    def strip_load(self, slot: int, rows_u8: np.ndarray, stream: int = 0) -> None:
        x = np.ascontiguousarray(rows_u8, np.uint8)
        assert x.size == getattr(self, "_strip_bytes", -1), "strip_load: expected the %d bytes of this handle's rows, got %d" % (getattr(self, "_strip_bytes", -1), x.size)
        _check(lib().qv_strip_load(self._h, slot, x.ctypes.data, stream or None))

    def strip_forward(self, slot: int, d_out: int, stream: int = 0) -> None:
        _check(lib().qv_strip_forward(self._h, slot, d_out, stream or None))

    def strip_forward_sse(self, slot: int, d_ori_rows: int, d_out: int, d_sse2: int, stream: int = 0) -> None:
        """strip_forward, and the SSEs of this handle's rows (anchor, reconstruction against d_ori_rows) ADDED to the device
        int64 pair d_sse2[0], d_sse2[1]; the strips' values add up to the frame's."""
        _check(lib().qv_strip_forward_sse(self._h, slot, d_ori_rows, d_out, d_sse2, stream or None))

    def strip_release(self) -> None:
        _check(lib().qv_strip_release(self._h))

    # -- controls ---------------------------------------------------------------------------
    def set_impl(self, impl: int) -> None:
        _check(lib().qv_set_impl(self._h, impl))

    def get_impl(self) -> int:
        return lib().qv_get_impl(self._h)

    def launch_count(self) -> int:
        return int(lib().qv_launch_count(self._h))

    def get_activation(self, which: int) -> np.ndarray:
        out = np.empty((64 if which == 1 else 48, self.height, self.width), np.int8)
        _check(lib().qv_get_activation(self._h, which, out.ctypes.data))
        return out


def strip_stream_yuv_pf(nets, anchor_yuv: str, ori_yuv: Optional[str], recon_yuv: Optional[str], first_frame: int, n_frames: int):
    """qv_strip_stream_yuv_pf: frames [first_frame, first_frame + n_frames) of the anchor file through the strip handles `nets`
    (QVRCNN objects after strip_setup / strip_export / strip_attach), each reading and writing only its own rows.  Returns
    (sse_before, sse_after), two np.int64 arrays of n_frames: the SSEs over these handles' rows of each frame (zeros without
    `ori_yuv`)."""
    before = np.zeros(max(n_frames, 0), np.int64)
    after = np.zeros(max(n_frames, 0), np.int64)
    handles = (C.c_void_p * len(nets))(*[n._h.value for n in nets])
    enc = lambda p: os.fsencode(p) if p else None
    _check(lib().qv_strip_stream_yuv_pf(handles, len(nets), enc(anchor_yuv), enc(ori_yuv), enc(recon_yuv), first_frame, n_frames,
                                        before.ctypes.data if ori_yuv else None, after.ctypes.data if ori_yuv else None))
    return before, after


def sse_device(d_a: int, d_b: int, n: int, d_accum: int, stream: int = 0) -> None:
    _check(lib().qv_sse_device(d_a, d_b, n, d_accum, stream or None))


def read_quant_params(filename) -> np.ndarray:
    q = np.zeros(18, np.int32)
    _check(lib().qv_read_quant_params(_b(filename), q.ctypes.data))
    return q.reshape(6, 3)


def convert_model_hwcn_to_vect_c(file_in, file_out) -> None:
    _check(lib().qv_convert_model_hwcn_to_vect_c(_b(file_in), _b(file_out)))


def solve_quant_params(stepw_in, blu_in) -> np.ndarray:
    """adjust_quant (training/quantization.py:55-64): -> rows [6][6] = [stepw, ratio, blu_adj, blu_q, mul, shift]."""
    a = np.ascontiguousarray(stepw_in, np.float64)
    b = np.ascontiguousarray(blu_in, np.float64)
    assert a.size == 6 and b.size == 6
    out = np.zeros(36, np.float64)
    _check(lib().qv_solve_quant_params(a.ctypes.data, b.ctypes.data, out.ctypes.data))
    return out.reshape(6, 6)


def write_quant_params_cpp(filename, rows) -> None:
    r = np.ascontiguousarray(rows, np.float64)
    assert r.size == 36
    _check(lib().qv_write_quant_params_cpp(_b(filename), r.ctypes.data))


def quantize_layer(w: np.ndarray, b: np.ndarray, stepw: float, ratio: float):
    """float [K,C,R,S] weights + [K] biases -> (int8 weights, int32 biases) as the inference path loads them."""
    wf = np.ascontiguousarray(w, np.float32)
    bf = np.ascontiguousarray(b, np.float32)
    wq = np.empty(wf.shape, np.int8)
    bq = np.empty(bf.shape, np.int32)
    _check(lib().qv_quantize_layer(wf.ctypes.data, wf.size, bf.ctypes.data, bf.size, float(stepw), float(ratio), wq.ctypes.data, bq.ctypes.data))
    return wq, bq


def psnr_from_sse(sse: int, n: int) -> float:
    return float(lib().qv_psnr_from_sse(sse, n))


class VRCNNData:
    """vrcnn_data(frame, height, width) -- inference/yuv_data.cpp:3-14: host buffers ori / input /
    recon of frame*h*w bytes each."""

    def __init__(self, frame: int, height: int, width: int):
        self.frame, self.h, self.w = frame, height, width
        self.nSize = frame * height * width
        self.ori = np.zeros((frame, height, width), np.uint8)
        self.input = np.zeros((frame, height, width), np.uint8)
        self.recon = np.zeros((frame, height, width), np.uint8)

    def read_data(self, orifile, inputfile) -> int:                  # inference/yuv_data.cpp:15-42
        _check(lib().qv_yuv_read_luma(_b(orifile), self.frame, self.h, self.w, self.ori.ctypes.data))
        _check(lib().qv_yuv_read_luma(_b(inputfile), self.frame, self.h, self.w, self.input.ctypes.data))
        return 0

    def read_frame(self, orifile, inputfile, n: int) -> int:         # inference/yuv_data.cpp:44-66
        self.frame = 1
        _check(lib().qv_yuv_read_frame(_b(orifile), n, self.h, self.w, self.ori.ctypes.data))
        _check(lib().qv_yuv_read_frame(_b(inputfile), n, self.h, self.w, self.input.ctypes.data))
        return 0

    def psnr(self, data: np.ndarray) -> float:                       # inference/yuv_data.cpp:87-97
        d = np.ascontiguousarray(data, np.uint8)
        return float(lib().qv_psnr(d.ctypes.data, self.ori.ctypes.data, self.nSize, None))

    def save_recon_as(self, filename) -> int:                        # inference/yuv_data.cpp:113-128
        _check(lib().qv_yuv_write_recon(_b(filename), self.recon.ctypes.data, self.frame, self.h, self.w))
        return 0
