"""The host-built structures of the fused tcgen05 path, checked without a GPU.

`qv_debug_fused_tables` returns what `fused_upload` hands to the kernel: the shared-memory weight image (B operands
as ring block sequences), the per-phase table with both 64-bit descriptors of each of the 27 MMAs of a row iteration,
and the layout / requantiser constants.  This test runs the kernel's DATAFLOW on them in numpy -- the same three roles
in the same order, shared memory as a byte array, TMEM as a [128 lanes][512 columns] int32 array that starts as
garbage, every MMA executed from its descriptors (no-swizzle K-major: 8-row x 16-byte core matrices, SBO = 128 B,
LBO from the descriptor) -- and compares the reconstructed frame and the activations with the CPU oracle.  A wrong
block sequence, ring rotation, descriptor, zero block or bias offset fails here, on the CPU.

The arithmetic of the roles is restated from qv_fused.cu (k_fused: workers, C4 warps); it is the tables that are under
test, so every address the emulation uses comes from the tables or from the constants the library reports."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle
from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, synth

NAMES = ["WIMG_BYTES", "SMEM_BYTES", "OFF_A1", "OFF_A2", "OFF_IM", "OFF_ZERO", "OFF_IN", "OFF_A3", "PW", "PLANE", "A1_ROW",
         "A2_ROW", "IM_BYTES", "IN_SLOTS", "IN_PITCH", "WT", "PIPE", "TM_D1", "TM_R22", "TM_R21", "TM_R31", "TM_D32", "N_PHASE",
         "N_MMA", "fast", "c4_bias", "c4_mul", "c4_shift"]


def fused_tables(model_bytes):
    L = api.lib()
    L.qv_debug_fused_tables.argtypes = [C.c_char_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_size_t)]
    L.qv_debug_fused_tables.restype = C.c_int
    sizes = (C.c_size_t * 3)(0, 0, 0)
    assert L.qv_debug_fused_tables(model_bytes, len(model_bytes), None, None, None, sizes) == 0
    wimg = np.zeros(sizes[0], np.uint8)
    ops = np.zeros(sizes[1], np.uint32)
    consts = np.zeros(sizes[2], np.int32)
    assert L.qv_debug_fused_tables(model_bytes, len(model_bytes), wimg.ctypes.data, ops.ctypes.data, consts.ctypes.data, sizes) == 0
    k = dict(zip(NAMES, consts[:len(NAMES)].tolist()))
    p = len(NAMES)
    groups = consts[p:p + 30].reshape(5, 6)            # q1, q22, q21, q31, q32 : hi, M, blu, mul, shift, rbias
    bias = consts[p + 30:p + 190]
    c4w = consts[p + 190:p + 298]
    assert len(consts) == p + 298
    per = k["N_MMA"] * 4 + 8
    ops = ops.reshape(k["N_PHASE"], per)
    return k, wimg, ops, groups, bias, c4w


class Emu:
    """One work unit (frame, strip 0, the whole height) of k_fused, sequentially."""

    def __init__(self, model_bytes, rng):
        self.k, wimg, self.ops, self.groups, self.bias, c4w = fused_tables(model_bytes)
        k = self.k
        self.sm = np.zeros(k["SMEM_BYTES"], np.uint8)
        self.sm[:k["WIMG_BYTES"]] = wimg
        self.tmem = rng.integers(-2**31, 2**31 - 1, size=(128, 512), dtype=np.int64).astype(np.int32)     # never initialised
        self.c4w = c4w.astype(np.int32).view(np.int8).reshape(3, 3, 3, 16)       # [dy][dx][plane][channel in plane]

    # ---- tensor core -------------------------------------------------------------------------------
    def operand(self, lo, hi, rows):
        assert hi == ((128 >> 4) | (1 << 14)), hex(hi)                           # SBO = 128 B, descriptor version 1
        start, lbo = (int(lo) & 0x3FFF) * 16, ((int(lo) >> 16) & 0x3FFF) * 16
        r = np.arange(rows)[:, None]
        kk = np.arange(32)[None, :]
        addr = start + (kk // 16) * lbo + (r // 8) * 128 + (r % 8) * 16 + (kk % 16)
        assert addr.max() < self.sm.size
        return self.sm[addr].view(np.int8).astype(np.int32)

    def mma(self, d, ab, n, acc):
        a = self.operand(ab[0], ab[1], 128)
        b = self.operand(ab[2], ab[3], n)
        prod = a @ b.T
        assert d + n <= 512
        self.tmem[:, d:d + n] = (self.tmem[:, d:d + n] if acc else 0) + prod

    def issue(self, ph):
        k, o = self.k, self.ops[ph]
        ab = o[:k["N_MMA"] * 4].reshape(k["N_MMA"], 4)
        d1, d32, z22, z21, z31 = (int(x) for x in o[k["N_MMA"] * 4:k["N_MMA"] * 4 + 5])
        r22, r21, r31 = k["TM_R22"], k["TM_R21"], k["TM_R31"]
        seq = [(d1, 64, 0), (z22, 16, 0), (z21, 32, 0), (z31, 16, 0), (r31, 64, 1), (r31, 64, 1), (d32, 32, 0), (r31, 64, 1),
               (r31, 64, 1), (d32, 32, 1), (r31, 64, 1)]
        for t in range(10):
            seq.append((r22, 96, 1))
            if 1 <= t // 2 <= 3:
                seq.append((r21, 128, 1))
        assert len(seq) == k["N_MMA"]
        for (d, n, acc), row in zip(seq, ab):
            self.mma(d, row, n, acc)

    # ---- workers: TMEM -> requantise -> activation rows ---------------------------------------------------
    def requant_store(self, col, boff, g, valid, dst):
        hi, M, blu, mul, shift, rbias = (int(v) for v in self.groups[g])
        acc = self.tmem[:, col:col + 16].astype(np.int64) + self.bias[boff:boff + 16].astype(np.int64)[None, :]
        if self.k["fast"]:
            # bias' = b + rbias: t = clamp(acc + bias', 0, blu + rbias), q = byte 3 of t * (mul << (24 - shift))
            q = ((np.clip(acc, 0, hi) * (M & 0xFFFFFFFF)) >> 24) & 0xFF
        else:
            # the reference formula on u = acc + b (mat.cu:286-291): int32 product, arithmetic shift, (char) store
            p = ((acc + rbias) * mul) & 0xFFFFFFFF
            p = np.where(p >= 1 << 31, p - (1 << 32), p)
            q = np.where(acc > blu, 127, np.where(acc < 0, 0, (p >> shift) & 0xFF))
        q = np.where(valid[:, None], q, 0).astype(np.uint8)
        m = np.arange(128)
        self.sm[dst + m[:, None] * 16 + np.arange(16)[None, :]] = q

    def drain(self, R1, H, W, X0=0):
        k = self.k
        m = np.arange(128)
        ok = lambda r: 0 <= r < H
        xa1 = (X0 - 4 + m >= 0) & (X0 - 4 + m < W)
        xa2 = (X0 - 2 + m >= 0) & (X0 - 2 + m < W)
        xa3 = (X0 - 1 + m >= 0) & (X0 - 1 + m < W)
        par = (R1 - 1) & 1
        PL = k["PLANE"]
        d1 = k["TM_D1"] + par * 64
        dst1 = k["OFF_A1"] + ((R1 - 1) % 3) * k["A1_ROW"] + 4 * 16
        for pl in range(4):
            self.requant_store(d1 + 16 * pl, 16 * pl, 0, xa1 & ok(R1 - 1), dst1 + pl * PL)
        dst2 = k["OFF_A2"] + ((R1 - 5) % 3) * k["A2_ROW"] + 6 * 16
        dst2n = k["OFF_A2"] + ((R1 - 4) % 3) * k["A2_ROW"] + 6 * 16
        self.requant_store(k["TM_R22"] + ((R1 - 5) % 6) * 16, 64, 1, xa2 & ok(R1 - 5), dst2 + 2 * PL)
        r21 = k["TM_R21"] + ((R1 - 4) & 3) * 32
        self.requant_store(r21, 80, 2, xa2 & ok(R1 - 4), dst2n)
        self.requant_store(r21 + 16, 96, 2, xa2 & ok(R1 - 4), dst2n + PL)
        self.requant_store(k["TM_R31"] + ((R1 - 8) & 3) * 16, 112, 3, xa3 & ok(R1 - 8), k["OFF_A3"] + ((R1 - 8) % 3) * k["A2_ROW"] + 7 * 16)
        d32 = k["TM_D32"] + par * 32
        dst3n = k["OFF_A3"] + ((R1 - 7) % 3) * k["A2_ROW"] + 7 * 16
        self.requant_store(d32, 128, 4, xa3 & ok(R1 - 7), dst3n + PL)
        self.requant_store(d32 + 16, 144, 4, xa3 & ok(R1 - 7), dst3n + 2 * PL)

    # ---- C4 warps: input ring, C1 operand, output layer ------------------------------------------------------
    def store_in(self, img, row, X0=0):
        k = self.k
        H, W = img.shape
        p = np.arange(k["PW"])
        col = X0 - 8 + p
        v = np.full(k["PW"], 128, np.uint8)
        if 0 <= row < H:
            okc = (col >= 0) & (col < W)
            v[okc] = img[row, col[okc]]
        base = k["OFF_IN"] + (row % k["IN_SLOTS"]) * k["IN_PITCH"]
        self.sm[base:base + k["PW"]] = v

    def in_row(self, row):
        k = self.k
        base = k["OFF_IN"] + (row % k["IN_SLOTS"]) * k["IN_PITCH"]
        return self.sm[base:base + k["IN_PITCH"]]

    def im2col(self, R, stage):
        k = self.k
        out = np.zeros((128, 32), np.uint8)
        m = np.arange(128)
        for r in range(5):
            row = self.in_row(R - 2 + r)
            for s in range(5):
                kk = 4 * r + s if s < 4 else 20 + r
                out[:, kk] = row[m + 2 + s] ^ 0x80
        dst = k["OFF_IM"] + stage * k["IM_BYTES"]
        self.sm[dst + m[:, None] * 16 + np.arange(16)[None, :]] = out[:, :16]
        self.sm[dst + 128 * 16 + m[:, None] * 16 + np.arange(16)[None, :]] = out[:, 16:]

    def c4(self, R1, state, out, y0, y1, W, X0=0):
        k = self.k
        mo = np.arange(128)
        row = k["OFF_A3"] + (R1 % 3) * k["A2_ROW"]
        acc = np.zeros((3, 128), np.int64)
        for dx in range(3):
            for pl in range(3):
                a = self.sm[row + pl * k["PLANE"] + (7 + mo[:, None] + dx) * 16 + np.arange(16)[None, :]].view(np.int8).astype(np.int64)
                for dy in range(3):
                    acc[dy] += a @ self.c4w[dy, dx, pl].astype(np.int64)
        u4 = state[1] + acc[2]
        state[1] = state[0] + acc[1]
        state[0] = acc[0]
        rowo = R1 - 10
        if y0 <= rowo < y1:
            x = self.in_row(rowo)[8 + mo].astype(np.int64)
            t = (((u4 + k["c4_bias"]) * k["c4_mul"] + (1 << (k["c4_shift"] - 1))) & 0xFFFFFFFF).astype(np.uint32).view(np.int32) >> k["c4_shift"]
            r = (x + t).astype(np.int16).astype(np.int64)
            okc = (mo < k["WT"]) & (X0 + mo < W)
            out[rowo, X0 + mo[okc]] = np.clip(r, 0, 255)[okc]

    # ---- the unit --------------------------------------------------------------------------------------------
    def run(self, img, taps=None):
        k = self.k
        H, W = img.shape
        assert W <= k["WT"]
        y0, y1 = 0, H
        niter = y1 - y0 + k["PIPE"]
        out = np.zeros_like(img)
        for r in range(y0 - 6, y0):
            self.store_in(img, r)
        self.im2col(y0 - 4, (y0 - 4) % 3)
        state = [np.zeros(128, np.int64), np.zeros(128, np.int64)]
        for i in range(niter):
            R1 = y0 - 4 + i
            if i >= 1:
                self.drain(R1, H, W)
                if taps is not None:
                    taps(self, R1)
            # C4 warps: C1 operand of the next row (its last input row arrived at the end of the previous iteration)
            if i + 1 < niter:
                self.im2col(R1 + 1, (R1 + 1) % 3)
            if i >= 3:
                self.c4(R1, state, out, y0, y1, W)
            self.store_in(img, R1 + 4)
            self.issue(R1 % k["N_PHASE"])
        return out


def plane_rows(emu, off, row_bytes, R, first_px, nplanes, W):
    """Channels-last view [W][16*nplanes] of activation row R in its 3-slot ring."""
    k = emu.k
    base = off + (R % 3) * row_bytes + first_px * 16
    px = np.arange(W)
    return np.concatenate([emu.sm[base + pl * k["PLANE"] + px[:, None] * 16 + np.arange(16)[None, :]] for pl in range(nplanes)], axis=1)


EDGE = {e[0]: e[1:] for e in synth.edge_models()}
CASES = [(32, 19, 37), (22, 12, 120), (37, 33, 8)] + [(mid, 17, 61) for mid in EDGE]


def _case_model(qp):
    if qp in EDGE:
        return synth.make_edge_model(*EDGE[qp])
    return synth.make_model(0xC0FFEE + qp, qp)


@pytest.mark.parametrize("qp,H,W", CASES)
def test_kernel_dataflow_on_host_tables_matches_oracle(qp, H, W):
    """qp: a calibrated model of that QP, or an edge model (synth.make_edge_model) by its id -- the generic families run the
    reference-formula requantiser, with the biases the host wrote for it."""
    rng = np.random.default_rng(1234 + (qp if isinstance(qp, int) else len(qp)))
    model = _case_model(qp)
    mb = formats.write_model_vect_c(model)
    img = synth.make_uniform_frames(0xBEEF + (qp if isinstance(qp, int) else H), 1, H, W)[0]
    rec, a1, a2, a3, _ = oracle.OracleModel(mb).forward_taps(img)
    emu = Emu(mb, rng)
    seen = {"a1": 0, "a2": 0, "a3": 0}

    def taps(e, R1):
        k = e.k
        # rows complete after this drain: a1 row R1-1, a2 row R1-5 (plane 2 arrived last), a3 row R1-8 (plane 0 arrived last)
        for name, ref, off, rb, first, npl, R in (("a1", a1, k["OFF_A1"], k["A1_ROW"], 8, 4, R1 - 1), ("a2", a2, k["OFF_A2"], k["A2_ROW"], 8, 3, R1 - 5),
                                                  ("a3", a3, k["OFF_A3"], k["A2_ROW"], 8, 3, R1 - 8)):
            if 0 <= R < H:
                got = plane_rows(e, off, rb, R, first, npl, W).view(np.int8)
                np.testing.assert_array_equal(got, ref[:, R, :].T, err_msg="%s row %d" % (name, R))
                seen[name] += 1

    out = emu.run(img, taps)
    assert seen == {"a1": H, "a2": H, "a3": H}
    np.testing.assert_array_equal(out, rec)


@pytest.mark.parametrize("mid", [e[0] for e in synth.edge_models()])
def test_fast_flag_is_all_or_nothing(mid):
    """qv_debug_fused_tables reports fast == 1 exactly when all five hidden rows pass the fast requantiser's precondition;
    one failing row sends the whole model to the generic kernels.  The fast path folds rbias into the biases it writes,
    the generic path writes the layer biases as they are."""
    model = synth.make_edge_model(*EDGE[mid])
    k, _, _, groups, bias, _ = fused_tables(formats.write_model_vect_c(model))
    want = all(synth.fast_row_ok(*q) for q in model.qparams[:5])
    assert k["fast"] == int(want)
    layer_of_group = (0, 2, 1, 3, 4)                   # q1, q22, q21, q31, q32 -> C1, C2_2, C2_1, C3_1, C3_2
    offsets = (0, 64, 80, 112, 128)
    for g, l in enumerate(layer_of_group):
        blu, mul, shift = model.qparams[l]
        rb = (1 << (shift - 1)) // mul
        assert groups[g][2:].tolist() == [blu, mul, shift, rb]
        b = model.b[l].astype(np.int64) + (rb if want else 0)
        assert bias[offsets[g]:offsets[g] + len(b)].tolist() == b.tolist(), l
