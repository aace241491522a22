"""Parity where a CTA of the fused kernel runs several work units, for every whole-frame build and every edge model.

The fused kernel is persistent: CTA b runs units b, b + grid, b + 2 grid, ...  Some of its state starts afresh with each
unit (ring phases, the input-ring and TMA prologues, the per-unit SSE flush); the rest carries over from the previous unit
(mbarrier phase counters, the named-barrier rotation, TMEM and shared-memory rings holding the previous unit's data, the
TMA ring's barrier parity).  A fault in that handover shows only once a CTA takes a second unit.  The shapes below are
chosen so that the plan, read back through the kernel's own unit_geo (qv_debug_fused_units), has that property:

  A  equal row segments and more units than CTAs: some CTAs take a second unit round-robin (narrow last column)
  B  the row line (P.linear): one CTA's pieces cover three or more columns of two or more frames, and the line's columns
     are permuted (perm_q / perm_s0 / perm_r), so CTA b does not start at column b of the line
  C  the row line with tall units (4 x the input ring's rows and more); the costliest shape for the oracle, so for
     the generic-requantiser models only

The *-tma shapes are A and B at a width the TMA input ring takes.  Every model -- the four calibrated ones and all edge
models -- runs A and B (and C for the generic requantiser, the TMA shapes for the fast one) through
forward_frames_device, forward_frames_device_sse and forward_frames_host on both implementations, bit for bit against
the C oracle; the profiling build (QV_FUSED_PROFILE) runs B.  The CPU test pins the shapes' plan properties at 148 SMs,
so that a change of the planner that moves a shape off its property fails without a GPU; the GPU tests check them again
at the device's SM count, which is what fused_upload plans with.
"""
import numpy as np
import pytest

from oracle import oracle
from qcnn_gpu_b200 import api
from qcnn_gpu_b200.host import formats, synth
from test_edge_models import _builds, _net, _np_sse, _sse_run
from test_frame_sse import _plain_run
from test_fused_units import WT, check_cover, units_of

SHAPES = {                         # (frames, H, W)
    "A": (100, 16, 121),           # 200 units of 16 rows for 148 CTAs; last column 1 pixel wide
    "B": (150, 16, 250),           # the line in chunks of 49 rows: up to 4 columns of 4 frames per CTA; last column 10 wide
    "C": (8, 480, 832),            # the line in chunks of 182 rows, two columns for some CTAs
    "A-tma": (100, 16, 160),       # W % 16 == 0 and W >= 144: the TMA input ring applies
    "B-tma": (152, 16, 160),
}
IN_SLOTS = 32                      # rows of the kernel's input ring (qv_fused.cu)

EDGE = synth.edge_models()
CELLS = ["qp%d" % qp for qp in (22, 27, 32, 37)] + [e[0] for e in EDGE]

# The builds a cell of the matrix launches, by requantiser; together with the profiling build these are the six
# whole-frame builds a CTA runs several units of.
FAST_BUILDS = {("k_fused", (1, 0, 0, 0)), ("k_fused", (1, 0, 0, 1)), ("k_enh_sse", (1, 0))}
GENERIC_BUILDS = {("k_fused", (0, 0, 0, 0)), ("k_enh_sse", (0, 0))}
PROFILE_BUILD = ("k_fused", (1, 1, 0, 0))
MULTI_UNIT_BUILDS = FAST_BUILDS | GENERIC_BUILDS | {PROFILE_BUILD}
_LAUNCHED = {}                     # test -> the builds the profiler saw it launch


def check_plan(sm, shape):
    """Asserts that a whole-frame launch of `shape` on `sm` SMs has the shape's plan property."""
    n, h, w = SHAPES[shape]
    u, grid = units_of(sm, n, h, w)
    check_cover(u, grid, n, h, w, 0, h)
    line = not np.array_equal(u, units_of(sm, n, h, w, line=False)[0])
    per_cta = [u[u[:, 0] == b] for b in range(grid)]
    heights = u[:, 4] - u[:, 3]
    where = "shape %s (%dx%dx%d) at %d SMs" % (shape, n, h, w, sm)
    if shape[0] == "A":
        assert not line, where + ": expected equal row segments, the plan took the row line"
        assert (heights[u[:, 4] < h] == heights.max()).all(), where + ": row segments of unequal height"
        assert len(u) > grid, where + ": %d units for %d CTAs" % (len(u), grid)
        assert any(len(set(zip(p[:, 1], p[:, 2]))) >= 2 for p in per_cta), where + ": no CTA takes a second column"
        return
    assert line, where + ": expected the row line"
    if shape[0] == "B":
        cols = [set(zip(p[:, 1], p[:, 2])) for p in per_cta]
        assert any(len(c) >= 3 and len({f for f, _ in c}) >= 2 for c in cols), \
            where + ": no CTA covers 3 columns of 2 frames (most: %d)" % max(len(c) for c in cols)
        # CTA b's chunk starts at line position b * chunk / H; the permutation puts some other column there
        chunk, nstrips = int(heights[u[:, 0] == 0].sum()), (w + WT - 1) // WT
        moved = sum(1 for b, p in enumerate(per_cta) if p[0, 1] * nstrips + p[0, 2] != b * chunk // h)
        assert moved > 0, where + ": the row line's columns are not permuted"
    else:
        rows = np.array([int((p[:, 4] - p[:, 3]).sum()) for p in per_cta])
        assert (rows[:-1] == rows[0]).all() and rows[0] >= 4 * IN_SLOTS, where + ": chunks of %s rows" % sorted(set(rows))
        assert any(len(p) >= 2 for p in per_cta), where + ": no CTA takes a second unit"


@pytest.mark.parametrize("shape", SHAPES)
def test_shape_has_its_plan_property_at_148_sms(shape):
    check_plan(148, shape)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(autouse=True)
def _plain_builds(monkeypatch):
    """The switches that pick another build at model upload are off unless a test sets them."""
    for k in ("QV_FUSED_PROFILE", "QV_FUSED_TMA", "QV_FUSED_EXPERIMENT"):
        monkeypatch.delenv(k, raising=False)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _model(cell, models):
    if cell.startswith("qp"):
        return models[int(cell[2:])]
    _, seed, family, variant = EDGE[CELLS.index(cell) - 4]
    return synth.make_edge_model(seed, family, variant)


def _is_fast(m):
    return all(synth.fast_row_ok(*m.qparams[l]) for l in synth.HIDDEN)


def _frames(seed, n, h, w, blocky):
    """(anchor, original): synth.make_frames' blocky content or uniform noise."""
    if blocky:
        return synth.make_frames(seed, n, h, w)
    return synth.make_uniform_frames(seed, n, h, w), synth.make_uniform_frames(seed + 1, n, h, w)


def _same(got, want, where):
    bad = int(np.count_nonzero(got != want))
    assert bad == 0, "%s: %d of %d pixels differ from the oracle" % (where, bad, want.size)


def _same_sse(sse, x, ori, want, where):
    ref = np.stack([_np_sse(x, ori), _np_sse(want, ori)], axis=1)
    bad = np.count_nonzero(sse != ref, axis=0)
    assert not bad.any(), "%s: SSE of %d (anchor) / %d (oracle frame) of %d frames differ from numpy" % (where, bad[0], bad[1], len(x))


def _launched(prof):
    return {b for b in (_builds(e.name) for e in prof.events()) if b}


PATHS = ((api.IMPL_FUSED, "fused"), (api.IMPL_LAYERED, "layered"))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", CELLS)
def test_every_model_where_ctas_run_several_units(cell, models, monkeypatch):
    """One oracle run per shape, shared by every entry point and path of the cell."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    m = _model(cell, models)
    fast = _is_fast(m)
    image = formats.write_model_vect_c(m)
    om = oracle.OracleModel(image)
    sm = _sm_count()
    shapes = ["A", "B"] + (["A-tma", "B-tma"] if fast else ["C"])
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for si, shape in enumerate(shapes):
            check_plan(sm, shape)
            n, h, w = SHAPES[shape]
            x, ori = _frames(0x3A17 + 16 * CELLS.index(cell) + si, n, h, w, (CELLS.index(cell) + si) % 2)
            want = om.forward_blu(x)
            tma = shape.endswith("-tma")
            if tma:
                monkeypatch.setenv("QV_FUSED_TMA", "1")                 # read when the model is uploaded
            for impl, path in PATHS[:1] if tma else PATHS:
                where = "%s, shape %s (%dx%dx%d), %s path%s" % (cell, shape, n, h, w, path, " with the TMA input ring" if tma else "")
                net = _net(image, n, h, w, impl)
                _same(_plain_run(net, x), want, where + ", forward_frames_device")
                _same(net.forward_frames_host(x), want, where + ", forward_frames_host")
                if not tma:
                    out, sse = _sse_run(net, x, ori)
                    _same(out, want, where + ", forward_frames_device_sse")
                    _same_sse(sse, x, ori, want, where + ", forward_frames_device_sse")
                net.close()
            monkeypatch.delenv("QV_FUSED_TMA", raising=False)
        torch.cuda.synchronize()
    launched = _launched(prof)
    want_builds = FAST_BUILDS if fast else GENERIC_BUILDS
    assert launched == want_builds, "%s: launched %s, expected %s" % (cell, sorted(launched), sorted(want_builds))
    _LAUNCHED[cell] = launched


@pytest.mark.gpu
def test_profiling_build_on_the_row_line(models, monkeypatch, capfd):
    """QV_FUSED_PROFILE=1 at upload: whole frames of a fast model run the profiling build, which reports its phase timers
    on stderr; a generic model runs the plain generic build and reports nothing; the SSE form is never profiled."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    shape = "B"
    check_plan(_sm_count(), shape)
    n, h, w = SHAPES[shape]
    x, ori = _frames(0x9F0F, n, h, w, True)
    monkeypatch.setenv("QV_FUSED_PROFILE", "1")
    launched = {}
    for cell in ("full_scale-fast", "full_scale-generic"):
        m = _model(cell, models)
        fast = _is_fast(m)
        assert fast == cell.endswith("-fast"), cell
        image = formats.write_model_vect_c(m)
        want = oracle.OracleModel(image).forward_blu(x)
        where = "%s, shape %s (%dx%dx%d), fused path under QV_FUSED_PROFILE" % (cell, shape, n, h, w)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            net = _net(image, n, h, w, api.IMPL_FUSED)
            capfd.readouterr()
            _same(_plain_run(net, x), want, where + ", forward_frames_device")
            err = capfd.readouterr().err
            if fast:
                assert "[qv fused profile]" in err, where + ": no profile report on stderr"
            else:
                assert "[qv fused profile]" not in err, where + ": a generic model must not run the profiling build"
            out, sse = _sse_run(net, x, ori)
            _same(out, want, where + ", forward_frames_device_sse")
            _same_sse(sse, x, ori, want, where + ", forward_frames_device_sse")
            assert "[qv fused profile]" not in capfd.readouterr().err, where + ": the SSE form ran the profiling build"
            net.close()
            torch.cuda.synchronize()
        launched[cell] = _launched(prof)
    want_builds = {"full_scale-fast": {PROFILE_BUILD, ("k_enh_sse", (1, 0))},
                   "full_scale-generic": {("k_fused", (0, 0, 0, 0)), ("k_enh_sse", (0, 0))}}
    assert launched == want_builds, "profiling build test: launched %s, expected %s" % (launched, want_builds)
    _LAUNCHED["profiling"] = set().union(*launched.values())


@pytest.mark.gpu
def test_the_matrix_launched_every_multi_unit_build():
    """Over the whole matrix: k_fused<1,0,0,0>, <0,0,0,0>, <1,0,0,1> (the TMA input ring, which falls back to the plain
    build without a word), <1,1,0,0> (profiling) and k_enh_sse<1,0>, <0,0>."""
    missing = [t for t in CELLS + ["profiling"] if t not in _LAUNCHED]
    if missing:
        pytest.skip("needs the whole matrix of this file in one session; did not run or failed: %s" % ", ".join(missing))
    seen = set().union(*_LAUNCHED.values())
    assert MULTI_UNIT_BUILDS <= seen, sorted(MULTI_UNIT_BUILDS - seen)
