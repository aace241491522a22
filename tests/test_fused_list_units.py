"""How a frame-list launch (qv_forward_frame_list_device) is dealt out to the persistent CTAs, checked on the CPU.

`qv_debug_fused_list_units` runs the host's list plan and reads it back through the same `list_unit_geo()` the kernel's
three warp roles call: every (frame, strip column, row) of every frame is covered exactly once, a unit never crosses a
column, every CTA gets the planned chunk of rows (the last one the rest), and it pays one pipeline fill per column its
chunk touches, no more.
"""
import random

import numpy as np
import pytest

from qcnn_gpu_b200 import api
from test_fused_units import WT, units_of

CTC = [(240, 416), (480, 832), (720, 1280), (1080, 1920), (1600, 2560)]      # (height, width) of the HEVC test classes D .. A
EDGE_W = [1, 7, 119, 120, 121, 240, 241, 2160]
CAP = api.FRAME_LIST_LAUNCH_MAX


def check_list(sm, hw):
    hs = [h for h, _ in hw]
    ws = [w for _, w in hw]
    u, grid = api.fused_list_units(sm, hs, ws)
    assert 1 <= grid <= sm
    cover = [np.zeros(((w + WT - 1) // WT, h), np.int32) for h, w in hw]
    for cta, f, s, y0, y1 in u:
        h, w = hw[f]
        assert 0 <= cta < grid and 0 <= s < (w + WT - 1) // WT and 0 <= y0 < y1 <= h, (cta, f, s, y0, y1)
        cover[f][s, y0:y1] += 1
    for f, c in enumerate(cover):
        assert (c == 1).all(), "frame %d (%dx%d): a row of some strip column is not covered exactly once" % (f, hw[f][1], hw[f][0])
    # the chunk: the row line over all columns in equal parts; a CTA pays one pipeline fill per column it touches
    line = sum(((w + WT - 1) // WT) * h for h, w in hw)
    chunk = -(-line // grid)
    rows = np.zeros(grid, np.int64)
    units = np.zeros(grid, np.int64)
    for cta, f, s, y0, y1 in u:
        rows[cta] += y1 - y0
        units[cta] += 1
    assert rows.max() <= chunk and (grid == 1 or rows[:-1].min() == chunk)
    # ... and exactly one unit (one pipeline fill) per column its chunk [b * chunk, (b + 1) * chunk) of the line intersects
    ends = np.cumsum([h for h, w in hw for _ in range((w + WT - 1) // WT)])
    starts = ends - np.repeat([h for h, _ in hw], [(w + WT - 1) // WT for _, w in hw])
    for b in range(grid):
        lo, hi = b * chunk, min(line, (b + 1) * chunk)
        assert units[b] == int(((starts < hi) & (ends > lo)).sum()), (b, units[b])
    return u, grid


def test_ctc_tick():
    hw = [CTC[0]] * 4 + [CTC[1]] * 4 + [CTC[2]] * 2 + [CTC[3]] * 2 + [CTC[4]]
    u, grid = check_list(148, hw)
    assert grid == 148                                         # a tick of mixed sizes fills every SM


def test_ragged_and_tiny_frames():
    check_list(148, [(33, 61), (7, 121), (1, 1), (300, 5)])
    check_list(148, [(1, 1)] * CAP)
    check_list(1, [(1, 1)])
    check_list(7, [(2160, 3840), (1, 1), (240, 416)])


def test_seeded_lists():
    rng = random.Random(0x1157)
    for _ in range(300):
        sm = rng.choice([1, 2, 7, 64, 132, 148, 160])
        n = rng.choice([1, 2, 3, 5, 13, 40, CAP]) if rng.random() < 0.3 else rng.randint(1, 24)
        hw = []
        for _ in range(n):
            r = rng.random()
            if r < 0.25:
                hw.append(rng.choice(CTC))
            elif r < 0.5:
                hw.append((rng.choice([1, 2, 119, 120, 121, 240, 241, 2160]), rng.choice(EDGE_W)))
            else:
                hw.append((rng.randint(1, 2160), rng.randint(1, 2160)))
        check_list(sm, hw)


@pytest.mark.parametrize("n,h,w", [(64, 1080, 1920), (8, 480, 832), (4, 720, 1280), (2, 1600, 2560), (16, 1080, 1920), (240, 2160, 3840)])
def test_uniform_list_cuts_the_whole_frame_line(n, h, w):
    """A list of one geometry cuts the same line as the whole-frame launch when that launch takes its row-line plan: the
    same grid and the same rows per CTA.  The units differ in which columns a CTA gets: the whole-frame line permutes its
    columns so that neighbouring CTAs work on neighbouring strip columns, the list walks them in (frame, column) order.
    (Where the whole-frame planner prefers equal row segments -- small launches -- the list still cuts the line.)"""
    u, grid = check_list(148, [(h, w)] * n)
    v, vgrid = units_of(148, n, h, w, line=True)
    line = n * ((w + WT - 1) // WT) * h
    g = max(1, min(148, line // 32))
    chunk = -(-line // g)
    want = np.full(-(-line // chunk), chunk)
    want[-1] = line - chunk * (len(want) - 1)
    rows_u = np.bincount(u[:, 0], weights=u[:, 4] - u[:, 3], minlength=grid)
    rows_v = np.bincount(v[:, 0], weights=v[:, 4] - v[:, 3], minlength=vgrid)
    assert np.array_equal(rows_u, want)
    if not np.array_equal(rows_v, want):
        pytest.skip("the whole-frame planner keeps equal row segments for this batch")
    assert grid == vgrid


def test_bad_lists_are_refused():
    too_long = ([1] * 10 + [65536], [1] * 10 + [120 * 16385])                     # one launch's line > 2^30 rows
    for sm, hs, ws in [(0, [16], [16]), (148, [], []), (148, [0], [16]), (148, [16], [0]), (148, [1] * (CAP + 1), [1] * (CAP + 1)),
                       (148,) + too_long]:
        with pytest.raises(api.QVError) as e:
            api.fused_list_units(sm, hs, ws)
        assert e.value.code == -1, (sm, len(hs))
    api.fused_list_units(148, [1] * CAP, [1] * CAP)
