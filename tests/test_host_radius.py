"""Host-side parts of the radius graph (engine.degree_radius) that need no GPU: argument validation of the
hsd_radius_* entry points, the float32 threshold, the panel plan and the default cap."""
import ctypes
import math

import numpy as np
import pytest


@pytest.fixture
def buf():
    b = (ctypes.c_float * 256)()
    return b, ctypes.addressof(b)


def test_radius_count_argument_validation_without_gpu(buf):
    """Bad arguments are rejected before any CUDA call, with an error string."""
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_radius_count(blk, elem_bytes, ld, n_rows, n_cols, radius, hits, hits_ld, row_cnt, col_cnt, stream)
    assert lib.hsd_radius_count(None, 4, 8, 2, 8, 1.0, p, 1, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_count(p, 4, 8, 2, 8, 1.0, None, 1, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_count(p, 4, 8, 2, 8, 1.0, p, 1, None, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_count(p, 4, 8, 2, 8, 1.0, p, 1, p, None, None) == -1 and b"null" in err()
    assert lib.hsd_radius_count(p, 2, 8, 2, 8, 1.0, p, 1, p, p, None) == -1 and b"elem_bytes" in err()
    assert lib.hsd_radius_count(p, 4, 7, 2, 8, 1.0, p, 1, p, p, None) == -1 and b"ld" in err()
    assert lib.hsd_radius_count(p, 4, 40, 2, 40, 1.0, p, 1, p, p, None) == -1 and b"hits_ld" in err()
    assert lib.hsd_radius_count(p, 4, 8, -1, 8, 1.0, p, 1, p, p, None) == -1                 # n_rows >= 0
    assert lib.hsd_radius_count(p, 8, 8, 2, 8, math.nan, p, 1, p, p, None) == -1 and b"radius" in err()
    assert lib.hsd_radius_count(p, 8, 8, 2, 8, -1e-30, p, 1, p, p, None) == -1 and b"radius" in err()
    assert lib.hsd_radius_count(p, 4, 8, 0, 8, math.inf, p, 1, p, p, None) == 0            # no rows: nothing to do


@pytest.mark.parametrize("name", ["hsd_radius_emit_rows", "hsd_radius_emit_cols"])
def test_radius_emit_argument_validation_without_gpu(buf, name):
    from hsd_b200._lib import lib
    _, p = buf
    f, err = getattr(lib, name), lib.hsd_last_error_string
    # (blk, elem_bytes, ld, n_rows, n_cols, hits, hits_ld, off, node0, idx_out, val_out, stream)
    assert f(None, 4, 8, 2, 8, p, 1, p, 0, p, p, None) == -1 and b"null" in err()
    assert f(p, 4, 8, 2, 8, None, 1, p, 0, p, p, None) == -1 and b"null" in err()
    assert f(p, 4, 8, 2, 8, p, 1, None, 0, p, p, None) == -1 and b"null" in err()
    assert f(p, 4, 8, 2, 8, p, 1, p, 0, None, p, None) == -1 and b"null" in err()
    assert f(p, 4, 8, 2, 8, p, 1, p, 0, p, None, None) == -1 and b"null" in err()
    assert f(p, 16, 8, 2, 8, p, 1, p, 0, p, p, None) == -1 and b"elem_bytes" in err()
    assert f(p, 4, 4, 2, 8, p, 1, p, 0, p, p, None) == -1 and b"ld" in err()
    assert f(p, 4, 64, 2, 64, p, 1, p, 0, p, p, None) == -1 and b"hits_ld" in err()
    assert f(p, 4, 8, 2, 8, p, 1, p, -1, p, p, None) == -1 and b"node ids" in err()
    assert f(p, 4, 8, 8, 8, p, 1, p, 2**31 - 4, p, p, None) == -1 and b"node ids" in err()
    assert f(p, 8, 8, 0, 8, p, 1, p, 0, p, p, None) == 0                                     # no rows


def test_radius_scatter_argument_validation_without_gpu(buf):
    from hsd_b200._lib import lib
    _, p = buf
    err = lib.hsd_last_error_string
    # hsd_radius_scatter(idx, val, elem_bytes, off, n_seg, node0, indptr, cursor, idx_out, val_out, stream)
    assert lib.hsd_radius_scatter(p, p, 4, None, 2, 0, p, p, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_scatter(p, p, 4, p, 2, 0, None, p, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_scatter(p, p, 4, p, 2, 0, p, None, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_scatter(p, p, 4, p, 2, 0, p, p, None, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_scatter(None, p, 4, p, 2, 0, p, p, p, p, None) == -1 and b"null" in err()
    assert lib.hsd_radius_scatter(p, p, 3, p, 2, 0, p, p, p, p, None) == -1 and b"elem_bytes" in err()
    assert lib.hsd_radius_scatter(p, p, 4, p, -1, 0, p, p, p, p, None) == -1                 # n_seg >= 0
    assert lib.hsd_radius_scatter(p, p, 4, p, 2, -5, p, p, p, p, None) == -1                 # node0 >= 0
    assert lib.hsd_radius_scatter(None, None, 8, p, 0, 0, p, p, p, p, None) == 0             # no segments


def _f32_below_or_at(r):
    """Reference: the largest float32 not above r, by scanning the neighbours of float32(r)."""
    c = np.float32(r) if r < 3.5e38 else np.float32(np.finfo(np.float32).max)
    for _ in range(3):
        if float(c) > r:
            c = np.nextafter(c, np.float32(-np.inf))
    while float(np.nextafter(c, np.float32(np.inf))) <= r and np.isfinite(np.nextafter(c, np.float32(np.inf))):
        c = np.nextafter(c, np.float32(np.inf))
    return c


@pytest.mark.parametrize("base", [0.0, 1.0, 0.1, 2.5, 1e-3, 17.25, 1e-40, 3.0e38])
def test_radius_threshold_f32_rounds_down(base):
    """r32 is the largest float32 <= radius, so for every float32 d: d <= r32 iff float(d) <= radius —
    checked at a float32 value, and just above and below it (the doubles between neighbouring floats)."""
    from hsd_b200.engine import radius_threshold_f32
    f = np.float32(base)
    up, down = np.nextafter(f, np.float32(np.inf)), np.nextafter(f, np.float32(0))
    for r in (float(f), float(f) + (float(up) - float(f)) / 3, float(f) - (float(f) - float(down)) / 3,
              math.nextafter(float(f), math.inf), math.nextafter(float(f), 0.0)):
        if r < 0:
            continue
        t = radius_threshold_f32(r)
        assert t.dtype == np.float32 and float(t) <= r
        assert t == _f32_below_or_at(r), (r, t)
        for d in (down, f, up):
            assert (d <= t) == (float(d) <= r), (r, d, t)
    assert radius_threshold_f32(math.inf) == np.float32(np.inf)
    assert radius_threshold_f32(1e39) == np.finfo(np.float32).max          # above FLT_MAX: the largest float
    assert radius_threshold_f32(0.0) == 0.0


def test_radius_rejects_nan_and_negative():
    from hsd_b200.engine import check_radius
    for bad in (math.nan, -1.0, -1e-300, float("-inf")):
        with pytest.raises(ValueError, match="radius"):
            check_radius(bad)
    assert check_radius(0) == 0.0 and check_radius(math.inf) == math.inf and check_radius(np.float32(2.5)) == 2.5


def test_radius_panel_rows_count_the_bitmap():
    from hsd_b200.engine import knn_panel_rows, radius_panel_rows
    gb = 1 << 30
    budget = 178 * gb // 2
    assert radius_panel_rows(20000, budget) == 20000
    assert radius_panel_rows(100000, budget) == 100000
    n = 300000
    r = radius_panel_rows(n, budget)
    row = 4 * n + 4 * ((n + 31) // 32)
    assert r % 128 == 0 and r * row <= budget < (r + 128) * row
    assert r <= knn_panel_rows(n, budget)
    assert radius_panel_rows(n, 1) == 128


def test_radius_max_pairs_formula():
    from hsd_b200.engine import RADIUS_PAIR_FRACTION, radius_max_pairs
    free = 10 ** 10
    assert radius_max_pairs(free, 4) == int(free * RADIUS_PAIR_FRACTION) // 16     # degree: 2 x (4 + 4) bytes
    assert radius_max_pairs(free, 8) == int(free * RADIUS_PAIR_FRACTION) // 24     # wavelet: 2 x (4 + 8) bytes
    assert radius_max_pairs(-5, 4) == 0


def test_chunk_rows_match_the_header():
    """The column counts' row chunk is a library constant the host code sizes its buffers with."""
    import os
    import re
    from hsd_b200.engine import RADIUS_CHUNK_ROWS
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "hsd_b200.h")).read()
    assert int(re.search(r"#define HSD_RADIUS_CHUNK_ROWS\s+(\d+)", hdr).group(1)) == RADIUS_CHUNK_ROWS


def test_radius_fixed_bytes_counts_every_buffer_beside_the_entries():
    """Panel buffer, bitmap, counts, the current panel's column-count scan, the offsets every panel keeps
    until the assembly, and the assembly's counts / indptr / cursor."""
    from hsd_b200.engine import RADIUS_CHUNK_ROWS, knn_panels, radius_fixed_bytes
    n = 100000
    panels = knn_panels(n, 128)
    chunks = -(-128 // RADIUS_CHUNK_ROWS)
    want = (4 * 128 * n + 4 * 128 * -(-n // 32) + 4 * 128 + 4 * n * chunks + 8 * (n * chunks + 1)
            + 8 * sum((r1 - r0 + 1) + (n - r0 + 1) for r0, r1 in panels) + 8 * (3 * n + 1))
    assert radius_fixed_bytes(n, panels) == want
    kept = 8 * sum((r1 - r0 + 1) + (n - r0 + 1) for r0, r1 in panels)
    assert kept > 0.3e9                                        # 782 panels of 128 rows: the offsets matter
    one = radius_fixed_bytes(n, [(0, n)], panel_buffer=False)   # resident matrix: no panel buffer
    assert one == (4 * n * -(-n // 32) + 4 * n + 4 * n * -(-n // RADIUS_CHUNK_ROWS)
                   + 8 * (n * -(-n // RADIUS_CHUNK_ROWS) + 1) + 8 * (2 * n + 2) + 8 * (3 * n + 1))
