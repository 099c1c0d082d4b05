"""Host-side parts of the panel-swept k-NN (engine.degree_knn) that need no GPU: argument validation of
the list-merge entry points, the panel plan and the dealing of panels to ranks."""
import ctypes

import pytest


@pytest.fixture
def buf():
    b = (ctypes.c_float * 256)()
    return b, ctypes.addressof(b)


def test_topk_merge_argument_validation_without_gpu(buf):
    """Bad arguments are rejected before any CUDA call, with an error string."""
    from hsd_b200._lib import lib
    _, p = buf
    # hsd_topk_merge(idx_in, val_in, n_lists, list_stride, idx_offset, n_rows, k, idx_io, val_io, stream)
    assert lib.hsd_topk_merge(None, p, 1, 8, 0, 2, 4, p, p, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 1, 8, 0, 2, 4, p, None, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 1, 8, 0, 2, 0, p, p, None) == -1 and b"k must be" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 1, 8, 0, 2, 65, p, p, None) == -1 and b"k must be" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 0, 8, 0, 2, 4, p, p, None) == -1 and b"n_lists" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 65, 8, 0, 2, 4, p, p, None) == -1 and b"n_lists" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 2, 7, 0, 2, 4, p, p, None) == -1 and b"list_stride" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge(p, p, 1, 8, 0, -1, 4, p, p, None) == -1                 # n_rows >= 0
    assert lib.hsd_topk_merge(p, p, 1, 8, -3, 2, 4, p, p, None) == -1                 # idx_offset >= 0
    assert lib.hsd_topk_merge(p, p, 2, 8, 0, 0, 4, p, p, None) == 0                   # no rows: nothing to do


def test_topk_merge_cols_argument_validation_without_gpu(buf):
    from hsd_b200._lib import lib
    _, p = buf
    # hsd_topk_merge_cols(blk, ld, n_rows, c_begin, n_cols, row_node0, col_node0, k, idx_io, val_io, stream)
    assert lib.hsd_topk_merge_cols(None, 8, 2, 0, 8, 0, 0, 4, p, p, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 8, 2, 0, 8, 0, 0, 4, None, p, None) == -1 and b"null" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 8, 2, 0, 8, 0, 0, 0, p, p, None) == -1 and b"k must be" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 8, 2, 0, 8, 0, 0, 65, p, p, None) == -1 and b"k must be" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 7, 2, 0, 8, 0, 0, 4, p, p, None) == -1 and b"ld" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 8, 2, 9, 8, 0, 0, 4, p, p, None) == -1 and b"c_begin" in lib.hsd_last_error_string()
    assert lib.hsd_topk_merge_cols(p, 8, 2, -1, 8, 0, 0, 4, p, p, None) == -1                # c_begin >= 0
    assert lib.hsd_topk_merge_cols(p, 8, -2, 0, 8, 0, 0, 4, p, p, None) == -1                # n_rows >= 0
    assert lib.hsd_topk_merge_cols(p, 8, 2, 0, 8, -1, 0, 4, p, p, None) == -1                # node ids >= 0
    assert lib.hsd_topk_merge_cols(p, 8, 2, 8, 8, 0, 0, 4, p, p, None) == 0                  # no columns: nothing to do


@pytest.mark.parametrize("n,rows", [(1, 128), (127, 128), (128, 128), (129, 128), (1000, 256), (4099, 1024),
                                    (20000, 2048), (300000, 8192), (300001, 37248), (5000, 5000), (5000, 99999)])
def test_knn_panels_tile_the_rows(n, rows):
    from hsd_b200.engine import knn_panels
    panels = knn_panels(n, rows)
    assert panels[0][0] == 0 and panels[-1][1] == n
    seen = [0] * n
    for r0, r1 in panels:
        assert r0 < r1
        for i in range(r0, r1) if n < 10000 else (r0, r1 - 1):
            seen[i] += 1
    if n < 10000:
        assert seen == [1] * n                                # every row in exactly one panel
    for (a0, a1), (b0, _) in zip(panels[:-1], panels[1:]):
        assert a1 == b0 and a0 % 128 == 0 and a1 % 128 == 0 and a1 - a0 == rows
    if rows < n:
        assert panels[-1][1] - panels[-1][0] == n - (len(panels) - 1) * rows    # ragged last panel
        assert len(panels) == -(-n // rows)
    else:
        assert panels == [(0, n)]
    with pytest.raises(ValueError):
        knn_panels(n + 1000, 100)                              # not a multiple of 128


def test_knn_panel_rows_from_the_budget():
    from hsd_b200.engine import knn_panel_rows
    gb = 1 << 30
    budget = 178 * gb // 2                                     # default: half the free memory of an idle B200
    assert knn_panel_rows(20000, budget) == 20000              # 1.6 GB matrix: one panel
    assert knn_panel_rows(100000, budget) == 100000            # 40 GB matrix: one panel
    r = knn_panel_rows(300000, budget)                         # 360 GB matrix: panels of the largest fitting R
    assert r % 128 == 0 and r * 300000 * 4 <= budget < (r + 128) * 300000 * 4
    assert knn_panel_rows(300000, 1) == 128                    # never below one tile row
    r8 = knn_panel_rows(300000, budget, world=8)               # several ranks: enough panels to deal
    assert r8 % 128 == 0 and -(-300000 // r8) >= 8 * 8


@pytest.mark.parametrize("world", [2, 3, 8])
@pytest.mark.parametrize("n,rows", [(20000, 512), (100000, 2048), (300000, 4608), (4099, 128)])
def test_knn_deal_balances_the_ranks(n, rows, world):
    from hsd_b200.engine import knn_deal, knn_panel_work, knn_panels
    panels = knn_panels(n, rows)
    deal = knn_deal(n, panels, world)
    assert deal == knn_deal(n, list(reversed(panels)), world)              # deterministic, order-free
    assert sorted(p for m in deal for p in m) == panels                     # every panel exactly once
    assert all(m == sorted(m) for m in deal)                                # each rank sweeps top to bottom
    load = [sum(knn_panel_work(n, *p) for p in m) for m in deal]
    mean = sum(load) / world
    assert max(load) - mean <= max(knn_panel_work(n, *p) for p in panels)   # within one panel of the mean
    assert abs(sum(load) - n * (n - 1) / 2 - n / 2) < 1e-6 * n * n          # every pair once (+ the diagonal)
