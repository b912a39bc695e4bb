"""CPU: argument validation of the batched row copy behind the rollout engine's snapshot / restore (tb_copy_rows)."""
import ctypes

import pytest

from trafficbotsv1_5_b200 import lib

TB_ERR_BAD_SHAPE, TB_ERR_UNSUPPORTED, TB_ERR_NULL = -1, -3, -5
TB_COPY_ROWS_MAX = 64


@pytest.fixture(scope="module")
def handle():
    lib.build()
    return lib.load()


def _items(*specs):
    """specs: (src, dst, row_bytes, n_rows, per_rollout) with fake device addresses (never dereferenced: validation
    fails before any launch)."""
    arr = (lib.RowCopy * max(len(specs), 1))()
    for i, s in enumerate(specs):
        arr[i] = lib.RowCopy(*s)
    return arr


def test_row_copy_struct_layout():
    assert ctypes.sizeof(lib.RowCopy) == 32
    assert lib.RowCopy.row_bytes.offset == 16 and lib.RowCopy.n_rows.offset == 24 and lib.RowCopy.per_rollout.offset == 28


def test_copy_rows_error_codes_without_gpu(handle):
    f = handle.tb_copy_rows
    a, b, m = 16, 4096, 8192  # distinct non-null fake addresses
    ok = (a, b, 12, 6, 1)
    assert f(None, 1, None, 3, None) == TB_ERR_NULL
    assert f(_items((None, b, 12, 6, 0)), 1, None, 3, None) == TB_ERR_NULL
    assert f(_items(ok, (a, None, 12, 6, 0)), 2, None, 3, None) == TB_ERR_NULL
    assert f(_items(ok), 0, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items(*[ok] * (TB_COPY_ROWS_MAX + 1)), TB_COPY_ROWS_MAX + 1, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items((a, b, 0, 6, 0)), 1, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items((a, b, -4, 6, 0)), 1, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items((a, b, 12, 0, 0)), 1, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items((a, b, 12, 7, 1)), 1, m, 3, None) == TB_ERR_BAD_SHAPE       # 7 rows are not whole scenes of R = 3
    assert f(_items((a, b, 12, 7, 1)), 1, None, 3, None) == TB_ERR_BAD_SHAPE
    assert f(_items(ok), 1, m, 0, None) == TB_ERR_BAD_SHAPE                    # per-rollout rows need R > 0
    assert f(_items((a, a, 12, 6, 1)), 1, m, 3, None) == TB_ERR_UNSUPPORTED     # in-place gather would race
    assert handle.tb_strerror(TB_ERR_UNSUPPORTED).decode() == "unsupported size"
