"""The C ABI's refusals of the two flip entry points of the row-sharded gradient (DESIGN.md section 15):
more than 64 flips, an index at or past ``n_global``, a negative index or a missing array is refused
before anything launches, and the flip-free ``egnn_adj_grad_degree_sharded`` is the same call without
flips.  The device pointers are fakes that are never dereferenced: with a device present a passing
check could reach a launch, so the tests skip there."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="fake device pointers: must not reach a launch")

N = 8


def ok(i):
    return (1 << 20) + 4096 * i          # 16-byte aligned fakes


_keep = []


def flips(row=0, col=1, n=1):
    rows, cols = np.zeros(n, dtype=np.int32), np.ones(n, dtype=np.int32)
    rows[0], cols[0] = row, col
    vals = np.ones(n, dtype=np.float32)
    _keep.append((rows, cols, vals))
    return rows.ctypes.data, cols.ctypes.data, vals.ctypes.data, n


BAD = [((None, None, None, 65), b"n_delta"), ((None, None, None, 1), b"delta arrays missing")] + \
    [(flips(r, c), b"delta index out of range") for r, c in ((N, 0), (0, N), (-1, 0), (0, -1))]


def test_degree_sharded_flips_refusals():
    from efficient_gnn_b200 import _cabi
    lib = _cabi.load()
    ws = int(lib.egnn_adj_grad_degree_sharded_ws_bytes(4))

    def call(d, g_flips=ok(12), wsb=ws, rows=(0, 4)):
        return lib.egnn_adj_grad_degree_sharded_flips(ok(1), ok(2), None, None, ok(4), ok(5), None, None, ok(7),
                                                      ok(8), N, rows[0], rows[1], 4, 3, 1.0, ok(10), ok(11), None,
                                                      None, *d, g_flips, ok(13), ok(14), ok(15), ok(16), wsb, None)

    for d, msg in BAD:
        assert call(d) == -1 and msg in lib.egnn_last_error(), (d, lib.egnn_last_error())
        assert call(d, wsb=ws - 1) == -1 and msg in lib.egnn_last_error()     # refused before the workspace
    assert call(flips(0, 1), g_flips=None) == -1 and b"g_flips_out" in lib.egnn_last_error()
    assert call(flips(0, 1), wsb=ws - 1) != 0 and b"too small" in lib.egnn_last_error()
    assert call(flips(N - 1, 0, n=64), rows=(4, 4)) == 0          # a rank without rows: nothing to do
    # the flip-free entry point is this call without flips
    assert lib.egnn_adj_grad_degree_sharded(ok(1), ok(2), None, None, ok(4), ok(5), None, None, ok(7), ok(8), N, 0,
                                            4, 4, 3, 1.0, ok(10), ok(11), None, None, ok(13), ok(14), ok(15),
                                            ok(16), ws - 1, None) != 0
    assert b"too small" in lib.egnn_last_error()


def test_flips_sharded_refusals():
    from efficient_gnn_b200 import _cabi
    lib = _cabi.load()

    def call(d, gw=ok(2), rows=(0, 4)):
        return lib.egnn_adj_grad_flips_sharded(*d, ok(1), gw, ok(3), N, rows[0], rows[1], 1.0, ok(4), None)

    for d, msg in BAD:
        assert call(d) == -1 and msg in lib.egnn_last_error(), (d, lib.egnn_last_error())
    assert call(flips(0, 1), gw=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert call(flips(0, 1), rows=(4, 9)) == -1 and b"row range" in lib.egnn_last_error()
    assert call((None, None, None, 0), gw=None) == 0                 # no flips: nothing to write
