"""No-GPU checks of the row-sharded backward entry points of the C ABI: argument errors come back as
status codes before anything is launched (the fake pointers below are never dereferenced)."""
import ctypes as C

import numpy as np

from efficient_gnn_b200 import _cabi

BASE = 1 << 20


def ok(i):
    return BASE + 4096 * i               # 16-byte aligned fakes


def _generic(lib, *, b_prev_local=ok(8), cbar=ok(11), tbar=None, acc=ok(12), f=4, app=1, k=3, phase=0,
             rows=(0, 4), n=8, n_delta=0):
    coeffs = np.ones(8 * (k + 1), dtype=np.float32)
    return lib.egnn_cheb_adjoint_sharded(ok(1), ok(2), ok(3), ok(4), ok(5), ok(6), ok(7), b_prev_local, None, ok(10),
                                         cbar, tbar, acc, n, 4, rows[0], rows[1], f, app, k, 1,
                                         coeffs.ctypes.data, 1.0, -1.0, phase, None, None, None, n_delta, None)


def test_cheb_adjoint_sharded_argument_errors():
    lib = _cabi.load()
    assert _generic(lib, cbar=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert _generic(lib, app=4) == -1 and b"bad application" in lib.egnn_last_error()
    assert _generic(lib, rows=(3, 9)) == -1 and b"row range" in lib.egnn_last_error()
    assert _generic(lib, phase=3) == -1 and b"phase" in lib.egnn_last_error()
    assert _generic(lib, b_prev_local=None) == -1 and b"b_{m+1}" in lib.egnn_last_error()
    for kw in ({"cbar": ok(11) + 4}, {"tbar": ok(13) + 8}, {"acc": ok(12) + 4}, {"b_prev_local": ok(8) + 4}):
        assert _generic(lib, **kw) == -1 and b"16-byte aligned" in lib.egnn_last_error()
    assert _generic(lib, cbar=ok(11) + 4, f=3, rows=(4, 4)) == 0   # f % 4 != 0: scalar accesses; no rows: nothing to do
    assert _generic(lib, n_delta=65, phase=1) == -1 and b"n_delta" in lib.egnn_last_error()


def _wide(lib, *, cbar=ok(6), xbar=ok(8), f=8, app=1, k=3, win=True, wf=8):
    coeffs = np.ones(8 * (k + 1), dtype=np.float32)
    w = _cabi.PeerWindowStruct()
    w.rank, w.world, w.rows_per, w.f = 0, 2, 4, wf
    w.base[0], w.base[1] = ok(20), ok(30)
    return lib.egnn_wide_adjoint_sharded(ok(1), ok(2), None, ok(4), ok(5), cbar, None, xbar, 8, 0, 4, f, app, k, 1,
                                         coeffs.ctypes.data, 1.0, -1.0, None, None, None, 0,
                                         C.byref(w) if win else None, None)


def test_wide_adjoint_sharded_argument_errors():
    lib = _cabi.load()
    assert _wide(lib, win=False) == -1 and b"null pointer" in lib.egnn_last_error()
    assert _wide(lib, f=4, wf=4) == -1 and b"f >= 8" in lib.egnn_last_error()
    assert _wide(lib, k=0, app=0) == -1 and b"k_max = 0" in lib.egnn_last_error()
    assert _wide(lib, app=3, xbar=None) == -1 and b"xbar" in lib.egnn_last_error()
    assert _wide(lib, cbar=ok(6) + 4) == -1 and b"16-byte aligned" in lib.egnn_last_error()
    assert _wide(lib, xbar=ok(8) + 8) == -1 and b"16-byte aligned" in lib.egnn_last_error()
    assert _wide(lib, wf=12) == -1 and b"window does not fit" in lib.egnn_last_error()
