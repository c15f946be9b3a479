"""No-GPU checks of the adjacency-gradient entry points of the C ABI: argument errors come back as
status codes before anything is launched (the fake pointers below are never dereferenced)."""
import numpy as np

from efficient_gnn_b200 import _cabi

BASE = 1 << 20


def ok(i):
    return BASE + 4096 * i               # 16-byte aligned fakes


def test_adjoint_all_refuses_null_and_misaligned_b_all():
    lib = _cabi.load()
    coeffs = np.ones(8, dtype=np.float32)
    args = [ok(1), ok(2), None, ok(3), ok(4), 4, 4, 4, 3, 1, coeffs.ctypes.data, 1.0, -1.0, ok(5), None, ok(6),
            None, None, None, 0, None, 0, None, None, None]
    assert lib.egnn_cheb_adjoint_all(*args, None) == -1
    assert b"b_all" in lib.egnn_last_error()
    assert lib.egnn_cheb_adjoint_all(*args, ok(7) + 4) == -1
    assert b"16-byte aligned" in lib.egnn_last_error()
    assert lib.egnn_cheb_adjoint_all(*args, ok(7)) == -4          # NULL workspace: refused, nothing launched


def test_adjacency_gradient_argument_errors():
    lib = _cabi.load()
    assert lib.egnn_adj_grad_degree_ws_bytes(1000) >= 2 * 8 * 1000
    rc = lib.egnn_adj_grad_degree(None, None, None, None, None, None, None, None, 4, 4, 1, 3, 1.0, None, None, None,
                                  None, None, None, None, 0, None)
    assert rc == -1 and b"null pointer" in lib.egnn_last_error()
    rc = lib.egnn_adj_grad_degree(ok(1), ok(2), ok(3), ok(4), ok(5), None, ok(6), ok(7), 4, 4, 1, 3, 1.0, ok(8),
                                  ok(9), None, None, ok(10), ok(11), None, 0, None)
    assert rc == -1 and b"vals and vals_t" in lib.egnn_last_error()
    rc = lib.egnn_adj_grad_degree(ok(1), ok(2), None, ok(4), ok(5), None, ok(6), ok(7), 4, 4, 1, 3, 1.0, ok(8),
                                  ok(9), None, None, ok(10), ok(11), None, 0, None)
    assert rc == -4 and b"workspace" in lib.egnn_last_error()
    assert lib.egnn_adj_grad_pairs(ok(1), ok(2), 5, ok(3), None, None, ok(4), ok(5), 4, 1, 3, 1.0, ok(6), None) == -1
    assert lib.egnn_adj_grad_pairs(None, None, 0, None, None, None, None, None, 4, 1, 3, 1.0, None, None) == 0
    assert lib.egnn_adj_grad_dense(ok(1), ok(2), ok(3), ok(4), ok(5), 8, 1, 3, 1.0, ok(6), 4, None) == -1
    assert b"ld" in lib.egnn_last_error()
    assert lib.egnn_adj_grad_dense(ok(1), None, None, ok(4), ok(5), 8, 1, 3, 1.0, ok(6), 8, None) == -1
