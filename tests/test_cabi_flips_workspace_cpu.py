"""No-GPU checks of the edge-flip and workspace arguments of every C ABI entry point that takes them:
65 flips, or a flip index equal to the node count the flips address, come back as invalid-argument
errors, and a workspace one byte short as a workspace error, before anything is launched.  The
generic row-sharded entries look at the flips only in the phases that gather from the exchanged
operand (1 and 2), not in phase 0.  The device pointers below are fakes that are never
dereferenced: with a device present a passing check could reach a launch, so the module skips."""
import ctypes as C

import numpy as np
import pytest
import torch

from efficient_gnn_b200 import _cabi

pytestmark = pytest.mark.skipif(torch.cuda.is_available(), reason="fake device pointers: must not reach a launch on a GPU")

BASE = 1 << 20
N = 8
COEFFS = np.ones(8 * 21, dtype=np.float32)
CPTR = COEFFS.ctypes.data


def ok(i):
    return BASE + 4096 * i               # 16-byte aligned fakes


def flips(row=0, col=1, n=1):
    """The four flip arguments: n flips, the first one at (row, col)."""
    rows = np.full(max(n, 1), 0, dtype=np.int32)
    cols = np.full(max(n, 1), 1, dtype=np.int32)
    rows[0], cols[0] = row, col
    vals = np.ones(max(n, 1), dtype=np.float32)
    flips.keep = (rows, cols, vals)      # alive until the next call
    return rows.ctypes.data, cols.ctypes.data, vals.ctypes.data, n


def too_many():
    return None, None, None, 65


def window(world=2, rows_per=4, f=8):
    w = _cabi.PeerWindowStruct()
    w.rank, w.world, w.rows_per, w.f = 0, world, rows_per, f
    for r in range(world):
        w.base[r] = ok(40 + r)
    window.keep = w
    return C.byref(w)


def sell_plan(n=N, n_cols=N, filled=True):
    p = _cabi.SellPlanStruct()
    p.n, p.n_blocks, p.col_block, p.lmax, p.n_cols, p.row0, p.n_cta = n, 1, 32, 256, n_cols, 0, 4
    if filled:
        for i, name in enumerate(("slice_off", "blk_slice_ptr", "idx", "rv_ptr", "vslot", "cta_info", "vpart",
                                  "sched", "hub")):
            setattr(p, name, ok(60 + i))
    sell_plan.keep = p
    return p


# ---- one call per entry point taking flips; `d` is the four flip arguments --------------------------
def patch_degrees(lib, d):
    return lib.egnn_patch_degrees(ok(1), ok(2), ok(3), ok(4), ok(5), N, *d, ok(6), ok(7), ok(8), 0, N, None)


def patch_nodes(lib, d):
    return lib.egnn_patch_nodes(ok(1), ok(2), ok(3), ok(4), ok(5), ok(6), N, *d, ok(7), ok(8), ok(9), ok(10), 0, None)


def wavelet(lib, d=(None, None, None, 0), f=4, ws_bytes=None):
    ws = int(lib.egnn_cheb_workspace_bytes(N, f)) if ws_bytes is None else ws_bytes
    return lib.egnn_cheb_wavelet(ok(1), ok(2), None, ok(3), ok(4), ok(5), N, 16, f, 3, 1, CPTR, 1.0, -1.0,
                                 ok(6), None, 0, *d, ok(7), ws, None, None, None, None, None, 0, None, None, 0)


def adjoint(lib, d=(None, None, None, 0), f=4, ws_bytes=None, keep_all=False):
    ws = int(lib.egnn_cheb_workspace_bytes(N, f)) if ws_bytes is None else ws_bytes
    args = (ok(1), ok(2), None, ok(3), ok(4), N, 16, f, 3, 1, CPTR, 1.0, -1.0, ok(5), None, ok(6), *d, ok(7), ws,
            None, None, None)
    return lib.egnn_cheb_adjoint_all(*args, ok(8)) if keep_all else lib.egnn_cheb_adjoint(*args)


def adjoint_all(lib, d=(None, None, None, 0), f=4, ws_bytes=None):
    return adjoint(lib, d, f, ws_bytes, keep_all=True)


def order_sharded(lib, d, phase=1, acc=ok(12)):
    return lib.egnn_cheb_order_sharded(ok(1), ok(2), ok(3), ok(4), ok(5), ok(6), ok(7), ok(8), ok(9), ok(10), ok(11),
                                       acc, N, 16, 0, 4, 4, 2, 3, 1, CPTR, 1.0, -1.0, 0, phase, *d, None)


def adjoint_sharded(lib, d, phase=1, acc=ok(12)):
    return lib.egnn_cheb_adjoint_sharded(ok(1), ok(2), ok(3), ok(4), ok(5), ok(6), ok(7), ok(8), ok(9), ok(10), ok(11),
                                         None, acc, N, 16, 0, 4, 4, 1, 3, 1, CPTR, 1.0, -1.0, phase, *d, None)


def sell_step_sharded(lib, d):
    # a row shard of 8 of 16 columns without a window: one order on a gathered operand
    plan = sell_plan(n=N, n_cols=2 * N)
    return lib.egnn_sell_step_sharded(C.byref(plan), ok(1), ok(2), ok(3), ok(4), ok(5), ok(6), ok(7), ok(8), None,
                                      ok(9), 1, 1, 3, 1, CPTR, 1.0, -1.0, 0, *d, None, None, 0, None, None)


def wide_order_sharded(lib, d):
    return lib.egnn_wide_order_sharded(ok(1), ok(2), None, None, ok(3), ok(4), ok(5), None, ok(6), N, 0, 4, 8, 2, 3, 1,
                                       CPTR, 1.0, -1.0, 0, *d, window(), None)


def wide_adjoint_sharded(lib, d):
    return lib.egnn_wide_adjoint_sharded(ok(1), ok(2), None, ok(3), ok(4), ok(5), None, ok(6), N, 0, 4, 8, 1, 3, 1,
                                         CPTR, 1.0, -1.0, *d, window(), None)


def gcn_propagate(lib, d):
    return lib.egnn_gcn_propagate(ok(1), ok(2), None, ok(3), None, ok(4), None, N, 4, *d, None)


def gcn_target_logits(lib, d):
    return lib.egnn_gcn_target_logits(ok(1), ok(2), None, ok(3), ok(4), ok(5), 0, N, 4, 2, ok(6), ok(7), *d, None)


def gcn_structure_grad(lib, d):
    return lib.egnn_gcn_structure_grad(ok(1), ok(2), None, ok(3), ok(4), ok(5), ok(6), ok(7), ok(8), ok(9), 0, N, 4,
                                       2, ok(10), ok(11), *d, None)


# entry point -> the node count its flip indices must stay below
FLIP_ENTRIES = [
    (patch_degrees, N), (patch_nodes, N), (wavelet, N), (adjoint, N), (adjoint_all, N),
    (order_sharded, N), (adjoint_sharded, N), (sell_step_sharded, 2 * N),
    (wide_order_sharded, N), (wide_adjoint_sharded, N),
    (gcn_propagate, N), (gcn_target_logits, N), (gcn_structure_grad, N),
]


def error(lib):
    return lib.egnn_last_error()


@pytest.mark.parametrize("call,bound", FLIP_ENTRIES, ids=[c.__name__ for c, _ in FLIP_ENTRIES])
def test_flips_are_checked(call, bound):
    lib = _cabi.load()
    assert call(lib, too_many()) == -1 and b"n_delta" in error(lib), error(lib)
    assert call(lib, (None, None, None, 1)) == -1 and b"delta arrays missing" in error(lib), error(lib)
    for row, col in ((bound, 0), (0, bound), (-1, 0)):
        assert call(lib, flips(row, col)) == -1 and b"delta index out of range" in error(lib), (row, col, error(lib))


@pytest.mark.parametrize("call", [order_sharded, adjoint_sharded], ids=["order_sharded", "adjoint_sharded"])
def test_sharded_flips_are_ignored_in_phase_0(call):
    lib = _cabi.load()
    for phase in (1, 2):
        assert call(lib, too_many(), phase=phase, acc=None) == -1 and b"n_delta" in error(lib)
        assert call(lib, flips(N, 0), phase=phase, acc=None) == -1 and b"delta index" in error(lib)
    # phase 0 reaches its own check (the missing accumulator) whatever the flips
    for d in (too_many(), flips(N, 0)):
        assert call(lib, d, phase=0, acc=None) == -1 and b"local half missing" in error(lib), error(lib)


def test_workspace_one_byte_short_is_refused():
    lib = _cabi.load()

    def refused(what, rc):
        assert rc == -4 and b"workspace too small" in error(lib), (what, rc, error(lib))

    for f in (1, 4, 5, 8, 13):                  # every layout of the Chebyshev workspace
        short = int(lib.egnn_cheb_workspace_bytes(N, f)) - 1
        for call in (wavelet, adjoint, adjoint_all):
            refused((call.__name__, f), call(lib, f=f, ws_bytes=short))
    short = int(lib.egnn_row_order_ws_bytes(N)) - 1
    refused("row_order", lib.egnn_row_order(ok(1), N, ok(2), ok(3), short, None))
    short = int(lib.egnn_cheb_coeff_grad_ws_bytes(3, 2)) - 1
    refused("coeff_grad", lib.egnn_cheb_coeff_grad(ok(1), ok(2), N, 4, 3, 2, ok(3), ok(4), short, None))
    short = int(lib.egnn_csr_transpose_ws_bytes(N, 16)) - 1
    refused("csr_transpose", lib.egnn_csr_transpose(ok(1), ok(2), None, N, 16, ok(3), ok(4), None, ok(5), short, None))
    short = int(lib.egnn_adj_grad_degree_ws_bytes(N)) - 1
    refused("adj_grad_degree", lib.egnn_adj_grad_degree(ok(1), ok(2), None, ok(3), ok(4), None, ok(5), ok(6), N, 16, 4,
                                                        3, 1.0, ok(7), ok(8), None, None, ok(9), ok(10), ok(11), short,
                                                        None))
    short = int(lib.egnn_sell_ws_bytes(N, 16, 1, 256)) - 1
    refused("sell_prepare", lib.egnn_sell_prepare(ok(1), ok(2), N, 16, C.byref(sell_plan(filled=False)), ok(3), short,
                                                  None))
    refused("sell_fill", lib.egnn_sell_fill(ok(1), ok(2), N, 16, C.byref(sell_plan()), ok(3), short, None))
    short = int(lib.egnn_calibration_metrics_ws_bytes(3, 10)) - 1
    refused("calibration_metrics", lib.egnn_calibration_metrics(ok(1), 0, ok(2), None, N, 3, 10, ok(3), ok(4), short,
                                                                None))
