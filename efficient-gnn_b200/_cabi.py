"""ctypes binding of ``lib/libegnn_b200.so`` (C ABI declared in include/egnn_b200.h).

There is deliberately no fallback: if the shared library is missing or the
device is not sm_100, every entry point raises.  Build it with
``python -c "import __graft_entry__ as g; g.build()"`` or
``efficient-gnn_b200/csrc/build.sh``.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EGNN_LIB_PATH") or os.path.join(_HERE, "lib", "libegnn_b200.so")   # override: tuning builds
ABI_VERSION = 13

# every symbol include/egnn_b200.h declares: name -> (restype, argtypes)
_P, _I32, _I64, _F32, _SZ = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t
SYMBOLS = {
    "egnn_abi_version": (C.c_int, []),
    "egnn_last_error": (C.c_char_p, []),
    "egnn_device_info": (C.c_int, [_P, _P, _P]),
    "egnn_dense_to_csr_count": (C.c_int, [_P, _I64, _I64, _P, _P, _P]),
    "egnn_dense_to_csr_fill": (C.c_int, [_P, _I64, _I64, _P, _P, _P, _P]),
    "egnn_graph_prep": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "egnn_degree_rows": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _P, _P, _P, _P, _P]),
    "egnn_graph_prep_finish": (C.c_int, [_P, _P, _P, _I64, _P, _P, _P, _P, _P]),
    "egnn_calibration_metrics_ws_bytes": (_SZ, [_I32, _I32]),
    "egnn_calibration_metrics": (C.c_int, [_P, _I32, _P, _P, _I64, _I32, _I32, _P, _P, _SZ, _P]),
    "egnn_temperature_head": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _I32, _P]),
    "egnn_gcn_propagate": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I64, _I32, _P, _P, _P, _I32, _P]),
    "egnn_gcn_target_logits": (C.c_int, [_P, _P, _P, _P, _P, _P, _I32, _I64, _I32, _I32, _P, _P, _P, _P, _P, _I32, _P]),
    "egnn_gcn_structure_grad": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I64, _I32, _I32, _P, _P,
                                          _P, _P, _P, _I32, _P]),
    "egnn_sell_geometry": (C.c_int, [_I64, _I64, _P, _P, _P]),
    "egnn_sell_ws_bytes": (_SZ, [_I64, _I64, _I32, _I32]),
    "egnn_sell_prepare": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _SZ, _P]),
    "egnn_sell_fill": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _SZ, _P]),
    "egnn_patch_degrees": (C.c_int, [_P, _P, _P, _P, _P, _I64, _P, _P, _P, _I32, _P, _P, _P, _I64, _I64, _P]),
    "egnn_patch_nodes": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _I32, _P, _P, _P, _P, _I32, _P]),
    "egnn_cheb_workspace_bytes": (_SZ, [_I64, _I32]),
    "egnn_cheb_wavelet": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, _I32, _P, _F32, _F32,
                                    _P, _P, _I32, _P, _P, _P, _I32, _P, _SZ, _P, _P, _P, _P, _P, _I32, _P, _P, _I32]),
    "egnn_cheb_adjoint": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, _I32, _P, _F32, _F32,
                                    _P, _P, _P, _P, _P, _P, _I32, _P, _SZ, _P, _P, _P]),
    "egnn_cheb_adjoint_all": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, _I32, _P, _F32, _F32,
                                        _P, _P, _P, _P, _P, _P, _I32, _P, _SZ, _P, _P, _P, _P]),
    "egnn_adj_grad_degree_ws_bytes": (_SZ, [_I64]),
    "egnn_adj_grad_degree": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, _F32, _P, _P, _P, _P,
                                       _P, _P, _P, _SZ, _P]),
    "egnn_adj_grad_degree_flips": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, _F32, _P, _P,
                                             _P, _P, _P, _P, _P, _I32, _P, _P, _P, _SZ, _P]),
    "egnn_adj_grad_pairs": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P, _P, _I64, _I32, _I32, _F32, _P, _P]),
    "egnn_adj_grad_dense": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _I32, _F32, _P, _I64, _P]),
    "egnn_l1_normalize": (C.c_int, [_P, _P, _I64, _I32, _P]),
    "egnn_l1_normalize_backward": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P]),
    "egnn_cheb_coeff_grad_ws_bytes": (_SZ, [_I32, _I32]),
    "egnn_cheb_coeff_grad": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P, _P, _SZ, _P]),
    "egnn_csr_transpose_ws_bytes": (_SZ, [_I64, _I64]),
    "egnn_csr_transpose": (C.c_int, [_P, _P, _P, _I64, _I64, _P, _P, _P, _P, _SZ, _P]),
    "egnn_row_order_ws_bytes": (_SZ, [_I64]),
    "egnn_row_order": (C.c_int, [_P, _I64, _P, _P, _SZ, _P]),
    "egnn_sell_step_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P,
                                         _F32, _F32, _I32, _P, _P, _P, _I32, _P, _P, _I32, _P, _P]),
    "egnn_peer_window_bytes": (_SZ, [_I64, _I32, _I32]),
    "egnn_peer_alloc": (C.c_int, [_SZ, _P, _P]),
    "egnn_peer_open": (C.c_int, [_P, _P]),
    "egnn_peer_close": (C.c_int, [_P]),
    "egnn_peer_free": (C.c_int, [_P]),
    "egnn_peer_operand": (_P, [_P, _I32]),
    "egnn_peer_error": (C.c_int, [_P, _P, _P]),
    "egnn_peer_wait_stats": (C.c_int, [_P, _P, _P, _I32, _P]),
    "egnn_peer_prescale_push": (C.c_int, [_P, _P, _I64, _I64, _I32, _P, _P]),
    "egnn_wide_order_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I32, _I32, _I32, _I32,
                                          _P, _F32, _F32, _I32, _P, _P, _P, _I32, _P, _P]),
    "egnn_prescale": (C.c_int, [_P, _P, _P, _I64, _I32, _I64, _P]),
    "egnn_graph_prep_sharded": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "egnn_cheb_order_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                          _I64, _I64, _I64, _I64, _I32, _I32, _I32, _I32, _P, _F32, _F32,
                                          _I32, _I32, _P, _P, _P, _I32, _P]),
    "egnn_cheb_adjoint_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                            _I64, _I64, _I64, _I64, _I32, _I32, _I32, _I32, _P, _F32, _F32, _I32,
                                            _P, _P, _P, _I32, _P]),
    "egnn_wide_adjoint_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I32, _I32, _I32, _I32,
                                            _P, _F32, _F32, _P, _P, _P, _I32, _P, _P]),
    "egnn_cheb_order_sharded_vals": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                               _I64, _I64, _I64, _I64, _I32, _I32, _I32, _I32, _P, _F32, _F32,
                                               _I32, _I32, _P, _P, _P, _I32, _P]),
    "egnn_cheb_adjoint_sharded_vals": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                                 _I64, _I64, _I64, _I64, _I32, _I32, _I32, _I32, _P, _F32, _F32,
                                                 _I32, _P, _P, _P, _I32, _P]),
    "egnn_wide_adjoint_sharded_all": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I32,
                                                _I32, _I32, _I32, _P, _F32, _F32, _P, _P, _P, _I32, _P, _P]),
    "egnn_adj_grad_stacks_sharded": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I64, _I64, _I32, _I32, _P, _P, _P]),
    "egnn_adj_grad_degree_sharded_ws_bytes": (_SZ, [_I64]),
    "egnn_adj_grad_degree_sharded": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _I32,
                                               _I32, _F32, _P, _P, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "egnn_adj_grad_entries_sharded": (C.c_int, [_P, _P, _I64, _I64, _I64, _I32, _P, _P, _P, _F32, _P, _P]),
    "egnn_adj_grad_degree_sharded_flips": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64,
                                                     _I32, _I32, _F32, _P, _P, _P, _P, _P, _P, _P, _I32, _P, _P,
                                                     _P, _P, _P, _SZ, _P]),
    "egnn_adj_grad_flips_sharded": (C.c_int, [_P, _P, _P, _I32, _P, _P, _P, _I64, _I64, _I64, _F32, _P, _P]),
}


class SellPlanStruct(C.Structure):
    """Mirror of ``egnn_sell_plan`` (include/egnn_b200.h)."""
    _fields_ = [("n", C.c_int32), ("n_blocks", C.c_int32), ("col_block", C.c_int32), ("lmax", C.c_int32),
                ("n_cols", C.c_int32), ("row0", C.c_int32), ("n_cta", C.c_int32), ("reserved", C.c_int32),
                ("n_slices", C.c_int64), ("n_vrows", C.c_int64), ("n_entries", C.c_int64), ("n_rowv", C.c_int64),
                ("slice_off", C.c_void_p), ("blk_slice_ptr", C.c_void_p), ("idx", C.c_void_p),
                ("rv_ptr", C.c_void_p), ("vslot", C.c_void_p), ("cta_info", C.c_void_p), ("vpart", C.c_void_p),
                ("sched", C.c_void_p), ("stamps", C.c_void_p), ("n_hub", C.c_int64), ("hub", C.c_void_p)]


MAX_RANKS = 16
IPC_HANDLE_BYTES = 64


class PeerWindowStruct(C.Structure):
    """Mirror of ``egnn_peer_window`` (include/egnn_b200.h)."""
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("rows_per", C.c_int64), ("f", C.c_int32),
                ("reserved", C.c_int32), ("base", C.c_void_p * MAX_RANKS)]


class EgnnError(RuntimeError):
    """A non-zero status from libegnn_b200 (message from egnn_last_error)."""


_lock = threading.Lock()
_lib = None


def load():
    """Load the shared library once; raise if it is absent (no CPU fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.isfile(LIB_PATH):
            raise EgnnError(
                f"{LIB_PATH} not found: the CUDA extension is required (there is no CPU "
                "fallback). Build it with efficient-gnn_b200/csrc/build.sh")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        got = lib.egnn_abi_version()
        if got != ABI_VERSION:
            raise EgnnError(f"libegnn_b200 ABI {got} != binding ABI {ABI_VERSION}; rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().egnn_last_error().decode("utf-8", "replace")
        raise EgnnError(f"{what or 'libegnn_b200'} failed (status {rc}): {msg}")


def ptr(t):
    """Device (or host) address of a tensor, or NULL for None."""
    return None if t is None else C.c_void_p(t.data_ptr())


def vec_ready(t):
    """``t`` as a contiguous float32 tensor whose data starts on a 16-byte boundary, copied only when
    needed.  The kernels read and write rows of ``F % 4 == 0`` values with 16-byte vector accesses;
    ``.contiguous()`` alone keeps a view at an odd element offset (``buf[1:1 + n * f].view(n, f)``,
    a slice of a ``torch.cat``), which the library refuses."""
    import torch
    t = t.to(torch.float32).contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def host_array(ctype, values):
    arr = (ctype * max(1, len(values)))(*values)
    return arr


def delta_args(deltas, transpose: bool = False):
    """Edge flips ``(rows, cols, vals)`` (or None) as the four flip arguments of the C ABI: three host
    arrays and the count.  ``transpose=True`` swaps rows and columns, for the adjoint of a pass."""
    d_rows, d_cols, d_vals = ([], [], []) if deltas is None else deltas
    if transpose:
        d_rows, d_cols = d_cols, d_rows
    return (host_array(C.c_int32, [int(v) for v in d_rows]), host_array(C.c_int32, [int(v) for v in d_cols]),
            host_array(C.c_float, [float(v) for v in d_vals]), len(d_rows))


_device_ok = {}


def require_device():
    """Fail loudly unless a B200-class device is current.  The answer is cached
    per device index (the query costs milliseconds)."""
    import torch
    if not torch.cuda.is_available():
        raise EgnnError("efficient-gnn-b200 needs a CUDA device (sm_100a); there is no CPU path")
    dev = torch.cuda.current_device()
    hit = _device_ok.get(dev)
    if hit is not None:
        return hit
    sm, major, minor = C.c_int32(0), C.c_int32(0), C.c_int32(0)
    check(load().egnn_device_info(C.byref(sm), C.byref(major), C.byref(minor)), "egnn_device_info")
    _device_ok[dev] = (sm.value, major.value, minor.value)
    return _device_ok[dev]


def current_stream():
    """Raw handle of torch's current CUDA stream on the current device, as the ``egnn_stream_t``
    argument of the C ABI.  ``torch.cuda.current_stream()`` costs ~15 us per call (device-index and
    availability lookups); the recompute loop makes three library calls per step, so the raw getter
    is used when this torch build has it."""
    import torch
    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:
        return C.c_void_p(raw(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
