"""Drop-in host side of the WATS wavelet-feature path (calibration/WATS.py).

Same names, positional signatures and defaults as the reference:

* ``compute_normalized_laplacian(adj)``            (calibration/WATS.py:24-27)
* ``chebyshev_polynomials(L, k, X0)``              (calibration/WATS.py:29-37)
* ``graph_wavelet_features(adj_matrix, k=3, s=0.8)`` (calibration/WATS.py:39-74)
* ``WATS(base_model, features, labels, adj, val_mask)`` (calibration/WATS.py:76-170)

New behaviour is keyword-only.  All arithmetic of the path runs in
libegnn_b200 (hand-written sm_100a CUDA behind a C ABI); this module is tensor
plumbing.  There is no CPU fallback: without the shared library or a CUDA
device every entry point raises ``EgnnError``.

``graph_wavelet_features``, ``chebyshev_polynomials`` and both operators'
``@`` are differentiable w.r.t. the signal (and the features w.r.t. a tensor
``s``): when grad mode is on and an input requires grad, the pass runs inside
an autograd function whose backward is the adjoint (Clenshaw) pass of
``egnn_cheb_adjoint``.  Otherwise nothing changes: same kernels, nothing saved.
``WATS``, ``WaveletSession`` and the sharded path stay forward-only.
"""
from __future__ import annotations

import ctypes as C
import time

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.autograd.function import once_differentiable

from . import _cabi
from .graph import CsrGraph, as_graph, deltas_from_dense

__all__ = ["LaplacianOperator", "ExplicitOperator", "compute_normalized_laplacian", "chebyshev_polynomials",
           "graph_wavelet_features", "heat_coefficients", "WaveletResult", "WaveletSession", "WATS", "accuracy"]


def _stream():
    return _cabi.current_stream()


WIDE_MIN_F = 8       # signals at least this wide run on the wide-row kernel (csrc/wide.cuh)


def heat_coefficients(k: int, s) -> np.ndarray:
    """``alpha[j, i] = exp(-s_j * i)`` (calibration/WATS.py:65), float64 on the
    host, rounded to float32 when handed to the kernel."""
    s = np.atleast_1d(np.asarray(s, dtype=np.float64))
    return np.exp(-s[:, None] * np.arange(k + 1, dtype=np.float64)[None, :])


class WaveletResult:
    """Outputs of one fused pass: ``features`` ``[N, S*F]`` (what the reference
    returns), plus the pre-normalisation pieces parity checks need."""

    def __init__(self, features, orders=None, combined=None):
        self.features = features
        self.orders = orders          # list of K+1 [N,F] tensors or None
        self.combined = combined      # [N, S, F] un-normalised S or None


def _run_cheb(graph: CsrGraph, x0: torch.Tensor, k: int, coeffs: np.ndarray, op_scale: float,
              op_shift: float, normalize: bool, want_orders: bool, deltas=None,
              degree_vectors=None, order_events=None, use_sell=None, default_signal=False, y0=None,
              patch_in_kernel=False):
    """One call of egnn_cheb_wavelet.  Returns (out [N,S,F], t_all or None).
    ``default_signal``: x0 is the graph's own log1p(degree) with its own degree
    vectors, so the first operand dinv * x0 is the one cached on the graph; ``y0``: that
    operand supplied by the caller (patched copy of the cached one, UGCA recompute).
    ``patch_in_kernel``: ``deltas`` come with the BASE graph's vectors; on the SELL plan path the
    step kernel re-derives the touched nodes itself (one launch per perturbed pass) - callers
    check :func:`_patches_in_kernel` first."""
    lib = _cabi.load()
    n, dev = graph.n, graph.device
    if x0.dim() == 1:
        x0 = x0.unsqueeze(1)
    if x0.shape[0] != n:
        raise ValueError(f"X0 has {x0.shape[0]} rows, graph has {n} nodes")
    x0 = _cabi.vec_ready(x0.detach().to(device=dev))
    f = int(x0.shape[1])
    n_scales = int(coeffs.shape[0])
    if coeffs.shape[1] != k + 1:
        raise ValueError("coeffs must be [S, K+1]")
    dinv, iso = (graph.dinv, graph.iso) if degree_vectors is None else degree_vectors
    d_rows, d_cols, d_vals = ([], [], []) if deltas is None else deltas
    plan = None
    blocked = 0                   # plan-free column-blocked kernel (csrc/blocked.cuh): first use of a large graph
    if use_sell == "blocked":     # tests: force it whatever the size
        blocked = 2 if (f == 1 and graph.rows_sorted()) else 0
    elif f == 1 and k >= 1 and use_sell is not False:
        # The SELL re-layout costs about as much as 25 generic-kernel orders on the Reddit shape, so it is
        # built when a graph is used for the second time (calibrator construction computes the features
        # once; the UGCA recompute loop and benchmarks call again and again on the same graph).
        graph.narrow_calls += 1
        if use_sell or graph.narrow_calls >= 2 or graph.has_sell_plan():
            plan = graph.sell_plan(force=bool(use_sell))
        if plan is None and graph.rows_sorted():
            blocked = 1
    row_order = graph.row_order() if (f >= WIDE_MIN_F and k >= 1) else None
    with torch.cuda.device(dev):
        out = torch.empty((n, n_scales, f), dtype=torch.float32, device=dev)
        t_all = torch.empty((k + 1, n, f), dtype=torch.float32, device=dev) if want_orders else None
        ws_bytes = int(lib.egnn_cheb_workspace_bytes(n, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        coeffs32 = np.ascontiguousarray(coeffs, dtype=np.float32)
        _cabi.check(lib.egnn_cheb_wavelet(
            _cabi.ptr(graph.rowptr), _cabi.ptr(graph.colidx), _cabi.ptr(graph.vals), _cabi.ptr(dinv),
            _cabi.ptr(iso), _cabi.ptr(x0), n, graph.nnz, f, k, n_scales,
            coeffs32.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift),
            _cabi.ptr(out), _cabi.ptr(t_all), 1 if normalize else 0,
            _cabi.host_array(C.c_int32, [int(v) for v in d_rows]),
            _cabi.host_array(C.c_int32, [int(v) for v in d_cols]),
            _cabi.host_array(C.c_float, [float(v) for v in d_vals]), len(d_rows),
            _cabi.ptr(ws), ws_bytes, _stream(), order_events,
            None if plan is None else C.byref(plan), _cabi.ptr(row_order),
            _cabi.ptr(y0 if y0 is not None else graph.y0()) if (plan is not None and (default_signal or y0 is not None)) else None,
            blocked,
            _cabi.ptr(graph.w) if patch_in_kernel else None, _cabi.ptr(graph.rowsum) if patch_in_kernel else None,
            1 if default_signal else 0), "egnn_cheb_wavelet")
    return out, t_all


def _run_adjoint(graph_t: CsrGraph, degree_vectors, k: int, coeffs: np.ndarray, op_scale: float, op_shift: float,
                 cbar: torch.Tensor, tbar=None, deltas=None, app_events=None) -> torch.Tensor:
    """One call of egnn_cheb_adjoint: the signal's gradient ``[N, F]`` from ``cbar`` ``[N, S, F]`` (and
    ``tbar`` ``[K+1, N, F]``).  ``graph_t``: the transposed graph (:meth:`CsrGraph.adjoint`),
    ``degree_vectors``: the forward's ``(dinv, iso)``, ``deltas``: the forward's flips, not yet
    transposed."""
    lib = _cabi.load()
    n, f, dev = graph_t.n, int(cbar.shape[2]), graph_t.device
    dinv, iso = degree_vectors
    d_rows, d_cols, d_vals = ([], [], []) if deltas is None else deltas
    row_order = graph_t.row_order() if (f >= WIDE_MIN_F and k >= 1) else None
    with torch.cuda.device(dev):
        xbar = torch.empty((n, f), dtype=torch.float32, device=dev)
        ws_bytes = int(lib.egnn_cheb_workspace_bytes(n, f))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        coeffs32 = np.ascontiguousarray(coeffs, dtype=np.float32)
        _cabi.check(lib.egnn_cheb_adjoint(
            _cabi.ptr(graph_t.rowptr), _cabi.ptr(graph_t.colidx), _cabi.ptr(graph_t.vals), _cabi.ptr(dinv),
            _cabi.ptr(iso), n, graph_t.nnz, f, k, int(coeffs.shape[0]), coeffs32.ctypes.data_as(C.c_void_p),
            float(op_scale), float(op_shift), _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(xbar),
            _cabi.host_array(C.c_int32, [int(v) for v in d_cols]),       # transposed flips: rows <-> cols
            _cabi.host_array(C.c_int32, [int(v) for v in d_rows]),
            _cabi.host_array(C.c_float, [float(v) for v in d_vals]), len(d_rows),
            _cabi.ptr(ws), ws_bytes, _stream(), app_events, _cabi.ptr(row_order)), "egnn_cheb_adjoint")
    return xbar


def _coeff_grad(cbar: torch.Tensor, t_all: torch.Tensor) -> torch.Tensor:
    """``G[s, k] = <cbar[:, s, :], T_k>`` in float64 on the device (egnn_cheb_coeff_grad)."""
    lib = _cabi.load()
    n, n_scales, f = cbar.shape
    k = int(t_all.shape[0]) - 1
    with torch.cuda.device(cbar.device):
        g = torch.empty((n_scales, k + 1), dtype=torch.float64, device=cbar.device)
        ws_bytes = int(lib.egnn_cheb_coeff_grad_ws_bytes(k, n_scales))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cbar.device)
        _cabi.check(lib.egnn_cheb_coeff_grad(_cabi.ptr(cbar), _cabi.ptr(t_all), n, f, k, n_scales, _cabi.ptr(g),
                                             _cabi.ptr(ws), ws_bytes, _stream()), "egnn_cheb_coeff_grad")
    return g


class _PassSpec:
    """Everything of one pass but its differentiable inputs (the signal and the scales)."""

    def __init__(self, graph, adjoint, k, coeffs, op_scale, op_shift, want_orders, deltas=None, degree_vectors=None,
                 use_sell=None, default_signal=False, y0=None):
        self.graph, self.adjoint, self.k, self.coeffs = graph, adjoint, k, coeffs
        self.op_scale, self.op_shift, self.want_orders = op_scale, op_shift, want_orders
        self.deltas, self.degree_vectors, self.use_sell = deltas, degree_vectors, use_sell
        self.default_signal, self.y0 = default_signal, y0


class _WaveletPass(torch.autograd.Function):
    """``(C [N,S,F], T [K+1,N,F])`` of one un-normalised pass as a function of the signal ``x0`` and
    the scales ``s`` (a tensor, or None when they need no gradient).  ``T`` is empty unless the
    orders are wanted or ``s`` needs a gradient (its backward reads them).  Backward: the adjoint
    pass on the transposed graph, and ``ds_j = -sum_k k alpha[j,k] <Cbar_j, T_k>``."""

    @staticmethod
    def forward(ctx, x0, s, spec):
        ctx.set_materialize_grads(False)        # an output nobody differentiates arrives as None
        s_grad = s is not None and ctx.needs_input_grad[1]
        comb, t_all = _run_cheb(spec.graph, x0, spec.k, spec.coeffs, spec.op_scale, spec.op_shift, False,
                                spec.want_orders or s_grad, spec.deltas, spec.degree_vectors, use_sell=spec.use_sell,
                                default_signal=spec.default_signal, y0=spec.y0)
        if t_all is None:
            t_all = comb.new_empty((0,))
            ctx.mark_non_differentiable(t_all)
        ctx.spec, ctx.x_shape = spec, x0.shape
        ctx.s_meta = None if s is None else (s.shape, s.device, s.dtype)
        ctx.save_for_backward(t_all if s_grad else None)
        return comb, t_all

    @staticmethod
    @once_differentiable
    def backward(ctx, g_comb, g_orders):
        spec = ctx.spec
        (t_all,) = ctx.saved_tensors
        g = spec.graph
        n_scales = int(spec.coeffs.shape[0])
        f = 1 if len(ctx.x_shape) == 1 else int(ctx.x_shape[1])
        cbar = (_cabi.vec_ready(g_comb) if g_comb is not None else
                torch.zeros((g.n, n_scales, f), dtype=torch.float32, device=g.device))
        tbar = _cabi.vec_ready(g_orders) if (g_orders is not None and g_orders.numel()) else None
        x_grad = s_grad = None
        if ctx.needs_input_grad[0]:
            dv = spec.degree_vectors if spec.degree_vectors is not None else (g.dinv, g.iso)
            x_grad = _run_adjoint(spec.adjoint(), dv, spec.k, spec.coeffs, spec.op_scale, spec.op_shift, cbar, tbar,
                                  spec.deltas).reshape(ctx.x_shape)
        if ctx.needs_input_grad[1]:
            G = _coeff_grad(cbar, t_all)
            alpha = torch.from_numpy(np.ascontiguousarray(spec.coeffs, dtype=np.float64)).to(G.device)
            kk = torch.arange(spec.k + 1, dtype=torch.float64, device=G.device)
            shape, dev, dtype = ctx.s_meta
            s_grad = (-(kk * alpha * G).sum(dim=1)).to(device=dev, dtype=dtype).reshape(shape)
        return x_grad, s_grad, None


class _L1Normalize(torch.autograd.Function):
    """``H = C / (sum_f |C| + 1e-8)`` per (row, scale) out of place, backward by egnn_l1_normalize_backward
    (``r`` recomputed from ``C``)."""

    @staticmethod
    def forward(ctx, comb):
        h = torch.empty_like(comb)
        n_vec = comb.shape[0] * comb.shape[1]
        with torch.cuda.device(comb.device):
            _cabi.check(_cabi.load().egnn_l1_normalize(_cabi.ptr(comb), _cabi.ptr(h), n_vec, comb.shape[2], _stream()),
                        "egnn_l1_normalize")
        ctx.save_for_backward(comb)
        return h

    @staticmethod
    @once_differentiable
    def backward(ctx, g_h):
        (comb,) = ctx.saved_tensors
        g_h = _cabi.vec_ready(g_h)
        cbar = torch.empty_like(comb)
        n_vec = comb.shape[0] * comb.shape[1]
        with torch.cuda.device(comb.device):
            _cabi.check(_cabi.load().egnn_l1_normalize_backward(_cabi.ptr(comb), _cabi.ptr(g_h), None, _cabi.ptr(cbar),
                                                                n_vec, comb.shape[2], _stream()),
                        "egnn_l1_normalize_backward")
        return cbar


def _needs_grad(x0, s=None) -> bool:
    """The autograd path engages only in grad mode with an input that requires grad."""
    return torch.is_grad_enabled() and (x0.requires_grad or (isinstance(s, torch.Tensor) and s.requires_grad))


def _differentiable_pass(spec: _PassSpec, x0: torch.Tensor, s=None):
    """``(C, T)`` through :class:`_WaveletPass`; the device / dtype conversion of ``x0`` stays outside
    the function, so autograd routes the gradient back to a CPU or float64 leaf."""
    x0 = x0.to(device=spec.graph.device, dtype=torch.float32)
    return _WaveletPass.apply(x0, s if (isinstance(s, torch.Tensor) and s.requires_grad) else None, spec)


def _patches_in_kernel(graph: CsrGraph, f: int, k: int, use_sell) -> bool:
    """Will a perturbed pass of this shape run on the SELL plan (whose kernel applies the degree
    patches of the flips itself)?  Mirrors the plan choice of :func:`_run_cheb`."""
    if f != 1 or k < 1 or use_sell is False or use_sell == "blocked":
        return False
    if use_sell or graph.narrow_calls >= 1 or graph.has_sell_plan():
        return graph.sell_plan(force=bool(use_sell)) is not None
    return False


class LaplacianOperator:
    """``scale * L_sym + shift * I`` of a device graph, never materialised.

    What ``compute_normalized_laplacian`` returns (scale 1, shift 0).  It
    supports exactly the algebra the reference applies to scipy's Laplacian -
    ``(2 / lambda_max) * L - identity(N)`` (calibration/WATS.py:55), ``2 * L``
    and ``L @ X`` (calibration/WATS.py:34,36) - so the reference's own function
    bodies run unchanged on it.
    """

    def __init__(self, graph: CsrGraph, scale: float = 1.0, shift: float = 0.0):
        self.graph = graph
        self.scale = float(scale)
        self.shift = float(shift)
        self.shape = (graph.n, graph.n)

    def __rmul__(self, c):
        return LaplacianOperator(self.graph, self.scale * float(c), self.shift * float(c))

    __mul__ = __rmul__

    @staticmethod
    def _identity_multiple(other, n):
        """c such that other == c * I_n, for scipy / numpy / torch identities."""
        try:
            import scipy.sparse as sp
            if sp.issparse(other):
                if other.shape != (n, n):
                    raise ValueError("shape mismatch")
                o = other.tocoo()
                d = other.diagonal()
                if np.any(o.row[o.data != 0] != o.col[o.data != 0]) or not np.all(d == d[0]):
                    raise ValueError("only multiples of the identity can be added to the operator")
                return float(d[0])
        except ImportError:   # pragma: no cover
            pass
        raise TypeError("only multiples of a scipy identity can be added to the operator")

    def __sub__(self, other):
        return LaplacianOperator(self.graph, self.scale, self.shift - self._identity_multiple(other, self.graph.n))

    def __add__(self, other):
        return LaplacianOperator(self.graph, self.scale, self.shift + self._identity_multiple(other, self.graph.n))

    def __matmul__(self, x):
        """One operator application through the fused kernel (order-1 pass); differentiable
        w.r.t. ``x`` (backward: one application of the transposed operator)."""
        xt = torch.as_tensor(x)
        vec = xt.dim() == 1
        coeffs = np.array([[0.0, 1.0]])
        if _needs_grad(xt):
            out, _ = _differentiable_pass(_PassSpec(self.graph, self.graph.adjoint, 1, coeffs, self.scale, self.shift,
                                                    False), xt)
        else:
            out, _ = _run_cheb(self.graph, xt, 1, coeffs, self.scale, self.shift, False, False)
        y = out[:, 0, :]
        return y[:, 0] if vec else y

    def rescaled(self, lambda_max: float = 2.0) -> "LaplacianOperator":
        """``(2/lambda_max) * L - I`` (calibration/WATS.py:55)."""
        c = 2.0 / float(lambda_max)
        return LaplacianOperator(self.graph, self.scale * c, self.shift * c - 1.0)


def compute_normalized_laplacian(adj) -> LaplacianOperator:
    """``L_sym = I - D^-1/2 A D^-1/2`` with scipy's ``csgraph.laplacian(adj,
    normed=True)`` semantics (calibration/WATS.py:24-27), as an implicit
    device operator: CSR adjacency + degree vectors, no materialised L."""
    return LaplacianOperator(as_graph(adj))


class ExplicitOperator:
    """An explicit sparse matrix (what the reference hands to ``chebyshev_polynomials``: the scipy
    ``L_rescaled`` of calibration/WATS.py:55) as a device operator.  The off-diagonal entries go
    through the same fused kernels as a weighted CSR (unit normaliser, no implicit diagonal), the
    stored diagonal is applied as a per-row scale; entries are rounded to float32.  ``@`` is
    differentiable w.r.t. its operand; the backward gathers over the transposed off-diagonal part,
    built on first use (the matrix is not assumed symmetric: scipy's two float32 divisions make the
    rescaled Laplacian asymmetric in the last bit)."""

    def __init__(self, mat):
        import scipy.sparse as sp
        m = sp.csr_matrix(mat, copy=True)
        if m.shape[0] != m.shape[1]:
            raise ValueError("operator must be square")
        m.sum_duplicates()
        m.sort_indices()
        n = m.shape[0]
        diag = np.asarray(m.diagonal(), dtype=np.float32)
        off = (m - sp.diags(m.diagonal(), format="csr")).tocsr()
        off.eliminate_zeros()
        off.sort_indices()
        _cabi.require_device()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.graph = CsrGraph(torch.from_numpy(off.indptr.astype(np.int32)).to(dev),
                              torch.from_numpy(off.indices.astype(np.int32)).to(dev),
                              torch.from_numpy(off.data.astype(np.float32)).to(dev), n)
        self.diag = torch.from_numpy(diag).to(dev)
        self.unit = (torch.ones(n, dtype=torch.float32, device=dev), torch.ones(n, dtype=torch.uint8, device=dev))
        self.shape = (n, n)
        self._off = off
        self._transposed = None

    def _transpose(self) -> CsrGraph:
        if self._transposed is None:
            t = self._off.T.tocsr()
            t.sort_indices()
            dev = self.diag.device
            self._transposed = CsrGraph(torch.from_numpy(t.indptr.astype(np.int32)).to(dev),
                                        torch.from_numpy(t.indices.astype(np.int32)).to(dev),
                                        torch.from_numpy(t.data.astype(np.float32)).to(dev), self.shape[0])
        return self._transposed

    def __matmul__(self, x):
        xt = torch.as_tensor(x)
        vec = xt.dim() == 1
        xt = (xt.unsqueeze(1) if vec else xt).to(device=self.diag.device, dtype=torch.float32)
        # kernel: theta * x - a * dinv_i * sum_{j != i} v_ij dinv_j x_j with a = -1, dinv = 1, theta = 0
        coeffs = np.array([[0.0, 1.0]])
        if _needs_grad(xt):
            out, _ = _differentiable_pass(_PassSpec(self.graph, self._transpose, 1, coeffs, -1.0, 0.0, False,
                                                    degree_vectors=self.unit, use_sell=False), xt)
        else:
            out, _ = _run_cheb(self.graph, xt, 1, coeffs, -1.0, 0.0, False, False,
                               degree_vectors=self.unit, use_sell=False)
        y = out[:, 0, :] + self.diag.unsqueeze(1) * xt
        return y[:, 0] if vec else y


def chebyshev_polynomials(L, k, X0):
    """``[T_0 .. T_k]`` with ``T_1 = L X0``, ``T_i = 2 L T_{i-1} - T_{i-2}``
    (calibration/WATS.py:29-37).  ``L`` is a :class:`LaplacianOperator` (what
    ``compute_normalized_laplacian`` returns, normally rescaled: all orders in the
    fused kernels) or an explicit scipy sparse matrix as in the reference (one
    kernel application per order); returns k+1 float32 device tensors ``[N,F]``,
    differentiable w.r.t. ``X0`` when it requires grad."""
    k = int(k)
    if not isinstance(L, LaplacianOperator):
        try:
            import scipy.sparse as sp
            explicit = sp.issparse(L)
        except ImportError:       # pragma: no cover
            explicit = False
        if not explicit:
            raise TypeError("L must be a LaplacianOperator (compute_normalized_laplacian) or a scipy sparse matrix")
        op = ExplicitOperator(L)
        x0 = torch.as_tensor(X0)
        x0 = (x0.unsqueeze(1) if x0.dim() == 1 else x0).to(device=op.diag.device, dtype=torch.float32)
        t_k = [x0]
        if k > 0:
            t_k.append(op @ x0)
        for _ in range(2, k + 1):
            t_k.append(2 * (op @ t_k[-1]) - t_k[-2])
        return t_k
    coeffs = np.zeros((1, k + 1))
    x0 = torch.as_tensor(X0)
    if _needs_grad(x0):
        _, t_all = _differentiable_pass(_PassSpec(L.graph, L.graph.adjoint, k, coeffs, L.scale, L.shift, True), x0)
    else:
        _, t_all = _run_cheb(L.graph, x0, k, coeffs, L.scale, L.shift, False, True)
    return [t_all[i] for i in range(k + 1)]


def graph_wavelet_features(adj_matrix, k=3, s=0.8, *, X0=None, lambda_max: float = 2.0,
                           normalize: bool = True, return_parts: bool = False, deltas=None,
                           _order_events=None, _use_sell=None):
    """Graph wavelet features by Chebyshev approximation of the heat kernel
    (calibration/WATS.py:39-74).

    Positional behaviour is the reference's: ``X0 = log1p(degree)``, ``k = 3``,
    one scale ``s = 0.8``, ``lambda_max = 2``, row-L1-normalised ``[N, F]``.
    Keyword-only extensions: ``s`` may be a sequence (all scales accumulated in
    the same pass, output ``[N, len(s)*F]``); ``X0`` a custom ``[N,F]`` signal;
    ``lambda_max``; ``return_parts`` -> :class:`WaveletResult` with the orders
    and the un-normalised combination; ``deltas=(rows, cols, vals)`` applies
    edge flips on top of the graph without rebuilding it (UGCA recompute).
    Returns a float32 tensor on the graph's device.

    Differentiable w.r.t. ``X0`` and a 0-d / 1-d tensor ``s`` (coefficients are
    computed from its values as for a float) when grad mode is on and one of
    them requires grad: every output (``features``, ``combined``, ``orders``)
    then carries a ``grad_fn``; ``deltas=`` is supported.  The forward then keeps
    the un-normalised combination and normalises out of place.
    """
    graph = as_graph(adj_matrix)
    k = int(k)
    s_vals = s.detach().cpu().numpy() if isinstance(s, torch.Tensor) else s
    coeffs = heat_coefficients(k, s_vals)
    degree_vectors = None
    x0 = graph.x0 if X0 is None else torch.as_tensor(X0)
    grad = _needs_grad(x0, s)
    y0 = None
    in_kernel = False
    if deltas is not None and len(deltas[0]) > 0:
        # the backward needs the patched degree vectors, so a differentiable pass patches them itself
        in_kernel = not grad and _patches_in_kernel(graph, 1 if x0.dim() == 1 else int(x0.shape[1]), k, _use_sell)
        if not in_kernel:
            # degree vectors of the flipped graph: only the touched entries of persistent scratch copies are
            # written, and put back once the pass is queued (no copies of the N-vectors per perturbation)
            dinv, iso, x0_patched, y0_patched = graph.patch_nodes(deltas)
            degree_vectors = (dinv, iso)
            if X0 is None:
                x0, y0 = x0_patched, y0_patched
        # else (SELL plan): the step kernel re-derives the touched nodes from the base vectors - one launch
    else:
        deltas = None
    op_scale = 2.0 / float(lambda_max)
    default_signal = X0 is None and (deltas is None or in_kernel)
    try:
        if grad:
            if degree_vectors is not None:       # the scratch vectors are restored below, the backward runs later
                degree_vectors = tuple(v.clone() for v in degree_vectors)
            spec = _PassSpec(graph, graph.adjoint, k, coeffs, op_scale, -1.0, return_parts, deltas, degree_vectors,
                             _use_sell, default_signal, y0)
            comb, t_all = _differentiable_pass(spec, x0, s)
            feats = _L1Normalize.apply(comb) if normalize else comb
            feats = feats.reshape(graph.n, -1)
            return WaveletResult(feats, [t_all[i] for i in range(k + 1)], comb) if return_parts else feats
        return _wavelet_pass(graph, x0, k, coeffs, op_scale, normalize, return_parts, deltas, degree_vectors,
                             _order_events, _use_sell, default_signal, y0, in_kernel)
    finally:
        if deltas is not None and not in_kernel:
            graph.patch_nodes(deltas, restore=True)


def _wavelet_pass(graph, x0, k, coeffs, op_scale, normalize, return_parts, deltas, degree_vectors, _order_events,
                  _use_sell, default_signal, y0, patch_in_kernel=False):
    if return_parts:
        comb, t_all = _run_cheb(graph, x0, k, coeffs, op_scale, -1.0, False, True, deltas, degree_vectors,
                                use_sell=_use_sell, default_signal=default_signal, y0=y0,
                                patch_in_kernel=patch_in_kernel)
        feats = comb / (comb.abs().sum(dim=2, keepdim=True) + 1e-8) if normalize else comb
        feats = feats.reshape(graph.n, -1)
        return WaveletResult(feats, [t_all[i] for i in range(k + 1)], comb)
    out, _ = _run_cheb(graph, x0, k, coeffs, op_scale, -1.0, normalize, False, deltas, degree_vectors,
                       _order_events, _use_sell, default_signal, y0, patch_in_kernel)
    return out.reshape(graph.n, -1)


def accuracy(outputs, labels):
    """Fraction of argmax hits (calibration/utils.py:139-167)."""
    if not isinstance(outputs, torch.Tensor) or not isinstance(labels, torch.Tensor):
        raise ValueError("Input arrays must be of type torch.Tensor.")
    if outputs.shape[0] != labels.shape[0]:
        raise ValueError("Input arrays must have the same number of elements.")
    return (torch.sum(torch.argmax(outputs, dim=1) == labels) / labels.shape[0]).item()


class WATS(nn.Module):
    """Wavelet-Aware Temperature Scaling (calibration/WATS.py:76-170).

    Same constructor, attributes (``wavelet_feats`` stays a plain attribute,
    not a buffer, so ``state_dict`` keys match the reference), ``forward`` and
    ``calib_train``.  The only difference on the default path is where
    ``wavelet_feats`` comes from: dense adjacency -> CSR -> fused Chebyshev
    kernels on the device instead of the host scipy detour (WATS.py:99-100).

    Keyword-only extensions: ``k``, ``s``, ``lambda_max`` (reference constants
    3 / 0.8 / 2.0), ``recompute_on_forward`` (recompute the features from the
    ``adj`` passed to ``forward`` - the reference always reuses the cached
    ones, WATS.py:123), ``train`` (skip ``calib_train`` when False), ``verbose``,
    ``fused_head`` (under ``torch.no_grad()`` the temperature MLP, the scaling
    and the log_softmax of WATS.py:123-130 run as one kernel; autograd paths
    keep the reference's torch ops).
    ``_features_override`` exists for parity tests only: it injects a feature
    matrix computed elsewhere so two instances differ in nothing else.
    The wavelet features are an input here, computed without gradients
    (forward-only, as in the reference).
    """

    def __init__(self, base_model, features, labels, adj, val_mask, *, k: int = 3, s=0.8,
                 lambda_max: float = 2.0, recompute_on_forward: bool = False, train: bool = True,
                 verbose: bool = True, fused_head: bool = True, _features_override=None):
        super().__init__()
        self.device = torch.device('cuda' if torch.cuda.is_available() else 'cpu')
        if _features_override is None:
            _cabi.require_device()
        self.base_model = base_model.to(self.device)
        self.x = features.to(self.device)
        self.y = labels.to(self.device)
        self.adj = adj.to(self.device)
        self.val_idx = val_mask.to(self.device)
        self.k, self.s, self.lambda_max = int(k), s, float(lambda_max)
        self.recompute_on_forward = bool(recompute_on_forward)
        self.verbose = bool(verbose)
        self.fused_head = bool(fused_head)

        if _features_override is not None:
            self.graph = None
            self.wavelet_feats = torch.as_tensor(_features_override, dtype=torch.float32).to(self.device)
        else:
            self.graph = as_graph(self.adj)
            self.wavelet_feats = graph_wavelet_features(self.graph, k=self.k, s=self.s,
                                                        lambda_max=self.lambda_max)
        self.net = nn.Sequential(
            nn.Linear(self.wavelet_feats.shape[1], 16),
            nn.ReLU(),
            nn.Linear(16, 1)
        ).to(self.device)
        for para in self.net.parameters():
            para.requires_grad = True
        if train:
            self.calib_train()

    def features_for(self, adj=None, *, deltas=None):
        """Wavelet features of a perturbed graph: either a full adjacency
        (re-converted on the device) or edge flips on top of the base graph
        (``deltas=(rows, cols, vals)``; no CSR rebuild)."""
        if deltas is not None:
            return graph_wavelet_features(self.graph, k=self.k, s=self.s, lambda_max=self.lambda_max,
                                          deltas=deltas)
        if adj is None:
            return self.wavelet_feats
        # a dense adjacency that differs from the calibrator's own in a few entries (what the attack
        # passes: calib_fga.py:897-908): take the flips and keep the resident graph and its plan
        if isinstance(adj, torch.Tensor) and adj.layout == torch.strided and self.graph is not None \
                and isinstance(self.adj, torch.Tensor) and adj.shape == self.adj.shape:
            flips = deltas_from_dense(self.adj, adj.to(self.adj.device))
            if flips is not None:
                if not flips[0]:
                    return self.wavelet_feats
                return graph_wavelet_features(self.graph, k=self.k, s=self.s, lambda_max=self.lambda_max,
                                              deltas=flips)
        return graph_wavelet_features(adj, k=self.k, s=self.s, lambda_max=self.lambda_max)

    def temperatures(self, wavelet_features):
        t = self.net(wavelet_features).squeeze()
        return torch.log(torch.exp(t) + torch.tensor(1.1, device=self.device)).to(self.device)

    def _fused_head(self, wavelet_features, logits):
        """MLP -> temperature -> scaled log_softmax in one kernel (egnn_temperature_head).
        Forward only: used when autograd is off and everything already sits on the GPU."""
        lin1, lin2 = self.net[0], self.net[2]
        feats = wavelet_features.detach().to(torch.float32).contiguous()
        logits = logits.detach().to(torch.float32).contiguous()
        out = torch.empty_like(logits)
        with torch.cuda.device(logits.device):
            _cabi.check(_cabi.load().egnn_temperature_head(
                _cabi.ptr(feats), _cabi.ptr(lin1.weight.detach().contiguous()), _cabi.ptr(lin1.bias.detach().contiguous()),
                _cabi.ptr(lin2.weight.detach().reshape(-1).contiguous()), _cabi.ptr(lin2.bias.detach().contiguous()),
                _cabi.ptr(logits), _cabi.ptr(out), None, logits.shape[0], feats.shape[1], lin1.out_features,
                logits.shape[1], _stream()), "egnn_temperature_head")
        return out

    def forward(self, x, adj, *, deltas=None):
        x, adj = x.to(self.device), adj.to(self.device)
        if deltas is not None:
            wavelet_features = self.features_for(deltas=deltas)
        elif self.recompute_on_forward and self.graph is not None:
            wavelet_features = self.features_for(adj)
        else:
            wavelet_features = self.wavelet_feats.to(x.device)
        logits = self.base_model(x, adj)
        if (self.fused_head and not torch.is_grad_enabled() and logits.is_cuda and logits.dim() == 2
                and wavelet_features.shape[1] <= 64 and self.net[0].out_features <= 64):
            return self._fused_head(wavelet_features, logits)
        temperatures = self.temperatures(wavelet_features)
        calibrated_logits = logits / temperatures.unsqueeze(1)
        return F.log_softmax(calibrated_logits, dim=1)

    def calib_train(self, patience=10):
        t = time.time()
        best_loss = float('inf')
        patience_counter = patience
        optimizer = torch.optim.Adam(self.net.parameters(), lr=0.01, weight_decay=5e-4)
        recompute, self.recompute_on_forward = self.recompute_on_forward, False
        try:
            for epoch in range(250):
                self.train()
                optimizer.zero_grad()
                output = self(self.x, self.adj)
                loss = F.nll_loss(output[self.val_idx], self.y[self.val_idx])
                loss.backward()
                optimizer.step()
                with torch.no_grad():
                    self.eval()
                    acc = accuracy(output[self.val_idx], self.y[self.val_idx])
                    if self.verbose:
                        print(f'epoch: {epoch}', f'loss_calibration: {loss.item():.4f}',
                              f'acc_calibration: {acc:.4f}', f'time: {time.time() - t:.4f}s')
                if loss < best_loss:
                    best_loss = loss
                    patience_counter = patience
                else:
                    patience_counter -= 1
                if patience_counter <= 0:
                    if self.verbose:
                        print(f'Early stopping at epoch {epoch}, best loss: {best_loss:.4f}')
                    break
        finally:
            self.recompute_on_forward = recompute


class WaveletSession:
    """A fixed-shape wavelet pass captured once into a CUDA graph and replayed.

    For small graphs the K order kernels are microseconds each and the pass is
    launch-latency-bound; for the row-sharded path every order adds an NCCL
    exchange and host-side orchestration.  Replaying one captured graph removes
    the per-launch host cost in both cases.  ``target`` is a :class:`CsrGraph`
    or a ``sharded.ShardedWavelet``; ``X0`` (optional) is copied into a static
    buffer before each replay.  The returned tensor is a static buffer that the
    next call overwrites.  Forward-only: a replay records no autograd graph.
    """

    def __init__(self, target, k=3, s=0.8, *, f: int = 1, lambda_max: float = 2.0, normalize: bool = True,
                 cuda_graph: bool = True, warmup: int = 3):
        self.target = target
        self.k, self.s, self.lambda_max, self.normalize = int(k), s, float(lambda_max), bool(normalize)
        self.sharded = hasattr(target, "features")
        dev = target.device
        rows = target.rows if self.sharded else target.n
        self.x0 = None if f == 1 else torch.zeros((rows, f), dtype=torch.float32, device=dev)
        self.graph = None
        self.out = None
        if not cuda_graph:
            return
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(1, warmup)):
                self._pass()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = self._pass()

    def _pass(self):
        if self.sharded:
            return self.target.features(k=self.k, s=self.s, X0_local=self.x0, lambda_max=self.lambda_max,
                                        normalize=self.normalize)
        return graph_wavelet_features(self.target, k=self.k, s=self.s, X0=self.x0, lambda_max=self.lambda_max,
                                      normalize=self.normalize)

    def __call__(self, X0=None):
        if X0 is not None:
            if self.x0 is None:
                raise ValueError("session was built for the default signal (f=1, X0 = log1p(degree))")
            self.x0.copy_(torch.as_tensor(X0), non_blocking=True)
        if self.graph is None:
            return self._pass()
        self.graph.replay()
        return self.out
