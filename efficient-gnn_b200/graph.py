"""Device-resident graph for the wavelet path: CSR adjacency + the degree
vectors that stand in for the (never materialised) normalised Laplacian.

Replaces the reference's host-side detour ``csr_matrix(adj.cpu().numpy())``
(calibration/WATS.py:99) and ``csgraph.laplacian`` (calibration/WATS.py:26).
All arithmetic happens in libegnn_b200 kernels; torch is used for allocation,
streams and (for inputs that are not already a dense device tensor) format
plumbing.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np
import torch

from . import _cabi

__all__ = ["CsrGraph", "as_graph", "deltas_from_dense", "enable_phase_stamps", "read_phase_stamps"]


def _stream():
    return _cabi.current_stream()


class CsrGraph:
    """CSR adjacency in HBM plus ``dinv``/``iso``/``x0`` (scipy Laplacian
    semantics, see include/egnn_b200.h::egnn_graph_prep).

    ``vals is None`` means a binary adjacency (every reference call site).
    """

    def __init__(self, rowptr: torch.Tensor, colidx: torch.Tensor, vals: Optional[torch.Tensor], n: int,
                 _prepare: bool = True):
        _cabi.require_device()
        if rowptr.dtype != torch.int32 or colidx.dtype != torch.int32:
            raise TypeError("rowptr/colidx must be int32")
        if not (rowptr.is_cuda and colidx.is_cuda):
            raise _cabi.EgnnError("CsrGraph arrays must live on the CUDA device")
        if rowptr.numel() != n + 1:
            raise ValueError("rowptr must have n+1 entries")
        self.n = int(n)
        self.rowptr = rowptr.contiguous()
        self.colidx = colidx.contiguous()
        self.vals = None if vals is None else vals.to(torch.float32).contiguous()
        self.nnz = int(colidx.numel())
        if self.nnz >= 2 ** 31:
            raise ValueError("nnz must fit int32")
        self.device = rowptr.device
        self._alloc_vectors()
        if _prepare:
            self._prepare()

    # -- construction -------------------------------------------------------
    @classmethod
    def from_dense(cls, adj: torch.Tensor) -> "CsrGraph":
        """Dense ``[N,N]`` float32 device tensor -> CSR, entirely on the GPU
        (two streaming passes over the matrix; replaces WATS.py:99)."""
        _cabi.require_device()
        if adj.dim() != 2 or adj.shape[0] != adj.shape[1]:
            raise ValueError("adjacency must be square")
        adj = adj.detach()
        if not adj.is_cuda:
            adj = adj.to("cuda", non_blocking=True)
        if adj.dtype != torch.float32:
            adj = adj.to(torch.float32)
        if adj.stride(1) != 1:
            adj = adj.contiguous()
        n = adj.shape[0]
        lib = _cabi.load()
        with torch.cuda.device(adj.device):
            rowptr = torch.empty(n + 1, dtype=torch.int32, device=adj.device)
            flag = torch.empty(1, dtype=torch.int32, device=adj.device)
            _cabi.check(lib.egnn_dense_to_csr_count(_cabi.ptr(adj), n, adj.stride(0), _cabi.ptr(rowptr),
                                                    _cabi.ptr(flag), _stream()), "egnn_dense_to_csr_count")
            meta = torch.stack([rowptr[n], flag[0]]).cpu()       # one sync: nnz + binary flag
            nnz, nonbinary = int(meta[0]), bool(meta[1])
            colidx = torch.empty(nnz, dtype=torch.int32, device=adj.device)
            vals = torch.empty(nnz, dtype=torch.float32, device=adj.device) if nonbinary else None
            if nnz > 0:
                _cabi.check(lib.egnn_dense_to_csr_fill(_cabi.ptr(adj), n, adj.stride(0), _cabi.ptr(rowptr),
                                                       _cabi.ptr(colidx), _cabi.ptr(vals), _stream()),
                            "egnn_dense_to_csr_fill")
        return cls(rowptr, colidx, vals, n)

    @classmethod
    def from_host_csr(cls, rowptr, colidx, vals, n: int, device="cuda") -> "CsrGraph":
        """Host CSR buffers (int32 torch tensors, ideally pinned) -> device
        graph: asynchronous H2D copies on the current stream, then the degree
        pass.  This is the entry the host-buffer (end-to-end) timing uses."""
        _cabi.require_device()
        rp_h, ci_h = torch.as_tensor(rowptr), torch.as_tensor(colidx)
        vv_h = None if vals is None else torch.as_tensor(vals)
        nnz = int(ci_h.numel())
        pipelined = ci_h.is_pinned() and nnz >= cls.PIPELINE_MIN_NNZ and (vv_h is None or vv_h.is_pinned())
        if not pipelined:
            rp = rp_h.to(device, non_blocking=True)
            ci = ci_h.to(device, non_blocking=True)
            vv = None if vv_h is None else vv_h.to(device, non_blocking=True)
            return cls(rp, ci, vv, n)
        # Large pinned CSR: the entries are copied in row-aligned pieces on a side stream and the
        # degree pass of each piece runs as soon as it has landed, so only the last piece's pass is
        # left when the copy ends.
        dev = torch.device(device)
        lib = _cabi.load()
        with torch.cuda.device(dev):
            main = torch.cuda.current_stream()
            rp = rp_h.to(dev, non_blocking=True)
            ci = torch.empty(nnz, dtype=torch.int32, device=dev)
            vv = None if vv_h is None else torch.empty(nnz, dtype=torch.float32, device=dev)
            g = cls(rp, ci, vv, n, _prepare=False)
            g._colsum.zero_()
            g._unsorted_flag.zero_()
            # equal row counts per piece (no host-side search over rowptr before the first copy is issued)
            pieces = max(2, min(16, nnz // cls.PIPELINE_PIECE_NNZ))
            rows = sorted({(n * i) // pieces for i in range(pieces + 1)})
            copy = cls._copy_stream(dev)
            copy.wait_stream(main)
            for r0, r1 in zip(rows[:-1], rows[1:]):
                lo, hi = int(rp_h[r0]), int(rp_h[r1])
                with torch.cuda.stream(copy):
                    ci[lo:hi].copy_(ci_h[lo:hi], non_blocking=True)
                    if vv is not None:
                        vv[lo:hi].copy_(vv_h[lo:hi], non_blocking=True)
                    landed = torch.cuda.Event()
                    landed.record(copy)
                main.wait_event(landed)
                _cabi.check(lib.egnn_degree_rows(_cabi.ptr(rp), _cabi.ptr(ci), _cabi.ptr(vv), n, r0, r1,
                                                 _cabi.ptr(g.rowsum), _cabi.ptr(g._diag), _cabi.ptr(g._colsum),
                                                 _cabi.ptr(g._unsorted_flag), _stream()), "egnn_degree_rows")
            _cabi.check(lib.egnn_graph_prep_finish(_cabi.ptr(g._colsum), _cabi.ptr(g._diag), _cabi.ptr(g.rowsum), n,
                                                   _cabi.ptr(g.dinv), _cabi.ptr(g.iso), _cabi.ptr(g.x0), _cabi.ptr(g.w),
                                                   _stream()), "egnn_graph_prep_finish")
            g._release_scratch()
        return g

    PIPELINE_MIN_NNZ = 1 << 24        # below this one copy + one pass is as fast
    PIPELINE_PIECE_NNZ = 1 << 23      # ~32 MB of indices per piece
    _copy_streams = {}

    @classmethod
    def _copy_stream(cls, dev):
        key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
        if key not in cls._copy_streams:
            cls._copy_streams[key] = torch.cuda.Stream(device=dev)
        return cls._copy_streams[key]

    @classmethod
    def from_scipy(cls, mat, device="cuda") -> "CsrGraph":
        import scipy.sparse as sp
        m = sp.csr_matrix(mat, copy=True)      # never canonicalise the caller's arrays in place
        m.sum_duplicates()
        m.eliminate_zeros()
        m.sort_indices()
        data = np.asarray(m.data, dtype=np.float32)
        vals = None if np.all(data == 1.0) else torch.from_numpy(data).to(device)
        return cls(torch.from_numpy(m.indptr.astype(np.int32)).to(device),
                   torch.from_numpy(m.indices.astype(np.int32)).to(device), vals, m.shape[0])

    @classmethod
    def from_edge_index(cls, edge_index, n: int, edge_weight=None, device="cuda") -> "CsrGraph":
        """``(edge_index [2,E], N)``; duplicate edges are summed like scipy does."""
        ei = torch.as_tensor(edge_index).to(device=device, dtype=torch.int64)
        key = ei[0] * n + ei[1]
        if edge_weight is None:
            uniq, counts = torch.unique(key, return_counts=True)
            vals = None if bool((counts == 1).all()) else counts.to(torch.float32)
        else:
            w = torch.as_tensor(edge_weight).to(device=device, dtype=torch.float32)
            uniq, inv = torch.unique(key, return_inverse=True)
            vals = torch.zeros(uniq.numel(), dtype=torch.float32, device=device).index_add_(0, inv, w)
            keep = vals != 0
            uniq, vals = uniq[keep], vals[keep]
            if bool((vals == 1).all()):
                vals = None
        rows = uniq // n
        rowptr = torch.zeros(n + 1, dtype=torch.int64, device=device)
        rowptr[1:] = torch.cumsum(torch.bincount(rows, minlength=n), 0)
        return cls(rowptr.to(torch.int32), (uniq % n).to(torch.int32), vals, n)

    # -- degree vectors -----------------------------------------------------
    def _alloc_vectors(self):
        n, dev = self.n, self.device
        with torch.cuda.device(dev):
            self.dinv = torch.empty(n, dtype=torch.float32, device=dev)
            self.iso = torch.empty(n, dtype=torch.uint8, device=dev)
            self.x0 = torch.empty(n, dtype=torch.float32, device=dev)
            self.w = torch.empty(n, dtype=torch.float32, device=dev)
            self.rowsum = torch.empty(n, dtype=torch.float32, device=dev)
            self._diag = torch.empty(n, dtype=torch.float32, device=dev)
            self._colsum = torch.empty(n, dtype=torch.float64, device=dev)
            self._unsorted_flag = torch.empty(1, dtype=torch.int32, device=dev)
        self._sell = None          # lazily built SELL plan (False: not applicable)
        self._sell_structural = False   # the False above is final (weighted / unsorted / empty), not a threshold
        self.narrow_calls = 0      # F = 1 passes run on this graph (the plan is built on the second)
        self._row_order = None     # lazily built processing order of the wide kernel
        self._sorted = None        # lazily read result of the degree pass's sortedness check
        self._scratch = None       # lazily built scratch copies of dinv / iso / x0 / y0 for the in-place UGCA patches
        self._y0 = None            # lazily built dinv * x0 (first operand of the narrow path, default signal)
        self._adjoint = None       # lazily built transposed graph of the backward pass (False: symmetric)

    def _release_scratch(self):
        self._diag = self._colsum = None

    def _prepare(self):
        lib = _cabi.load()
        with torch.cuda.device(self.device):
            _cabi.check(lib.egnn_graph_prep(_cabi.ptr(self.rowptr), _cabi.ptr(self.colidx), _cabi.ptr(self.vals), self.n,
                                            _cabi.ptr(self.dinv), _cabi.ptr(self.iso), _cabi.ptr(self.x0),
                                            _cabi.ptr(self.w), _cabi.ptr(self.rowsum), _cabi.ptr(self._diag),
                                            _cabi.ptr(self._colsum), _cabi.ptr(self._unsorted_flag), _stream()),
                        "egnn_graph_prep")
        self._release_scratch()

    def rows_sorted(self) -> bool:
        """Every CSR row is sorted by column (checked by the degree pass; one
        4-byte D2H read on first use)."""
        if self._sorted is None:
            self._sorted = not bool(self._unsorted_flag.item())
        return self._sorted

    def y0(self):
        """``dinv * x0`` of the default signal: the first gather operand of the
        narrow path, fixed per graph (one small kernel on first use)."""
        if self._y0 is None:
            with torch.cuda.device(self.device):
                y = torch.empty(max(1, self.n), dtype=torch.float32, device=self.device)
                if self.n:
                    _cabi.check(_cabi.load().egnn_prescale(_cabi.ptr(self.x0), _cabi.ptr(self.dinv), _cabi.ptr(y), self.n, 1, 0,
                                                           _stream()), "egnn_prescale")
            self._y0 = y
        return self._y0

    def adjoint(self) -> "CsrGraph":
        """The graph the backward pass gathers over: ``self`` when the sorted CSR
        equals its transpose (every undirected graph), else the transposed
        adjacency carrying THIS graph's degree vectors (scipy normalises by the
        column sums on both sides of ``L``, so they are not re-derived from the
        transpose).  Built once on the device (one 1-byte host read)."""
        if self._adjoint is None:
            lib = _cabi.load()
            n, nnz = self.n, self.nnz
            with torch.cuda.device(self.device):
                rp = torch.empty(n + 1, dtype=torch.int32, device=self.device)
                ci = torch.empty(nnz, dtype=torch.int32, device=self.device)
                vv = None if self.vals is None else torch.empty(nnz, dtype=torch.float32, device=self.device)
                ws_bytes = int(lib.egnn_csr_transpose_ws_bytes(n, nnz))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
                _cabi.check(lib.egnn_csr_transpose(_cabi.ptr(self.rowptr), _cabi.ptr(self.colidx), _cabi.ptr(self.vals),
                                                   n, nnz, _cabi.ptr(rp), _cabi.ptr(ci), _cabi.ptr(vv), _cabi.ptr(ws),
                                                   ws_bytes, _stream()), "egnn_csr_transpose")
                same = torch.equal(rp, self.rowptr) and torch.equal(ci, self.colidx) and \
                    (vv is None or torch.equal(vv, self.vals))
            if same:
                self._adjoint = False
            else:
                g = CsrGraph(rp, ci, vv, n, _prepare=False)
                g.dinv, g.iso, g.x0, g.w, g.rowsum = self.dinv, self.iso, self.x0, self.w, self.rowsum
                g._release_scratch()
                g._sorted = True                     # the transpose comes out with sorted rows
                self._adjoint = g
        return self._adjoint or self

    # -- processing order for the wide (F >= 8) kernel ----------------------------
    def row_order(self):
        """``int32[n + 1]``: rows by descending stored-entry count, then the
        number of leading rows a whole CTA sums (include/egnn_b200.h
        ``egnn_row_order``).  Built once per graph on the device."""
        if self._row_order is None:
            lib = _cabi.load()
            with torch.cuda.device(self.device):
                order = torch.empty(self.n + 1, dtype=torch.int32, device=self.device)
                ws_bytes = int(lib.egnn_row_order_ws_bytes(self.n))
                ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
                _cabi.check(lib.egnn_row_order(_cabi.ptr(self.rowptr), self.n, _cabi.ptr(order), _cabi.ptr(ws),
                                               ws_bytes, _stream()), "egnn_row_order")
            self._row_order = order
        return self._row_order

    # -- SELL plan for the narrow (F = 1) path ---------------------------------
    SELL_MIN_NNZ = 1 << 22         # below this the CSR is L2-resident and launch-bound anyway
    SELL_MIN_SEGMENT = 16.0        # mean entries per (row, column block); padding grows below it

    def has_sell_plan(self) -> bool:
        return bool(self._sell)

    def sell_plan(self, force: bool = False):
        """The column-blocked sliced-ELL re-layout the F = 1 orders run on
        (include/egnn_b200.h ``egnn_sell_plan``), built once per graph on the
        device.  Returns ``None`` when the graph does not qualify (weighted,
        unsorted rows, small or very sparse): the generic CSR kernel serves it."""
        if self._sell is not None and (self._sell or not force or self._sell_structural):
            return self._sell or None
        # structural disqualifiers are final; the size / density thresholds are re-evaluated under force
        self._sell = False
        self._sell_structural = True
        if self.vals is not None or self.n < 1 or self.nnz == 0:
            return None
        if not self.rows_sorted():
            return None
        self._sell_structural = False
        lib = _cabi.load()
        nb, cb, lmax = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _cabi.check(lib.egnn_sell_geometry(self.n, self.nnz, C.byref(nb), C.byref(cb), C.byref(lmax)),
                    "egnn_sell_geometry")
        if not force and (self.nnz < self.SELL_MIN_NNZ or
                          self.nnz / (self.n * nb.value) < self.SELL_MIN_SEGMENT):
            return None
        plan = build_sell_plan(self.rowptr, self.colidx, self.n, self.n, 0, (nb.value, cb.value, lmax.value))
        self._sell = plan
        return plan

    def patched(self, delta_rows: Sequence[int], delta_cols: Sequence[int], delta_vals: Sequence[float]):
        """(dinv, iso, x0) of this graph with edge flips applied (UGCA
        recompute): flip e adds ``delta_vals[e]`` to ``A[rows[e], cols[e]]``."""
        n, dev = self.n, self.device
        lib = _cabi.load()
        with torch.cuda.device(dev):
            dinv = torch.empty_like(self.dinv)
            iso = torch.empty_like(self.iso)
            x0 = torch.empty_like(self.x0)
            _cabi.check(lib.egnn_patch_degrees(
                _cabi.ptr(self.w), _cabi.ptr(self.rowsum), _cabi.ptr(self.dinv), _cabi.ptr(self.iso),
                _cabi.ptr(self.x0), n, *_cabi.delta_args((delta_rows, delta_cols, delta_vals)),
                _cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(x0), 0, n, _stream()), "egnn_patch_degrees")
        return dinv, iso, x0

    def patch_nodes(self, deltas, restore: bool = False):
        """UGCA recompute loop: the degree vectors (and ``y0 = dinv * x0``) of the graph
        with the flips applied, in persistent scratch vectors - only the touched entries
        are written (``restore=True`` puts the base values back; queue it after the
        pass that used them).  Returns ``(dinv, iso, x0, y0)``.  One pass at a time per graph."""
        if self._scratch is None:
            self._scratch = (self.dinv.clone(), self.iso.clone(), self.x0.clone(), self.y0().clone())
        lib = _cabi.load()
        with torch.cuda.device(self.device):
            _cabi.check(lib.egnn_patch_nodes(
                _cabi.ptr(self.w), _cabi.ptr(self.rowsum), _cabi.ptr(self.dinv), _cabi.ptr(self.iso), _cabi.ptr(self.x0),
                _cabi.ptr(self.y0()), self.n, *_cabi.delta_args(deltas),
                *[_cabi.ptr(t) for t in self._scratch], 1 if restore else 0, _stream()), "egnn_patch_nodes")
        return self._scratch

    def to_scipy(self):
        """Host copy as scipy CSR float32 (tests / oracle side only)."""
        import scipy.sparse as sp
        data = np.ones(self.nnz, np.float32) if self.vals is None else self.vals.cpu().numpy()
        return sp.csr_matrix((data, self.colidx.cpu().numpy(), self.rowptr.cpu().numpy()),
                             shape=(self.n, self.n))


def build_sell_plan(rowptr: torch.Tensor, colidx: torch.Tensor, n_rows: int, n_cols: int, row0: int, geometry):
    """Build the SELL plan of ``n_rows`` CSR rows (a whole graph or a row shard
    starting at global row ``row0``) over ``n_cols`` columns: prepare (counts,
    one stream synchronisation), allocate the plan arrays as torch tensors,
    fill.  ``geometry`` = (n_blocks, col_block, lmax) from egnn_sell_geometry."""
    lib = _cabi.load()
    dev = rowptr.device
    nnz = int(colidx.numel())
    nb, cb, lmax = geometry
    with torch.cuda.device(dev):
        plan = _cabi.SellPlanStruct()
        plan.n, plan.n_blocks, plan.col_block, plan.lmax = n_rows, nb, cb, lmax
        plan.n_cols, plan.row0 = n_cols, row0
        ws_bytes = int(lib.egnn_sell_ws_bytes(n_rows, nnz, nb, lmax))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _cabi.check(lib.egnn_sell_prepare(_cabi.ptr(rowptr), _cabi.ptr(colidx), n_rows, nnz,
                                          C.byref(plan), _cabi.ptr(ws), ws_bytes, _stream()), "egnn_sell_prepare")
        bufs = {
            "slice_off": torch.empty(plan.n_slices + 1, dtype=torch.int32, device=dev),
            "blk_slice_ptr": torch.empty(plan.n_blocks + 1, dtype=torch.int32, device=dev),
            "idx": torch.empty(max(1, plan.n_entries), dtype=torch.int16, device=dev),
            "rv_ptr": torch.empty(n_rows + 1, dtype=torch.int32, device=dev),
            "vslot": torch.empty(max(1, plan.n_vrows), dtype=torch.int32, device=dev),
            "cta_info": torch.empty(3 * plan.n_cta + 65, dtype=torch.int32, device=dev),
            "hub": torch.empty(plan.n_cta + 1 + plan.n_hub, dtype=torch.int32, device=dev),
            "vpart": torch.empty(max(1, plan.n_rowv), dtype=torch.float32, device=dev),
            "sched": torch.zeros(64 * 32 + 64, dtype=torch.int32, device=dev),
        }
        for name, t in bufs.items():
            setattr(plan, name, t.data_ptr())
        _cabi.check(lib.egnn_sell_fill(_cabi.ptr(rowptr), _cabi.ptr(colidx), n_rows, nnz,
                                       C.byref(plan), _cabi.ptr(ws), ws_bytes, _stream()), "egnn_sell_fill")
    plan._keepalive = bufs
    return plan


def enable_phase_stamps(plan, on: bool = True, trace: bool = False):
    """Ask the step kernel to record CTA 0's ``globaltimer`` at kernel start,
    after every grid barrier and at the end (``egnn_sell_plan.stamps``); read
    them with :func:`read_phase_stamps`.  A measurement aid for bench.py."""
    if on:
        if "stamps" not in plan._keepalive:      # 64 global stamps + (trace) 64 per CTA
            plan._keepalive["stamps"] = torch.zeros(64 + 64 * plan.n_cta, dtype=torch.int64,
                                                    device=plan._keepalive["sched"].device)
        plan.stamps = plan._keepalive["stamps"].data_ptr()
        plan.reserved = 1 if trace else 0
    else:
        plan.stamps = None
        plan.reserved = 0


def read_phase_stamps(plan, k: int, first_operand_in_kernel: bool = True):
    """Phase durations (microseconds) of the last step-kernel launch of ``k``
    orders: ``{"prologue", "spmv": [...], "epilogue": [...], "total"}``.  The
    SpMV figure of an order runs from the previous barrier to the barrier that
    closes it (operand staging included); the epilogue of the last order ends
    with the kernel."""
    st = plan._keepalive["stamps"].cpu().numpy().astype("int64")
    i = 0
    t0 = st[i]; i += 1
    res = {"prologue": 0.0, "spmv": [], "epilogue": []}
    prev = t0
    if first_operand_in_kernel:
        res["prologue"] = (st[i] - prev) / 1e3
        prev = st[i]; i += 1
    for order in range(1, k + 1):
        res["spmv"].append((st[i] - prev) / 1e3)
        prev = st[i]; i += 1
        res["epilogue"].append((st[i] - prev) / 1e3)       # barrier after the epilogue, or the end stamp for the last order
        prev = st[i]; i += 1
    res["total"] = (prev - t0) / 1e3
    return res


def deltas_from_dense(base_adj: torch.Tensor, adj: torch.Tensor, limit: int = 64):
    """Edge flips that turn the dense adjacency ``base_adj`` into ``adj``:
    ``(rows, cols, vals)`` with ``vals = adj - base_adj`` at the entries that
    differ, or ``None`` when more than ``limit`` entries differ (EGNN_MAX_DELTA).

    This is what lets the UNMODIFIED attack code (calib_attack/calib_fga.py:868,
    908,952 calls ``surrogate(features, perturbed_adj)`` with a dense matrix and
    never passes a flip list) take the no-rebuild path: one elementwise pass
    over the two ``[N,N]`` tensors instead of dense->CSR + degree pass + a cold
    first-use kernel.  Index plumbing only (torch ops)."""
    if base_adj.shape != adj.shape or base_adj.device != adj.device:
        return None
    idx = torch.nonzero(adj != base_adj)                        # [D, 2]; synchronises (the count goes to the host)
    if idx.shape[0] > limit:
        return None
    if idx.shape[0] == 0:
        return ([], [], [])
    vals = (adj[idx[:, 0], idx[:, 1]] - base_adj[idx[:, 0], idx[:, 1]]).to(torch.float32)
    return (idx[:, 0].tolist(), idx[:, 1].tolist(), vals.tolist())


def as_graph(adj, device="cuda") -> CsrGraph:
    """Accept what callers of the reference hold: dense torch / numpy, scipy
    sparse, torch sparse, ``(edge_index, N)`` or an existing :class:`CsrGraph`."""
    if isinstance(adj, CsrGraph):
        return adj
    _cabi.require_device()
    if hasattr(adj, "graph") and isinstance(getattr(adj, "graph"), CsrGraph):
        return adj.graph
    if isinstance(adj, tuple) and len(adj) == 2:
        return CsrGraph.from_edge_index(adj[0], int(adj[1]), device=device)
    if isinstance(adj, torch.Tensor):
        if adj.layout in (torch.sparse_coo, torch.sparse_csr):
            coo = adj.to_sparse_coo().coalesce()
            return CsrGraph.from_edge_index(coo.indices(), adj.shape[0], coo.values(), device=device)
        return CsrGraph.from_dense(adj if adj.is_cuda else adj.to(device))
    try:
        import scipy.sparse as sp
        if sp.issparse(adj):
            return CsrGraph.from_scipy(adj, device=device)
    except ImportError:       # pragma: no cover
        pass
    arr = np.asarray(adj)
    if arr.ndim == 2:
        return CsrGraph.from_dense(torch.from_numpy(np.ascontiguousarray(arr, dtype=np.float32)).to(device))
    raise TypeError(f"cannot interpret {type(adj)!r} as an adjacency")
