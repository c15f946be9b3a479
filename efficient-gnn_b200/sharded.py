"""Row-sharded wavelet features: one process per GPU, 1-D contiguous row
partition, one exchange of the order's operand per Chebyshev order
(SURVEY.md section 8e; new in this build - the reference is single-device).

Rank r owns rows ``[r * rows_per, (r + 1) * rows_per)`` of the CSR, of
``T_k`` and of the output.  Per order k:

* wide signals (generic CSR kernel): the rank's CSR is split once into a
  local-column and a remote-column half; the local half runs while
  ``all_gather_into_tensor`` of the ``T_{k-1}`` slabs is in flight on a side
  stream, the remote half + fused epilogue run when it lands;
* F = 1 on a binary graph (SELL plan over the rank's rows): the pre-scaled
  operand ``dinv * T_{k-1}`` (0.93 MB at Reddit size) is gathered, then the
  shared-memory SpMV + epilogue run on the local rows.

The backward (autograd w.r.t. the local signal and ``s``) runs the adjoint applications the same
way over the rank's rows of the transposed adjacency (DESIGN.md section 12).

The compute engine is injectable so the host logic (partition, column split,
exchange order, buffer rotation) is testable on CPU with the gloo backend;
the product engine is :class:`CudaEngine` (C ABI, no fallback).
"""
from __future__ import annotations

import ctypes as C
import heapq
import json
import os
import time
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist
from torch.autograd.function import once_differentiable

from . import _cabi
from .wats import WIDE_MIN_F, _heat_scale_grad, _needs_grad, _structure_input, heat_coefficients

_COEFF_GRAD_MAX_ROWS = 8            # EGNN_MAX_SCALES: rows of cbar one egnn_cheb_coeff_grad takes

__all__ = ["RowPartition", "BalancedOrder", "split_columns", "CudaEngine", "DistComm", "PeerExchange", "ShardedWavelet"]


class RowPartition:
    """Equal contiguous row blocks (the last one may be short)."""

    def __init__(self, n: int, world: int):
        self.n, self.world = int(n), int(world)
        self.rows_per = (self.n + self.world - 1) // self.world

    def begin(self, rank: int) -> int:
        return min(self.n, rank * self.rows_per)

    def end(self, rank: int) -> int:
        return min(self.n, (rank + 1) * self.rows_per)

    def rows(self, rank: int) -> int:
        return self.end(rank) - self.begin(rank)

    def slice_csr(self, rowptr: torch.Tensor, colidx: torch.Tensor, rank: int):
        """The rank's rows of a full CSR (global column ids, rowptr rebased)."""
        b, e = self.begin(rank), self.end(rank)
        lo, hi = int(rowptr[b]), int(rowptr[e])
        return (rowptr[b:e + 1] - rowptr[b]).to(torch.int32).contiguous(), colidx[lo:hi].contiguous()


class BalancedOrder:
    """Node relabelling that makes the equal-rows partition nnz-balanced.

    The exchange addresses the operand by global node id and every rank owns one contiguous,
    equally long id range (:class:`RowPartition`), so the entries per rank are balanced by
    renumbering the nodes instead of moving the boundaries: nodes are handed to the ranks longest
    row first, each to the rank with the fewest entries so far (LPT rule, within the fixed
    length of every range), every rank keeps its nodes in their original relative order (what locality the ordering had inside a rank stays), and rank
    r's nodes get the ids of its range.  The features are per node, so the result of the
    relabelled graph is the original one with its rows permuted (:meth:`to_original`).
    Orderings whose equal-rows shards are already balanced (random ids) gain nothing; a
    degree-sorted or community-sorted ordering goes from the heaviest shard setting the step time
    to equal shards.  Index plumbing only (torch ops on whatever device the CSR lives on).

    ``perm[new] = old``, ``inv[old] = new``.
    """

    def __init__(self, perm: torch.Tensor, world: int):
        self.perm = perm.to(torch.int64)
        self.world = int(world)
        self.n = int(perm.numel())
        self.inv = torch.empty_like(self.perm)
        self.inv[self.perm] = torch.arange(self.n, dtype=torch.int64, device=perm.device)

    @classmethod
    def from_rowptr(cls, rowptr: torch.Tensor, world: int) -> "BalancedOrder":
        rp = rowptr.detach().to("cpu", torch.int64)
        n = int(rp.numel()) - 1
        part = RowPartition(n, world)
        deg = rp[1:] - rp[:-1]
        by_len = torch.argsort(deg, descending=True, stable=True).tolist()  # longest row first
        deg_l = deg.tolist()
        # longest-processing-time rule: the next-longest row goes to the rank with the fewest
        # entries so far that still has room in its (fixed-length) id range; one pass over the
        # nodes on the host, once per graph
        heap = [(0, r) for r in range(world) if part.rows(r) > 0]
        room = [part.rows(r) for r in range(world)]
        owner_l = [0] * n
        for node in by_len:
            load, r = heapq.heappop(heap)
            owner_l[node] = r
            room[r] -= 1
            if room[r] > 0:
                heapq.heappush(heap, (load + deg_l[node], r))
        owner = torch.tensor(owner_l, dtype=torch.int64)
        perm = torch.argsort(owner * n + torch.arange(n, dtype=torch.int64))   # by (rank, original id)
        return cls(perm.to(rowptr.device), world)

    @staticmethod
    def shard_entries(rowptr: torch.Tensor, world: int):
        """Entries per rank of the equal-rows partition (to judge an ordering)."""
        part = RowPartition(int(rowptr.numel()) - 1, world)
        return [int(rowptr[part.end(r)]) - int(rowptr[part.begin(r)]) for r in range(world)]

    def relabel_csr(self, rowptr: torch.Tensor, colidx: torch.Tensor, vals: Optional[torch.Tensor] = None):
        """CSR of the relabelled graph: row ``new`` holds the entries of row ``perm[new]`` with
        their columns renumbered, ascending (the narrow path needs column-sorted rows)."""
        dev, n = rowptr.device, self.n
        perm, inv = self.perm.to(dev), self.inv.to(dev)
        counts = (rowptr[1:] - rowptr[:-1]).long()
        rows_old = torch.repeat_interleave(torch.arange(n, device=dev), counts)
        key = inv[rows_old] * n + inv[colidx.long()]
        del rows_old
        if vals is None:
            key = key.sort().values
            vals2 = None
        else:
            key, order = key.sort()
            vals2 = vals[order].contiguous()
        rowptr2 = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        rowptr2[1:] = torch.cumsum(counts[perm], 0)
        return rowptr2.to(torch.int32), (key % n).to(torch.int32), vals2

    def relabel_ids(self, ids):
        """Original node ids -> ids of the relabelled graph (edge-flip lists, target nodes, masks' indices)."""
        ids = torch.as_tensor(ids, dtype=torch.int64)
        return self.inv.to(ids.device)[ids]

    def relabel_deltas(self, deltas):
        rows, cols, vals = deltas
        return self.relabel_ids(rows).tolist(), self.relabel_ids(cols).tolist(), list(vals)

    def from_original(self, x: torch.Tensor) -> torch.Tensor:
        """Per-node rows in original order -> relabelled order (signals X0 going in)."""
        return x[self.perm.to(x.device)]

    def to_original(self, feats: torch.Tensor) -> torch.Tensor:
        """Per-node rows in relabelled order -> original order (features coming out)."""
        return feats[self.inv.to(feats.device)]


def split_columns(rowptr: torch.Tensor, colidx: torch.Tensor, col_begin: int, col_end: int, vals=None):
    """Split a row shard into (local-column CSR, remote-column CSR); entry
    order inside each row is preserved.  Each half is ``(rowptr, colidx)``, or
    ``(rowptr, colidx, vals)`` when the shard's values are given.  Index
    plumbing only (torch ops)."""
    n_rows = rowptr.numel() - 1
    counts = (rowptr[1:] - rowptr[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(n_rows, device=rowptr.device), counts)
    is_local = (colidx >= col_begin) & (colidx < col_end)
    out = []
    for mask in (is_local, ~is_local):
        ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=rowptr.device)
        ptr[1:] = torch.cumsum(torch.bincount(rows[mask], minlength=n_rows), 0)
        half = (ptr.to(torch.int32), colidx[mask].contiguous())
        out.append(half if vals is None else half + (vals[mask].contiguous(),))
    return out[0], out[1]


def _stream():
    return _cabi.current_stream()


class CudaEngine:
    """Device side of the sharded path: thin calls into libegnn_b200."""

    SELL_MIN_SEGMENT = 8.0

    def __init__(self, device):
        _cabi.require_device()
        self.device = torch.device(device)
        self.lib = _cabi.load()
        self.comm_stream = torch.cuda.Stream(device=self.device)
        self._one = torch.zeros(1, dtype=torch.float32, device=self.device)

    def _vals(self, v):
        """Values argument: None (binary), else a valid pointer even for an empty half."""
        return None if v is None else _cabi.ptr(v if v.numel() else self._one)

    # -- degree vectors -----------------------------------------------------
    def prep(self, rowptr, colidx, n_global, row_begin, n_rows, allreduce, vals=None):
        """``(dinv, iso, x0_local, unsorted)`` of the sharded graph (collective); ``vals``: the shard's
        weights.  Keeps ``w_full`` / ``rowsum_local`` for the degree patches of edge flips."""
        dev, lib = self.device, self.lib
        colsum = torch.empty(n_global, dtype=torch.float64, device=dev)
        diag = torch.empty(n_global, dtype=torch.float32, device=dev)
        rowsum = torch.empty(max(1, n_rows), dtype=torch.float32, device=dev)
        dinv = torch.empty(n_global, dtype=torch.float32, device=dev)
        iso = torch.empty(n_global, dtype=torch.uint8, device=dev)
        x0 = torch.empty(max(1, n_rows), dtype=torch.float32, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        w = torch.empty(n_global, dtype=torch.float32, device=dev)
        args = (_cabi.ptr(rowptr), _cabi.ptr(colidx), self._vals(vals), n_global, row_begin, n_rows)
        _cabi.check(lib.egnn_graph_prep_sharded(*args, 0, _cabi.ptr(colsum), _cabi.ptr(diag), _cabi.ptr(rowsum),
                                                None, None, None, _cabi.ptr(flag), None, _stream()), "prep phase 0")
        allreduce(colsum)
        allreduce(diag)
        _cabi.check(lib.egnn_graph_prep_sharded(*args, 1, _cabi.ptr(colsum), _cabi.ptr(diag), _cabi.ptr(rowsum),
                                                _cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(x0), None, _cabi.ptr(w),
                                                _stream()), "prep phase 1")
        self.w_full, self.rowsum_local = w, rowsum[:n_rows]      # kept for the UGCA degree patches
        return dinv, iso, x0[:n_rows], bool(flag.item())

    def patch_degrees(self, dinv, iso, x0_local, n_global, row_begin, n_rows, deltas):
        """(dinv, iso, x0_local) of the graph with edge flips applied (global ids)."""
        dinv2, iso2 = torch.empty_like(dinv), torch.empty_like(iso)
        x02 = torch.empty(max(1, n_rows), dtype=torch.float32, device=self.device)
        _cabi.check(self.lib.egnn_patch_degrees(
            _cabi.ptr(self.w_full), _cabi.ptr(self.rowsum_local), _cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(x0_local),
            n_global, *_cabi.delta_args(deltas), _cabi.ptr(dinv2), _cabi.ptr(iso2), _cabi.ptr(x02), row_begin, n_rows,
            _stream()), "egnn_patch_degrees")
        return dinv2, iso2, x02[:n_rows]

    # -- generic CSR kernel, one order ---------------------------------------
    def order(self, phase, local, remote, dinv, iso, t_prev_full, t_prev_local, t_prev2_local, t_out_local,
              out_local, acc_ws, n_global, nnz_hint, row_begin, row_end, f, order, k_max, n_scales, coeffs,
              op_scale, op_shift, normalize, deltas=None):
        """One order on the rank's rows.  ``local`` / ``remote``: the halves of :func:`split_columns`
        (3-tuples with the values on a weighted shard: egnn_cheb_order_sharded_vals)."""
        halves, weighted = self._halves(local, remote)
        tail = (_cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(t_prev_full), _cabi.ptr(t_prev_local),
                _cabi.ptr(t_prev2_local), _cabi.ptr(t_out_local), _cabi.ptr(out_local), _cabi.ptr(acc_ws), n_global,
                nnz_hint, row_begin, row_end, f, order, k_max, n_scales, coeffs.ctypes.data_as(C.c_void_p),
                float(op_scale), float(op_shift), 1 if normalize else 0, phase, *_cabi.delta_args(deltas), _stream())
        if weighted:
            _cabi.check(self.lib.egnn_cheb_order_sharded_vals(*halves, *tail), "egnn_cheb_order_sharded_vals")
        else:
            _cabi.check(self.lib.egnn_cheb_order_sharded(*halves, *tail), "egnn_cheb_order_sharded")

    def _halves(self, local, remote):
        """C arguments of the two halves: ``(rowptr, colidx)`` each, or ``(rowptr, colidx, vals)`` each
        when either carries values; and whether they do."""
        weighted = any(h is not None and len(h) == 3 for h in (local, remote))
        out = []
        for h in (local, remote):
            rp_, ci_, v_ = (None, None, None) if h is None else (tuple(h) + (None,))[:3]
            out += [_cabi.ptr(rp_), _cabi.ptr(ci_)] + ([self._vals(v_) if h is not None else _cabi.ptr(self._one)]
                                                        if weighted else [])
        return out, weighted

    # -- narrow path -----------------------------------------------------------
    def sell_plan(self, rowptr, colidx, n_rows, n_cols, row0, unsorted):
        if unsorted or n_rows == 0 or colidx.numel() == 0:
            return None
        lib, dev = self.lib, self.device
        nnz = int(colidx.numel())
        nb, cb, lmax = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _cabi.check(lib.egnn_sell_geometry(n_cols, nnz, C.byref(nb), C.byref(cb), C.byref(lmax)), "egnn_sell_geometry")
        if nnz / (n_rows * nb.value) < self.SELL_MIN_SEGMENT:
            return None
        from .graph import build_sell_plan
        return build_sell_plan(rowptr, colidx, n_rows, n_cols, row0, (nb.value, cb.value, lmax.value))

    def prescale(self, x_local, dinv, y_local, n_rows, f, row0):
        _cabi.check(self.lib.egnn_prescale(_cabi.ptr(x_local), _cabi.ptr(dinv), _cabi.ptr(y_local), n_rows, f, row0,
                                           _stream()), "egnn_prescale")

    def sell_step(self, plan, dinv, iso, x0, y_first_full, y_slabs, tbufs, t_all, out, order_begin, order_end, k_max,
                  n_scales, coeffs, op_scale, op_shift, normalize, deltas=None, window=None, base_rowsum=None,
                  default_signal=False):
        """Orders order_begin..order_end of the narrow path in one persistent launch
        (include/egnn_b200.h ``egnn_sell_step_sharded``).  ``base_rowsum`` (full length): the
        vectors passed are the base graph's and the kernel applies the flips' degree patches itself."""
        ys = (None, None) if y_slabs is None else y_slabs
        tb = (None, None) if tbufs is None else tbufs
        _cabi.check(self.lib.egnn_sell_step_sharded(
            C.byref(plan), _cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(x0), _cabi.ptr(y_first_full),
            _cabi.ptr(ys[0]), _cabi.ptr(ys[1]), _cabi.ptr(tb[0]), _cabi.ptr(tb[1]), _cabi.ptr(t_all), _cabi.ptr(out),
            order_begin, order_end, k_max, n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale),
            float(op_shift), 1 if normalize else 0, *_cabi.delta_args(deltas),
            _cabi.ptr(self.w_full) if base_rowsum is not None else None, _cabi.ptr(base_rowsum),
            1 if default_signal else 0,
            None if window is None else C.byref(window), _stream()), "egnn_sell_step_sharded")

    def peer_prescale_push(self, x_local, dinv, n_rows, row0, f, window):
        _cabi.check(self.lib.egnn_peer_prescale_push(_cabi.ptr(x_local), _cabi.ptr(dinv), n_rows, row0, f,
                                                     C.byref(window), _stream()), "egnn_peer_prescale_push")

    # -- wide path with the exchange fused ---------------------------------------
    def row_order(self, rowptr, n_rows):
        order = torch.empty(n_rows + 1, dtype=torch.int32, device=self.device)
        ws_bytes = int(self.lib.egnn_row_order_ws_bytes(n_rows))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        _cabi.check(self.lib.egnn_row_order(_cabi.ptr(rowptr), n_rows, _cabi.ptr(order), _cabi.ptr(ws), ws_bytes,
                                            _stream()), "egnn_row_order")
        return order

    def wide_order(self, rowptr, colidx, row_order, dinv, iso, x0_local, t_out, out, n_global, row_begin, row_end, f,
                   order, k_max, n_scales, coeffs, op_scale, op_shift, normalize, window, deltas=None, vals=None):
        _cabi.check(self.lib.egnn_wide_order_sharded(
            _cabi.ptr(rowptr), _cabi.ptr(colidx), self._vals(vals), _cabi.ptr(row_order), _cabi.ptr(dinv), _cabi.ptr(iso),
            _cabi.ptr(x0_local), _cabi.ptr(t_out), _cabi.ptr(out), n_global, row_begin, row_end, f, order, k_max,
            n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift), 1 if normalize else 0,
            *_cabi.delta_args(deltas), C.byref(window), _stream()), "egnn_wide_order_sharded")

    # -- backward ------------------------------------------------------------------
    def adjoint(self, phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local, b_out_local, cbar,
                tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs, op_scale,
                op_shift, deltas_t=None):
        """Application ``app`` of the adjoint on the rank's rows (include/egnn_b200.h
        ``egnn_cheb_adjoint_sharded``, ``_vals`` when the halves carry values); ``deltas_t``: the
        forward's flips, rows and columns swapped."""
        halves, weighted = self._halves(local, remote)
        tail = (_cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(b_prev_full), _cabi.ptr(b_prev_local),
                _cabi.ptr(b_prev2_local), _cabi.ptr(b_out_local), _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(acc_ws),
                n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs.ctypes.data_as(C.c_void_p),
                float(op_scale), float(op_shift), phase, *_cabi.delta_args(deltas_t), _stream())
        if weighted:
            _cabi.check(self.lib.egnn_cheb_adjoint_sharded_vals(*halves, *tail), "egnn_cheb_adjoint_sharded_vals")
        else:
            _cabi.check(self.lib.egnn_cheb_adjoint_sharded(*halves, *tail), "egnn_cheb_adjoint_sharded")

    def wide_adjoint(self, rowptr, colidx, row_order, dinv, iso, cbar, tbar, xbar, n_global, row_begin, row_end, f,
                     app, k_max, n_scales, coeffs, op_scale, op_shift, window, deltas_t=None, vals=None, b_out=None):
        """``vals``: the transposed shard's values; ``b_out``: [rows, f] rows receiving b_m (app 0: b_K),
        both through egnn_wide_adjoint_sharded_all."""
        if vals is None and b_out is None:
            _cabi.check(self.lib.egnn_wide_adjoint_sharded(
                _cabi.ptr(rowptr), _cabi.ptr(colidx), _cabi.ptr(row_order), _cabi.ptr(dinv), _cabi.ptr(iso),
                _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(xbar), n_global, row_begin, row_end, f, app, k_max,
                n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift),
                *_cabi.delta_args(deltas_t), C.byref(window), _stream()), "egnn_wide_adjoint_sharded")
            return
        _cabi.check(self.lib.egnn_wide_adjoint_sharded_all(
            _cabi.ptr(rowptr), _cabi.ptr(colidx), self._vals(vals), _cabi.ptr(row_order), _cabi.ptr(dinv),
            _cabi.ptr(iso), _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(xbar), _cabi.ptr(b_out), n_global, row_begin,
            row_end, f, app, k_max, n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift),
            *_cabi.delta_args(deltas_t), C.byref(window), _stream()), "egnn_wide_adjoint_sharded_all")

    # -- edge-weight gradient (DESIGN.md section 13) ---------------------------------
    def adj_grad_stacks(self, b_all, t_all, dinv, n_global, row_begin, row_end, rows_per, f, k):
        """Pre-scaled node-major stacks ``(pl, pt)`` ``[rows_per, K*F]`` of the own rows: ``pl[i] = (m_k d_i
        b_k[i])_k``, ``pt[i] = (d_i T_{k-1}[i])_k`` (egnn_adj_grad_stacks_sharded); rows past the rank's
        are not written (exchanged, never read)."""
        pl = torch.empty((rows_per, k * f), dtype=torch.float32, device=self.device)
        pt = torch.empty_like(pl)
        _cabi.check(self.lib.egnn_adj_grad_stacks_sharded(
            _cabi.ptr(b_all), int(b_all.shape[1]), _cabi.ptr(t_all), int(t_all.shape[1]), _cabi.ptr(dinv), n_global,
            row_begin, row_end, f, k, _cabi.ptr(pl), _cabi.ptr(pt), _stream()), "egnn_adj_grad_stacks_sharded")
        return pl, pt

    def adj_grad_degree(self, shard, shard_t, row_orders, dinv, iso, n_global, row_begin, row_end, f, k, op_scale,
                        pl_full, pt_full, xbar, rowsum):
        """``(g [nnz_local], gw [rows], grho [rows])``: ``g_ij`` at the shard's stored entries and the degree
        terms of the own rows (egnn_adj_grad_degree_sharded).  ``shard`` / ``shard_t``: ``(rowptr, colidx,
        vals or None)`` of the rank's rows of A and of A^T."""
        rows = row_end - row_begin
        (rp_, ci_, v_), (rpt, cit, vt) = shard, shard_t
        g = torch.empty(max(1, int(ci_.numel())), dtype=torch.float32, device=self.device)
        gw = torch.empty(max(1, rows), dtype=torch.float32, device=self.device)
        grho = torch.empty_like(gw)
        ws_bytes = int(self.lib.egnn_adj_grad_degree_sharded_ws_bytes(rows))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        _cabi.check(self.lib.egnn_adj_grad_degree_sharded(
            _cabi.ptr(rp_), _cabi.ptr(ci_), self._vals(v_), _cabi.ptr(row_orders[0]), _cabi.ptr(rpt), _cabi.ptr(cit),
            self._vals(vt), _cabi.ptr(row_orders[1]), _cabi.ptr(dinv), _cabi.ptr(iso), n_global, row_begin, row_end,
            f, k, float(op_scale), _cabi.ptr(pl_full), _cabi.ptr(pt_full), _cabi.ptr(xbar), _cabi.ptr(rowsum),
            _cabi.ptr(g), _cabi.ptr(gw), _cabi.ptr(grho), _cabi.ptr(ws), ws_bytes, _stream()),
            "egnn_adj_grad_degree_sharded")
        return g[:ci_.numel()], gw[:rows], grho[:rows]

    def adj_grad_degree_flips(self, shard, shard_t, row_orders, dinv, iso, n_global, row_begin, row_end, f, k,
                              op_scale, pl_full, pt_full, xbar, rowsum, deltas):
        """:meth:`adj_grad_degree` of the flipped graph ``A + delta`` (``dinv`` / ``iso`` / stacks / ``rowsum``
        of ``A'``; egnn_adj_grad_degree_sharded_flips): ``(g, gw, grho, g_flips [n_delta])``, the flips'
        ``g_p`` on every rank and their part of the own rows' degree terms."""
        rows = row_end - row_begin
        (rp_, ci_, v_), (rpt, cit, vt) = shard, shard_t
        g = torch.empty(max(1, int(ci_.numel())), dtype=torch.float32, device=self.device)
        gw = torch.empty(max(1, rows), dtype=torch.float32, device=self.device)
        grho = torch.empty_like(gw)
        g_flips = torch.empty(len(deltas[0]), dtype=torch.float32, device=self.device)
        ws_bytes = int(self.lib.egnn_adj_grad_degree_sharded_ws_bytes(rows))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=self.device)
        _cabi.check(self.lib.egnn_adj_grad_degree_sharded_flips(
            _cabi.ptr(rp_), _cabi.ptr(ci_), self._vals(v_), _cabi.ptr(row_orders[0]), _cabi.ptr(rpt), _cabi.ptr(cit),
            self._vals(vt), _cabi.ptr(row_orders[1]), _cabi.ptr(dinv), _cabi.ptr(iso), n_global, row_begin, row_end,
            f, k, float(op_scale), _cabi.ptr(pl_full), _cabi.ptr(pt_full), _cabi.ptr(xbar), _cabi.ptr(rowsum),
            *_cabi.delta_args(deltas), _cabi.ptr(g_flips), _cabi.ptr(g), _cabi.ptr(gw), _cabi.ptr(grho), _cabi.ptr(ws),
            ws_bytes, _stream()), "egnn_adj_grad_degree_sharded_flips")
        return g[:ci_.numel()], gw[:rows], grho[:rows], g_flips

    def adj_grad_flips(self, deltas, g_flips, gw_full, grho, n_global, row_begin, row_end, op_scale):
        """``dLoss/dv_p`` of the flips whose row this rank owns, 0 for the others, ``[n_delta]``
        (egnn_adj_grad_flips_sharded)."""
        out = torch.empty(len(deltas[0]), dtype=torch.float32, device=self.device)
        _cabi.check(self.lib.egnn_adj_grad_flips_sharded(
            *_cabi.delta_args(deltas), _cabi.ptr(g_flips), _cabi.ptr(gw_full), _cabi.ptr(grho), n_global, row_begin,
            row_end, float(op_scale), _cabi.ptr(out), _stream()), "egnn_adj_grad_flips_sharded")
        return out

    def adj_grad_entries(self, rowptr, colidx, n_global, row_begin, row_end, k, g, gw_full, grho, op_scale):
        """dLoss/dA at the shard's stored entries ``[nnz_local]`` (egnn_adj_grad_entries_sharded)."""
        out = torch.empty(max(1, int(colidx.numel())), dtype=torch.float32, device=self.device)
        _cabi.check(self.lib.egnn_adj_grad_entries_sharded(
            _cabi.ptr(rowptr), _cabi.ptr(colidx), n_global, row_begin, row_end, k, _cabi.ptr(g), _cabi.ptr(gw_full),
            _cabi.ptr(grho), float(op_scale), _cabi.ptr(out), _stream()), "egnn_adj_grad_entries_sharded")
        return out[:colidx.numel()]

    def coeff_grad(self, cbar, t_all):
        """``G[s, k] = <cbar[:, s, :], T_k>`` of the local rows, float64 (egnn_cheb_coeff_grad)."""
        from .wats import _coeff_grad
        return _coeff_grad(cbar, t_all)

    def l1_normalize(self, comb):
        """Out-of-place row L1 normalisation with its backward (egnn_l1_normalize)."""
        from .wats import _L1Normalize
        return _L1Normalize.apply(comb)

    # -- stream plumbing ---------------------------------------------------------
    def side_stream(self):
        return torch.cuda.stream(self.comm_stream)

    def fork(self):
        """Side stream waits for everything queued on the compute stream."""
        self.comm_stream.wait_stream(torch.cuda.current_stream())

    def join(self):
        """Compute stream waits for the side stream (the exchange)."""
        torch.cuda.current_stream().wait_stream(self.comm_stream)


class DistComm:
    """Collectives of the path over ``torch.distributed`` (NCCL on GPUs)."""

    def __init__(self, group=None):
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1

    def allreduce(self, t):
        if self.world > 1:
            dist.all_reduce(t, group=self.group)

    def allgather(self, full, slab):
        """``full[rank * rows_per ...] = slab`` of every rank (equal-size slabs)."""
        if self.world > 1:
            dist.all_gather_into_tensor(full, slab, group=self.group)
        else:
            full.copy_(slab)

    def alltoall(self, out, inp, out_splits, in_splits):
        """Rows ``inp[sum(in_splits[:r]) ...]`` go to rank r; ``out`` receives rank r's rows for this
        rank at ``sum(out_splits[:r])`` (``all_to_all_single``: NCCL and gloo)."""
        if self.world > 1:
            dist.all_to_all_single(out, inp, out_splits, in_splits, group=self.group)
        else:
            out.copy_(inp)


class PeerExchange:
    """This rank's exchange window plus the peers' windows mapped over CUDA IPC
    (include/egnn_b200.h ``egnn_peer_window``).  With it an order needs no
    collective: the epilogue stores the next operand into every rank's window
    over NVLink and the next SpMV waits on flags (csrc/peer.cuh).  One process
    per GPU on one node; handles travel through ``torch.distributed``."""

    def __init__(self, rows_per: int, f: int, group=None, device=None):
        self.lib = _cabi.load()
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > _cabi.MAX_RANKS:
            raise ValueError(f"at most {_cabi.MAX_RANKS} ranks per exchange window")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.device = dev
        self._opened = []
        self._own = None
        with torch.cuda.device(dev):
            nbytes = int(self.lib.egnn_peer_window_bytes(rows_per, self.world, f))
            own = C.c_void_p()
            handle = (C.c_ubyte * _cabi.IPC_HANDLE_BYTES)()
            _cabi.check(self.lib.egnn_peer_alloc(nbytes, C.byref(own), handle), "egnn_peer_alloc")
            self._own = own.value
            mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
            every = torch.empty(self.world * _cabi.IPC_HANDLE_BYTES, dtype=torch.uint8, device=dev)
            dist.all_gather_into_tensor(every, mine, group=group)
            every = every.cpu().numpy().reshape(self.world, _cabi.IPC_HANDLE_BYTES)
            win = _cabi.PeerWindowStruct()
            win.rank, win.world, win.rows_per, win.f = self.rank, self.world, int(rows_per), int(f)
            for r in range(self.world):
                if r == self.rank:
                    win.base[r] = self._own
                    continue
                buf = (C.c_ubyte * _cabi.IPC_HANDLE_BYTES)(*[int(v) for v in every[r]])
                mapped = C.c_void_p()
                _cabi.check(self.lib.egnn_peer_open(buf, C.byref(mapped)), "egnn_peer_open")
                self._opened.append(mapped.value)
                win.base[r] = mapped.value
            self.window = win
        dist.barrier(group=group)          # every window is zeroed and mapped before anyone stores into it
        self.group = group

    def error(self) -> int:
        """Non-zero when a flag wait timed out (synchronises the stream)."""
        out = C.c_int32(0)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.egnn_peer_error(C.byref(self.window), C.byref(out), _stream()), "egnn_peer_error")
        return out.value

    def wait_stats(self, reset: bool = True):
        """(total ns, count) of the flag waits seen by the first CTA (diagnostic)."""
        ns, cnt = C.c_uint64(0), C.c_uint64(0)
        with torch.cuda.device(self.device):
            _cabi.check(self.lib.egnn_peer_wait_stats(C.byref(self.window), C.byref(ns), C.byref(cnt),
                                                      1 if reset else 0, _stream()), "egnn_peer_wait_stats")
        return ns.value, cnt.value

    def close(self):
        """Unmap the peers' windows and free this rank's (collective: nobody may
        still be storing into a window that is being freed)."""
        if self._own is None:
            return
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        with torch.cuda.device(self.device):
            for p in self._opened:
                self.lib.egnn_peer_close(C.c_void_p(p))
            dist.barrier(group=self.group)
            self.lib.egnn_peer_free(C.c_void_p(self._own))
        self._opened, self._own = [], None


class _ShardGraph:
    """The shard one pass runs on: its values (None: binary), column halves, degree vectors, default
    signal, and the in-degree weights / row sums the degree patches of edge flips start from."""

    def __init__(self, vals, halves, dinv, iso, x0, w_full, rowsum_local):
        self.vals, (self.local_half, self.remote_half) = vals, halves
        self.dinv, self.iso, self.x0 = dinv, iso, x0
        self.w_full, self.rowsum_local = w_full, rowsum_local
        self.adjoint_vals = None       # the values moved to the transpose, built once per graph (_adjoint_vals)


class _ShardedSpec:
    """Everything of one sharded pass but its differentiable inputs: ``s`` holds the scales' values,
    ``graph`` the :class:`_ShardGraph` of the call, ``default_signal`` whether ``x0`` is its log1p(degree)."""

    def __init__(self, k, s, lambda_max, want_orders, deltas, graph=None, default_signal=False):
        self.k, self.s, self.lambda_max, self.want_orders, self.deltas = k, s, lambda_max, want_orders, deltas
        self.graph, self.default_signal = graph, default_signal


class _ShardedPass(torch.autograd.Function):
    """``(C [rows, S, F], T [K+1, rows, F])`` of the rank's rows of one un-normalised pass as a function
    of the local signal ``x0`` (None: the default signal), the scales ``s``, this rank's edge weights
    ``ew``, a 0-d ``lam`` = ``lambda_max`` and the values ``dv`` ``[n_delta]`` of the flips
    ``spec.deltas`` (each None when it needs no gradient; the pass applies the flips' values as
    ``spec.deltas`` holds them, detached).  ``T`` is empty unless the orders are wanted or ``s``, ``ew``,
    ``lam`` or ``dv`` needs a gradient.  Backward: the flipped graph's degree vectors are patched once
    and shared by the adjoint pass over the transposed shard (:meth:`ShardedWavelet._adjoint`, keeping
    every Clenshaw vector for ``ew`` / ``lam`` / ``dv``) and the adjacency terms; the scale gradient
    comes from every rank's float64 partials (:meth:`ShardedWavelet._scale_grad`) and the edge-weight,
    ``lambda_max`` and flip-value terms from :meth:`ShardedWavelet._structure_grad`; all are
    collective."""

    @staticmethod
    def forward(ctx, x0, s, ew, lam, dv, sw, spec):
        ctx.set_materialize_grads(False)
        s_grad = s is not None and ctx.needs_input_grad[1]
        structure = any(v is not None and ctx.needs_input_grad[i] for i, v in ((2, ew), (3, lam), (4, dv)))
        want = spec.want_orders or s_grad or structure
        comb, orders = sw._pass(spec.k, spec.s, None if x0 is None else x0.detach(), spec.lambda_max, False, want,
                                spec.deltas, spec.graph)
        f = comb.shape[2]
        if want:
            t_all = torch.stack([o.reshape(sw.rows, f) for o in orders])
        else:
            t_all = comb.new_empty((0,))
            ctx.mark_non_differentiable(t_all)
        ctx.sw, ctx.spec, ctx.f = sw, spec, f
        ctx.x_shape = None if x0 is None else x0.shape
        ctx.s_meta = None if s is None else (s.shape, s.device, s.dtype)
        ctx.lam_meta = None if lam is None else (lam.shape, lam.device, lam.dtype)
        ctx.dv_shape = None if dv is None else dv.shape
        ctx.save_for_backward(t_all if (s_grad or structure) else None)
        return comb, t_all

    @staticmethod
    @once_differentiable
    def backward(ctx, g_comb, g_orders):
        sw, spec, f = ctx.sw, ctx.spec, ctx.f
        (t_all,) = ctx.saved_tensors
        n_scales = int(np.atleast_1d(spec.s).shape[0])
        cbar = (_cabi.vec_ready(g_comb) if g_comb is not None else
                torch.zeros((sw.rows, n_scales, f), dtype=torch.float32, device=sw.device))
        tbar = _cabi.vec_ready(g_orders) if (g_orders is not None and g_orders.numel()) else None
        x_grad = s_grad = ew_grad = lam_grad = dv_grad = None
        structure = ctx.needs_input_grad[2] or ctx.needs_input_grad[3] or ctx.needs_input_grad[4]
        vectors = None
        if spec.deltas is not None and (ctx.needs_input_grad[0] or structure):
            # the flipped graph's dinv / iso, patched once for the adjoint and the adjacency terms
            vectors = sw._patch(sw._base if spec.graph is None else spec.graph, spec.deltas)[:2]
        if ctx.needs_input_grad[0] or structure:
            xbar = sw._adjoint(spec, cbar, tbar, f, keep_all=structure, vectors=vectors)
            if structure:
                xbar, b_all = xbar
            if ctx.needs_input_grad[0]:
                x_grad = xbar.reshape(ctx.x_shape)
        if ctx.needs_input_grad[1]:
            shape, dev, dtype = ctx.s_meta
            s_grad = sw._scale_grad(spec, cbar, t_all).to(device=dev, dtype=dtype).reshape(shape)
        if structure:
            ew_grad, lam_grad, dv_grad = sw._structure_grad(spec, b_all, t_all, f, ctx.needs_input_grad[2],
                                                            ctx.needs_input_grad[3], ctx.needs_input_grad[4],
                                                            vectors=vectors)
            if lam_grad is not None:
                shape, dev, dtype = ctx.lam_meta
                lam_grad = lam_grad.to(device=dev, dtype=dtype).reshape(shape)
            if dv_grad is not None:
                dv_grad = dv_grad.reshape(ctx.dv_shape)
        return x_grad, s_grad, ew_grad, lam_grad, dv_grad, None, None


class ShardedWavelet:
    """Wavelet features of a row-sharded graph.

    ``rowptr_local`` / ``colidx_local``: the rank's rows (global column ids),
    rows assigned by :class:`RowPartition`.  ``engine`` defaults to the CUDA
    engine; tests inject a CPU engine to drive this logic over gloo.

    ``vals_local``: float32 weights of the rank's stored entries, in
    ``colidx_local`` order (None: a binary shard).  Every call uses them: the
    forward, edge flips (their degree patches start from the weighted in-degree
    and row sums) and the backward.  The SELL plan is binary only, so when any
    rank is weighted no rank takes it (the generic loop runs, or the fused wide
    path at F >= 8 with peers), and a rank that passed no weights takes unit
    weights, so that every rank runs the same kernels and collectives.

    :meth:`features` is differentiable w.r.t. ``X0_local``, a tensor ``s``, the
    rank's edge weights (``edge_weight=``) and a 0-d tensor ``lambda_max``
    (DESIGN.md sections 12 and 13).  The backward is collective, like DDP's:
    every rank calls ``backward`` on a loss of its own rows, and the gradients
    are those of the sum of the ranks' losses.
    """

    def __init__(self, rowptr_local, colidx_local, n_global: int, *, vals_local=None, group=None, engine=None,
                 device=None, use_sell: Optional[bool] = None, comm=None, peer_exchange: Optional[bool] = None):
        self.comm = comm if comm is not None else DistComm(group)
        self.rank, self.world = self.comm.rank, self.comm.world
        self.n = int(n_global)
        self.part = RowPartition(self.n, self.world)
        self.row_begin, self.row_end = self.part.begin(self.rank), self.part.end(self.rank)
        self.rows = self.row_end - self.row_begin
        if rowptr_local.numel() != self.rows + 1:
            raise ValueError(f"rank {self.rank} owns {self.rows} rows but rowptr has {rowptr_local.numel()} entries")
        self.device = rowptr_local.device if device is None else torch.device(device)
        self.engine = engine if engine is not None else CudaEngine(self.device)
        self.rowptr = rowptr_local.to(torch.int32).contiguous()
        self.colidx = colidx_local.to(torch.int32).contiguous()
        self.nnz_local = int(self.colidx.numel())
        self.vals = None if vals_local is None else self._check_weights(vals_local)
        self.dinv, self.iso, self.x0, unsorted = self._prep(self.vals)
        self.local_half, self.remote_half = split_columns(self.rowptr, self.colidx, self.row_begin, self.row_end,
                                                          vals=self.vals)
        self._base = _ShardGraph(self.vals, (self.local_half, self.remote_half), self.dinv, self.iso, self.x0,
                                 getattr(self.engine, "w_full", None), getattr(self.engine, "rowsum_local", None))
        self.plan = None
        if use_sell is not False and self.vals is None:      # the SELL plan is binary only
            self.plan = self.engine.sell_plan(self.rowptr, self.colidx, self.rows, self.n, self.row_begin, unsorted)
        # The narrow path exchanges the PRE-SCALED operand dinv * T, the generic path plain T:
        # every rank must run the same one.  A rank whose shard does not qualify for the plan
        # (unsorted rows, too sparse, no rows) takes the plan away from all of them.  Weights are
        # agreed on in the same all-reduce: when any rank is weighted, a binary rank takes unit
        # weights, so that every rank runs the weighted kernels and the same collectives (the
        # transpose of a weighted shard moves values) - its degree vectors do not change.
        if self.world > 1:
            have = torch.tensor([1.0 if self.plan is not None else 0.0, 0.0 if self.vals is None else 1.0],
                                dtype=torch.float64, device=self.device)
            self._allreduce(have)
            plan_ranks, weighted_ranks = (int(round(float(v))) for v in have.tolist())
            if plan_ranks != self.world:
                self.plan = None
            if weighted_ranks and self.vals is None:
                self.plan = None
                self.vals = torch.ones(self.nnz_local, dtype=torch.float32, device=self.device)
                self.local_half, self.remote_half = split_columns(self.rowptr, self.colidx, self.row_begin,
                                                                  self.row_end, vals=self.vals)
                self._base = _ShardGraph(self.vals, (self.local_half, self.remote_half), self.dinv, self.iso,
                                         self.x0, self._base.w_full, self._base.rowsum_local)
        # Fused exchange over peer memory for the narrow path: needs real peers
        # (one process per GPU, NCCL group) and the plan on every rank.
        self.peer = None
        self._wide_peers = {}          # padded width -> PeerExchange of the wide path (built on first use)
        self._row_order = None
        self._group = group
        real_group = (comm is None and engine is None and self.world > 1 and dist.is_initialized()
                      and dist.get_backend(group) == "nccl")
        borrowed = None
        if isinstance(peer_exchange, ShardedWavelet):     # reuse the windows of another instance (same partition)
            borrowed, peer_exchange = peer_exchange, False
            if borrowed.peer is not None:
                if self.plan is None:
                    raise _cabi.EgnnError("a shared exchange window needs the SELL plan on this rank")
                self.peer = borrowed.peer
            self._wide_peers = borrowed._wide_peers
        elif isinstance(peer_exchange, PeerExchange):     # reuse an existing narrow-path window
            if self.plan is None:
                raise _cabi.EgnnError("a shared exchange window needs the SELL plan on this rank")
            self.peer, peer_exchange = peer_exchange, False
        if peer_exchange is None:
            peer_exchange = real_group and os.environ.get("EGNN_EXCHANGE", "peer") != "nccl"
        self._owned_peers = []         # windows this instance allocated (closed by close(); borrowed ones are not)
        self._lender = borrowed        # instance whose windows (and window table) this one shares
        if peer_exchange:
            if not real_group:
                raise _cabi.EgnnError("peer exchange needs one process per GPU in an NCCL group")
            if self.plan is not None:      # agreed on by every rank above
                self.peer = PeerExchange(self.part.rows_per, 1, group=group, device=self.device)
                self._owned_peers.append(self.peer)
        self.fused_wide = borrowed.fused_wide if borrowed is not None else bool(real_group and peer_exchange)
        # default signal X0 = log1p(degree): every rank keeps the whole pre-scaled vector (one
        # all-gather at build time), so order 1 of the fused narrow path needs no exchange
        self.y0_full = self._rowsum_full = None
        if self.peer is not None and self.world > 1:
            rp_ = self.part.rows_per
            pad = torch.zeros(rp_, dtype=torch.float32, device=self.device)
            pad[:self.rows] = self.x0
            full = torch.empty(self.world * rp_, dtype=torch.float32, device=self.device)
            self._allgather(full, pad)
            self.y0_full = (self.dinv * full[:self.n]).contiguous()
            # and the row sums of every node, so that each rank can re-derive the vectors of any node
            # an edge flip touches without an exchange (UGCA recompute, features(deltas=...))
            rowsum_local = getattr(self.engine, "rowsum_local", None)
            if rowsum_local is not None and isinstance(self.engine, CudaEngine):
                pad = torch.zeros(rp_, dtype=torch.float32, device=self.device)
                pad[:self.rows] = rowsum_local
                self._allgather(full, pad)
                self._rowsum_full = full[:self.n].clone()
        self._adjoint_shard = None     # what the backward gathers over (built on first use, see _adjoint_csr)
        self._adjoint_order = None
        self._t_route = None           # how the entries travel to the transpose (values of weighted calls)
        self._half_index = {}          # positions of each half's entries, per CSR (_with_vals)
        self.launches = 0

    def _check_weights(self, v):
        v = torch.as_tensor(v).detach().to(device=self.device, dtype=torch.float32).reshape(-1).contiguous()
        if v.numel() != self.nnz_local:
            raise ValueError(f"rank {self.rank} stores {self.nnz_local} entries but got {v.numel()} weights")
        return v

    def _prep(self, vals):
        """The sharded degree pass (collective); the weights travel only on a weighted shard, so an
        injected engine sees the binary call it always saw."""
        args = (self.rowptr, self.colidx, self.n, self.row_begin, self.rows, self._allreduce)
        return self.engine.prep(*args) if vals is None else self.engine.prep(*args, vals=vals)

    def _graph(self, edge_weight):
        """:class:`_ShardGraph` of one call: the shard's own, or with ``edge_weight`` (detached) in place
        of the stored weights and the degree vectors re-derived for them (collective)."""
        if edge_weight is None:
            return self._base
        vals = self._check_weights(edge_weight)
        eng = self.engine
        kept = (getattr(eng, "w_full", None), getattr(eng, "rowsum_local", None))
        dinv, iso, x0, _ = self._prep(vals)
        halves = self._with_vals("fwd", self.colidx, (self.local_half, self.remote_half), vals)
        g = _ShardGraph(vals, halves, dinv, iso, x0, getattr(eng, "w_full", None), getattr(eng, "rowsum_local", None))
        eng.w_full, eng.rowsum_local = kept      # the shard's own vectors stay the engine's base
        return g

    def _with_vals(self, key, colidx, halves, vals):
        """``halves`` (of :func:`split_columns` over ``colidx``) with ``vals`` split alongside: the entries'
        positions in each half are found once per CSR, so a call's weights cost two gathers."""
        if key not in self._half_index:
            local = (colidx >= self.row_begin) & (colidx < self.row_end)
            self._half_index[key] = (local.nonzero().squeeze(1), (~local).nonzero().squeeze(1))
        il, ir = self._half_index[key]
        (lp, lc), (rp_, rc) = (h[:2] for h in halves)
        return (lp, lc, vals.index_select(0, il)), (rp_, rc, vals.index_select(0, ir))

    def _patch(self, g, deltas):
        """``(dinv, iso, x0_local)`` of ``g`` with the flips applied (the engine patches from ``g``'s
        in-degree weights and row sums)."""
        eng = self.engine
        if g is self._base:
            return eng.patch_degrees(g.dinv, g.iso, g.x0, self.n, self.row_begin, self.rows, deltas)
        kept = (eng.w_full, eng.rowsum_local)
        eng.w_full, eng.rowsum_local = g.w_full, g.rowsum_local
        try:
            return eng.patch_degrees(g.dinv, g.iso, g.x0, self.n, self.row_begin, self.rows, deltas)
        finally:
            eng.w_full, eng.rowsum_local = kept

    def _wide_window(self, ldy: int):
        """Exchange window for ``ldy``-wide operand rows (collective on first use)."""
        if ldy not in self._wide_peers:
            self._wide_peers[ldy] = PeerExchange(self.part.rows_per, ldy, group=self._group, device=self.device)
            (self._lender or self)._owned_peers.append(self._wide_peers[ldy])
        return self._wide_peers[ldy]

    def exchange_error(self) -> int:
        """Non-zero when any flag wait of the fused exchange timed out."""
        err = 0 if self.peer is None else self.peer.error()
        for px in self._wide_peers.values():
            err |= px.error()
        return err

    def check_exchange(self):
        """Raise when a flag wait of the fused exchange timed out (a peer never
        signalled within the kernel's 30 s limit): the kernels keep running on
        stale operands after a timeout, so results since the last check are not
        to be trusted.  Synchronises the stream (one 4-byte D2H copy per window)."""
        if self.exchange_error():
            raise _cabi.EgnnError(f"rank {self.rank}: a peer-exchange flag wait timed out; features computed since "
                                  "the last check used stale operands")

    def close(self):
        """Free the exchange windows this instance allocated (collective: every
        rank calls it).  Windows borrowed from another instance stay open."""
        owned, self._owned_peers = self._owned_peers, []
        for px in owned:
            px.close()
        if self.peer in owned:
            self.peer = None
        for k in [k for k, v in self._wide_peers.items() if v in owned]:
            del self._wide_peers[k]

    # -- collectives -------------------------------------------------------------
    def _allreduce(self, t):
        self.comm.allreduce(t)

    def _allgather(self, full, slab):
        self.comm.allgather(full, slab)

    # -- the path ------------------------------------------------------------------
    def features(self, k=3, s=0.8, *, X0_local=None, lambda_max=2.0, normalize: bool = True,
                 return_parts: bool = False, deltas=None, edge_weight=None):
        """Features of the local rows ``[rows, S*F]`` (reference defaults
        k=3, s=0.8, X0 = log1p(degree)); with ``return_parts`` also the local
        slabs of every order and the un-normalised combination.

        ``deltas=(rows, cols, vals)``: edge flips with GLOBAL node ids applied
        on top of the sharded graph without rebuilding it - the UGCA
        per-perturbation recompute (calib_attack/calib_fga.py:868,908,952) on a
        graph that spans several GPUs.  Every rank passes the same list; each
        patches its replicated dinv/iso and the x0 of its own rows, and the
        order kernels add the flipped entries of the rows they own.

        ``edge_weight``: a ``[nnz_local]`` tensor that replaces this rank's
        stored weights for this call (the degree vectors are re-derived:
        collective, so every rank passes one or none does).

        Differentiable w.r.t. ``X0_local``, a 0-d / 1-d tensor ``s``,
        ``edge_weight``, a 0-d tensor ``lambda_max`` and a 1-d tensor of flip
        values ``deltas[2]`` when grad mode is on and one of them requires
        grad: every output then carries a ``grad_fn``.  ``X0_local.grad``
        receives this rank's rows of the gradient, ``edge_weight.grad``
        dLoss/dA at this rank's stored entries, ``s.grad`` and
        ``lambda_max.grad`` the full gradients, identical bits on every rank
        (DESIGN.md sections 12 and 13).  With ``deltas``, the pass runs on
        ``A' = A + delta`` and the gradients are those of ``A'``: a flip-value
        tensor (one value per flip) receives ``dLoss/dA'`` at each flip, the
        full ``[n_delta]`` vector with the same bits on every rank (a repeated
        entry gives each of its flips the entry's value; a zero-valued flip
        scores a candidate edge without changing the graph), and
        ``lambda_max`` that of the flipped pass (section 15).  An
        ``edge_weight`` that requires grad together with ``deltas`` raises
        ``ValueError``.  The backward is collective: every rank must call
        ``backward`` (once per call of ``features``, in the same order on every
        rank), with the same inputs requiring grad."""
        k = int(k)
        if deltas is not None and len(deltas[0]) == 0:
            deltas = None
        grad_on = torch.is_grad_enabled()
        ew_in = edge_weight if (grad_on and isinstance(edge_weight, torch.Tensor) and edge_weight.requires_grad) \
            else None
        lam_in = lambda_max if (grad_on and isinstance(lambda_max, torch.Tensor) and lambda_max.requires_grad) \
            else None
        if lam_in is not None and lam_in.dim() != 0:
            raise ValueError("a lambda_max that requires grad must be a 0-d tensor")
        if deltas is not None and ew_in is not None:
            raise ValueError("edge flips (deltas=) cannot come with an edge_weight that requires grad")
        dv_in = _structure_input(None, None, deltas)[2]
        if dv_in is not None:        # host values for the C ABI and the degree patches, read once
            deltas = (deltas[0], deltas[1], dv_in.detach().cpu().tolist())
        lam_val = float(lambda_max.detach() if isinstance(lambda_max, torch.Tensor) else lambda_max)
        graph = self._graph(edge_weight)
        x_in = None if X0_local is None else torch.as_tensor(X0_local)
        if _needs_grad(graph.x0 if x_in is None else x_in, s, ew_in, lam_in, dv_in):
            # un-normalised combination (and the orders) through the autograd function, then the
            # out-of-place normalisation (as graph_wavelet_features); the device / dtype conversions stay
            # outside the function, so autograd routes the gradients back to the callers' tensors
            s_vals = s.detach().cpu().numpy() if isinstance(s, torch.Tensor) else s
            x0 = None if x_in is None else x_in.to(device=self.device, dtype=torch.float32)
            s_in = s if (isinstance(s, torch.Tensor) and s.requires_grad) else None
            ew = None if ew_in is None else ew_in.to(device=self.device, dtype=torch.float32).reshape(-1)
            dv = None if dv_in is None else dv_in.to(device=self.device, dtype=torch.float32)
            spec = _ShardedSpec(k, s_vals, lam_val, return_parts, deltas, graph, default_signal=x_in is None)
            comb, t_all = _ShardedPass.apply(x0, s_in, ew, lam_in, dv, self, spec)
            feats = self.engine.l1_normalize(comb) if (normalize and self.rows) else comb
            orders = [t_all[i] for i in range(k + 1)] if return_parts else None
        else:
            comb, orders = self._pass(k, s, X0_local, lam_val, normalize, return_parts, deltas, graph)
            feats = comb / (comb.abs().sum(dim=2, keepdim=True) + 1e-8) if (normalize and return_parts) else comb
        feats = feats.flatten(1)          # [rows, S*F], also for a rank without rows
        return (feats, orders, comb) if return_parts else feats

    def _pass(self, k, s, X0_local, lambda_max, normalize, return_parts, deltas, graph=None):
        """The rank's rows of one pass: ``(out [rows, S, F], [T_0 .. T_K])``, the orders only when
        ``return_parts`` (else just ``[T_0]``).  ``out`` is L1-normalised when ``normalize`` and not
        ``return_parts``, else the un-normalised combination.  ``deltas``: a non-empty flip list or None.
        ``graph``: the call's :class:`_ShardGraph` (None: the shard's own)."""
        eng, dev = self.engine, self.device
        g = self._base if graph is None else graph
        plan = self.plan if g.vals is None else None          # the SELL plan is binary only
        vals_kw = {} if g.vals is None else {"vals": g.vals}
        coeffs = np.ascontiguousarray(heat_coefficients(k, s), dtype=np.float32)
        n_scales = coeffs.shape[0]
        dinv, iso, x0_default = g.dinv, g.iso, g.x0
        base_rowsum = None
        if deltas is not None:
            x_in = None if X0_local is None else torch.as_tensor(X0_local)
            f_in = 1 if (x_in is None or x_in.dim() == 1) else int(x_in.shape[1])
            if k >= 1 and f_in == 1 and plan is not None and self.peer is not None and self._rowsum_full is not None:
                # fused narrow path: the step kernel gets the base graph's vectors plus the row sums of every
                # node and re-derives the nodes the flips touch itself (same arithmetic on every rank) - a
                # perturbed pass is one launch, and the first operand dinv * x0 stays known everywhere
                base_rowsum = self._rowsum_full
            else:
                dinv, iso, x0_default = self._patch(g, deltas)
        x0 = x0_default.reshape(-1, 1) if X0_local is None else torch.as_tensor(X0_local)
        if x0.dim() == 1:
            x0 = x0.reshape(-1, 1)
        if x0.shape[0] != self.rows:
            raise ValueError(f"X0_local has {x0.shape[0]} rows, this rank owns {self.rows}")
        x0 = _cabi.vec_ready(x0.to(device=dev))
        f = int(x0.shape[1])
        rp = self.part.rows_per
        op_scale, op_shift = 2.0 / float(lambda_max), -1.0
        fused_norm = normalize and not return_parts

        def slab():
            # rows beyond self.rows (short last shard) are exchanged but never read: no fill needed
            return torch.empty((rp, f), dtype=torch.float32, device=dev)

        # order 1 writes every (row, scale, column) of out, so it is not cleared either
        out = torch.empty((max(1, self.rows), n_scales, f), dtype=torch.float32, device=dev)
        orders = [x0]
        if k == 0:
            out[:self.rows] = torch.from_numpy(coeffs[:, 0]).to(dev).reshape(1, -1, 1) * x0.unsqueeze(1)
            out = out[:self.rows]
            if fused_norm:            # no kernel ran to fuse it into
                out = out / (out.abs().sum(dim=2, keepdim=True) + 1e-8)
            return out, orders
        use_plan = plan is not None and f == 1
        fused = use_plan and self.peer is not None
        fused_wide = self.fused_wide and f >= WIDE_MIN_F
        if fused_wide:
            # wide signal, exchange fused: operand rows live in the peers' windows (16-byte padded rows)
            win = self._wide_window((f + 3) // 4 * 4).window
            if self._row_order is None:
                self._row_order = eng.row_order(self.rowptr, self.rows)
            eng.peer_prescale_push(x0, dinv, self.rows, self.row_begin, f, win)
            self.launches += 1
            for order in range(1, k + 1):
                t_out = torch.empty((self.rows, f), dtype=torch.float32, device=dev) if return_parts else None
                eng.wide_order(self.rowptr, self.colidx, self._row_order, dinv, iso,
                               x0 if order == 1 else None, t_out, out, self.n, self.row_begin, self.row_end, f, order,
                               k, n_scales, coeffs, op_scale, op_shift, fused_norm, win, deltas, **vals_kw)
                self.launches += 1
                if return_parts:
                    orders.append(t_out)
            return out[:self.rows], orders
        if use_plan:
            # narrow path: the persistent step kernel over the rank's SELL plan (csrc/sell_step.cuh)
            rows1 = max(1, self.rows)
            t_all = None
            tbufs = None
            if return_parts:
                t_all = torch.empty((k + 1, rows1), dtype=torch.float32, device=dev)
                t_all[0, :self.rows] = x0[:, 0]
            elif k >= 2:
                tbufs = (torch.empty(rows1, dtype=torch.float32, device=dev),
                         torch.empty(rows1, dtype=torch.float32, device=dev))
            tail = (k, n_scales, coeffs, op_scale, op_shift, fused_norm, deltas)
            if fused:
                # the whole step is ONE launch: operands travel through the exchange windows, the
                # kernel waits on the owners' flags per column block and signals from its epilogue
                y0 = self.y0_full if X0_local is None and (deltas is None or base_rowsum is not None) else None
                eng.sell_step(self.plan, dinv, iso, x0, y0, None, tbufs, t_all, out, 1, k, *tail,
                              window=self.peer.window, base_rowsum=base_rowsum, default_signal=X0_local is None)
                self.launches += 1
            elif self.world == 1:
                y_slabs = (torch.empty(self.n, dtype=torch.float32, device=dev),
                           torch.empty(self.n, dtype=torch.float32, device=dev))
                eng.sell_step(self.plan, dinv, iso, x0, None, y_slabs, tbufs, t_all, out, 1, k, *tail)
                self.launches += 1
            else:
                # collective exchange (NCCL all-gather or an injected comm): one launch per order
                y_slabs = (slab(), slab())
                full = torch.empty((self.world * rp, 1), dtype=torch.float32, device=dev)
                if self.rows:
                    eng.prescale(x0, dinv, y_slabs[0], self.rows, 1, self.row_begin)
                for order in range(1, k + 1):
                    self._allgather(full, y_slabs[(order - 1) & 1])
                    if self.rows:
                        eng.sell_step(self.plan, dinv, iso, x0, full, y_slabs, tbufs, t_all, out, order, order, *tail)
                        self.launches += 1
            if return_parts:
                if base_rowsum is not None:       # T_0 of the flipped graph: the kernel wrote the touched rows
                    orders[0] = t_all[0, :self.rows].reshape(-1, 1)
                orders += [t_all[i, :self.rows].reshape(-1, 1) for i in range(1, k + 1)]
            return out[:self.rows], orders
        # generic CSR kernel, local / remote column halves around the exchange of T_{k-1}
        if self.rows == rp:
            t_prev = x0
        else:
            t_prev = slab()
            t_prev[:self.rows] = x0
        t_prev2 = None
        full = torch.empty((self.world * rp, f), dtype=torch.float32, device=dev)
        acc_ws = slab()
        for order in range(1, k + 1):
            last = order == k
            if return_parts:
                t_out = slab()
            elif last:
                t_out = None                  # T_K itself is never read again
            elif order <= 2:
                t_out = slab()
            else:
                t_out = t_prev2               # in place over T_{k-2} (read-then-write per element)
            # exchange T_{k-1} on the side stream while the local-column half runs
            eng.fork()
            with eng.side_stream():
                self._allgather(full, t_prev)
            common = (dinv, iso)
            tail = (self.n, max(1, self.nnz_local), self.row_begin, self.row_end, f, order, k, n_scales, coeffs,
                    op_scale, op_shift, fused_norm)
            if self.rows:
                eng.order(0, g.local_half, None, *common, None, t_prev, t_prev2, t_out, out, acc_ws, *tail)
            eng.join()
            if self.rows:
                eng.order(1, None, g.remote_half, *common, full, t_prev, t_prev2, t_out, out, acc_ws, *tail,
                          deltas=deltas)
                self.launches += 2
            if return_parts:
                orders.append(t_out[:self.rows])
            t_prev2, t_prev = t_prev, t_out
        return out[:self.rows], orders

    def gather_features(self, local_feats):
        """All ranks' feature rows, ``[N, S*F]`` on every rank.  A natural
        synchronisation point: the error words of the fused exchange are
        checked here (:meth:`check_exchange`)."""
        if self.peer is not None or self._wide_peers:
            self.check_exchange()
        rp = self.part.rows_per
        pad = torch.zeros((rp, local_feats.shape[1]), dtype=local_feats.dtype, device=local_feats.device)
        pad[:self.rows] = local_feats
        full = torch.empty((self.world * rp, local_feats.shape[1]), dtype=local_feats.dtype, device=local_feats.device)
        self._allgather(full, pad)
        return full[:self.n]

    # -- backward ------------------------------------------------------------------
    def _adjoint_csr(self):
        """``(rowptr, colidx, local half, remote half)`` the adjoint gathers over: this rank's rows of
        ``A^T`` (the columns ``[row_begin, row_end)`` of A, whose entries every rank holds some of),
        global column ids, rows sorted.  Built once, collectively (one ``all_to_all`` of the entries);
        when every rank's transpose equals its own shard (every symmetric graph with sorted rows) the
        copy is dropped and the forward's CSR, halves and row order are used."""
        if self._adjoint_shard is None:
            dev, n, world = self.device, self.n, self.world
            counts = (self.rowptr[1:] - self.rowptr[:-1]).long()
            rows_g = torch.repeat_interleave(torch.arange(self.rows, dtype=torch.int64, device=dev) + self.row_begin,
                                             counts)
            cols = self.colidx.long()
            owner = torch.div(cols, self.part.rows_per, rounding_mode="floor")
            by_owner = torch.argsort(owner, stable=True)
            send = torch.stack([cols[by_owner], rows_g[by_owner]], dim=1).contiguous()    # (row, column) in A^T
            send_counts = torch.bincount(owner, minlength=world)
            recv_counts = torch.empty_like(send_counts)
            self.comm.alltoall(recv_counts, send_counts, [1] * world, [1] * world)
            recv = torch.empty((int(recv_counts.sum()), 2), dtype=torch.int64, device=dev)
            self.comm.alltoall(recv, send, recv_counts.tolist(), send_counts.tolist())
            key, order = ((recv[:, 0] - self.row_begin) * n + recv[:, 1]).sort(stable=True)
            # the route of the entries, for the values of weighted calls (_adjoint_vals)
            self._t_route = (by_owner, send_counts.tolist(), recv_counts.tolist(), order)
            rowptr_t = torch.zeros(self.rows + 1, dtype=torch.int64, device=dev)
            rowptr_t[1:] = torch.cumsum(torch.bincount(torch.div(key, n, rounding_mode="floor"), minlength=self.rows), 0)
            rowptr_t, colidx_t = rowptr_t.to(torch.int32), (key % n).to(torch.int32)
            same = torch.equal(rowptr_t, self.rowptr) and torch.equal(colidx_t, self.colidx)
            differs = torch.tensor([0.0 if same else 1.0], dtype=torch.float64, device=dev)
            self._allreduce(differs)
            if float(differs.item()) == 0.0:
                self._adjoint_shard = False
            else:
                self._adjoint_shard = (rowptr_t, colidx_t) + split_columns(rowptr_t, colidx_t, self.row_begin,
                                                                           self.row_end)
        if self._adjoint_shard is False:
            return self.rowptr, self.colidx, self.local_half, self.remote_half
        return self._adjoint_shard

    def _adjoint_vals(self, g):
        """``(vals_t, local half, remote half)`` of :meth:`_adjoint_csr` with the values of the
        :class:`_ShardGraph` ``g`` moved to their places in the transpose: one collective ``all_to_all``
        along the route the entries took, once per graph (the shard's own, or one call's edge weights,
        whose adjoint and gradient terms share it)."""
        if g.adjoint_vals is not None:
            return g.adjoint_vals
        vals = g.vals
        rowptr_t, colidx_t, local, remote = self._adjoint_csr()
        by_owner, send_counts, recv_counts, order = self._t_route
        recv = torch.empty(sum(recv_counts), dtype=torch.float32, device=self.device)
        self.comm.alltoall(recv, vals.index_select(0, by_owner), recv_counts, send_counts)
        vals_t = recv.index_select(0, order)
        out = (vals_t,) + self._with_vals("fwd" if self._adjoint_shard is False else "adj", colidx_t, (local, remote),
                                          vals_t)
        g.adjoint_vals = out
        return out

    def _adjoint_row_order(self):
        """egnn_row_order of :meth:`_adjoint_csr` (the fused wide adjoint's processing order)."""
        rowptr = self._adjoint_csr()[0]
        if self._adjoint_shard is False:
            if self._row_order is None:
                self._row_order = self.engine.row_order(self.rowptr, self.rows)
            return self._row_order
        if self._adjoint_order is None:
            self._adjoint_order = self.engine.row_order(rowptr, self.rows)
        return self._adjoint_order

    def _adjoint(self, spec, cbar, tbar, f, keep_all=False, vectors=None):
        """This rank's rows of the signal's gradient ``[rows, F]`` from its rows of ``cbar`` ``[rows, S, F]``
        and ``tbar`` ``[K+1, rows, F]`` (collective: the operand of every application is exchanged).  The
        forward's flips are applied transposed, with the forward's patched ``dinv`` / ``iso`` (``vectors``
        when the caller patched them already, else patched here).  ``keep_all``: returns ``(xbar, b_all)``
        with every Clenshaw vector ``b_all [K+1, rows_per, F]`` (slab 0: ``xbar``; the sharded analogue of
        egnn_cheb_adjoint_all)."""
        eng, dev, k = self.engine, self.device, spec.k
        g = self._base if spec.graph is None else spec.graph
        coeffs = np.ascontiguousarray(heat_coefficients(k, spec.s), dtype=np.float32)
        n_scales = coeffs.shape[0]
        op_scale, op_shift = 2.0 / spec.lambda_max, -1.0
        dinv, iso, deltas_t = g.dinv, g.iso, None
        if spec.deltas is not None:
            dinv, iso = self._patch(g, spec.deltas)[:2] if vectors is None else vectors
            d_rows, d_cols, d_vals = spec.deltas
            deltas_t = (d_cols, d_rows, d_vals)
        rp = self.part.rows_per
        if self.rows == 0:            # the fused kernels still take part in the exchange: valid pointers
            cbar = torch.zeros((1, n_scales, f), dtype=torch.float32, device=dev)
        b_all = torch.empty((k + 1, rp, f), dtype=torch.float32, device=dev) if keep_all else None
        xbar = b_all[0] if keep_all else torch.empty((max(1, self.rows), f), dtype=torch.float32, device=dev)

        def done():
            return (xbar[:self.rows], b_all) if keep_all else xbar[:self.rows]

        coef = (k, n_scales, coeffs, op_scale, op_shift)
        if k == 0:                    # xbar = v_0: no operator application, nothing exchanged
            if self.rows:
                eng.adjoint(2, None, None, dinv, iso, None, None, None, xbar, cbar, tbar, None, self.n, 1,
                            self.row_begin, self.row_end, f, 0, *coef)
                self.launches += 1
            return done()
        rowptr_t, colidx_t, local, remote = self._adjoint_csr()
        vals_t = None
        if g.vals is not None:
            vals_t, local, remote = self._adjoint_vals(g)
        if self.fused_wide and f >= WIDE_MIN_F:
            # exchange fused: the operand dinv (.) b travels through the forward's window and flags
            win = self._wide_window((f + 3) // 4 * 4).window
            order = self._adjoint_row_order()
            for app in range(k + 1):
                extra = {} if vals_t is None else {"vals": vals_t}
                if keep_all and app < k:
                    extra["b_out"] = b_all[k - app]
                eng.wide_adjoint(rowptr_t, colidx_t, order, dinv, iso, cbar, tbar, xbar, self.n, self.row_begin,
                                 self.row_end, f, app, *coef, win, deltas_t, **extra)
                self.launches += 2 if (keep_all and app == 0 and self.rows) else 1
            return done()
        # generic CSR kernel, local / remote column halves around the exchange of b_{m+1} (as the forward)

        def slab():
            return torch.empty((rp, f), dtype=torch.float32, device=dev)

        tail = (self.n, max(1, int(colidx_t.numel())), self.row_begin, self.row_end, f)
        b_prev = b_all[k] if keep_all else slab()
        if self.rows:
            eng.adjoint(2, None, None, dinv, iso, None, None, None, b_prev, cbar, tbar, None, *tail, 0, *coef)
            self.launches += 1
        b_prev2 = None
        full = torch.empty((self.world * rp, f), dtype=torch.float32, device=dev)
        acc_ws = slab()
        for app in range(1, k + 1):
            m = k - app
            if keep_all:
                b_out = b_all[m]                                                 # every b_m kept
            else:
                b_out = xbar if m == 0 else (slab() if app <= 2 else b_prev2)    # in place over b_{m+2}
            eng.fork()
            with eng.side_stream():
                self._allgather(full, b_prev)
            if self.rows:
                eng.adjoint(0, local, None, dinv, iso, None, b_prev, b_prev2, b_out, cbar, tbar, acc_ws, *tail, app,
                            *coef)
            eng.join()
            if self.rows:
                eng.adjoint(1, None, remote, dinv, iso, full, b_prev, b_prev2, b_out, cbar, tbar, acc_ws, *tail, app,
                            *coef, deltas_t=deltas_t)
                self.launches += 2
            b_prev2, b_prev = b_prev, b_out
        return done()

    def _scale_grad(self, spec, cbar, t_all):
        """``ds_j = -sum_k k alpha[j,k] G[j,k]`` with ``G = sum_r <cbar_r, T_r>`` over the ranks' rows: every
        rank's float64 partial is all-gathered and added in rank order, so each rank holds the same bits."""
        coeffs = heat_coefficients(spec.k, spec.s)
        n_scales, k1 = coeffs.shape
        if self.rows:
            g = self.engine.coeff_grad(cbar, t_all)
        else:
            g = torch.zeros((n_scales, k1), dtype=torch.float64, device=self.device)
        full = torch.empty((self.world * n_scales, k1), dtype=torch.float64, device=self.device)
        self._allgather(full, g.contiguous())
        parts = full.reshape(self.world, n_scales, k1)
        total = parts[0]
        for r in range(1, self.world):
            total = total + parts[r]
        return _heat_scale_grad(coeffs, total)

    def _structure_grad(self, spec, b_all, t_all, f, want_weights, want_lam, want_flips=False, vectors=None):
        """``(dLoss/dA at this rank's stored entries [nnz_local], dLoss/dlambda_max, dLoss/dv [n_delta])``
        (each None unless wanted) from the Clenshaw vectors ``b_all [K+1, rows_per, F]`` and the orders
        ``t_all [K+1, rows, F]`` (DESIGN.md sections 13 and 15, collective).  Edge weights and flip values:
        the pre-scaled stacks ``m_k d (.) b_k`` and ``d (.) T_{k-1}`` of every rank are all-gathered, each
        rank forms ``g``, ``R`` over its shard, ``Q`` over its rows of the transpose (plus the flips' part of
        both) and ``gw`` / ``grho`` of its rows, ``gw`` is all-gathered and the values at the stored entries
        follow; each flip's value comes from the rank that owns its row, and the ranks' ``[n_delta]`` rows
        are all-gathered and added in rank order.  ``lambda_max``: every rank's float64 partials
        ``<b_k, T_j>`` are all-gathered and added in rank order, so every rank holds the same bits.  With
        flips, ``vectors`` holds the flipped graph's ``(dinv, iso)`` (patched here when None), and the
        default signal's row sums are those of ``A + delta``."""
        eng, dev, k = self.engine, self.device, spec.k
        g = self._base if spec.graph is None else spec.graph
        rp, rb, re_ = self.part.rows_per, self.row_begin, self.row_end
        a = 2.0 / spec.lambda_max
        ew_grad = lam_grad = dv_grad = None
        deltas = spec.deltas
        dinv, iso = g.dinv, g.iso
        if deltas is not None and (want_weights or want_flips):
            dinv, iso = self._patch(g, deltas)[:2] if vectors is None else vectors
        if want_weights or want_flips:
            plf = ptf = None
            if k >= 1:
                pl, pt = eng.adj_grad_stacks(b_all, t_all, dinv, self.n, rb, re_, rp, f, k)
                self.launches += 1 if self.rows else 0
                plf = torch.empty((self.world * rp, k * f), dtype=pl.dtype, device=dev)
                ptf = torch.empty_like(plf)
                self._allgather(plf, pl)
                self._allgather(ptf, pt)
                rowptr_t, colidx_t = self._adjoint_csr()[:2]
                vals_t = None if g.vals is None else self._adjoint_vals(g)[0]
                orders = (self._forward_row_order(), self._adjoint_row_order())
            else:                     # g = 0 and no transposed rows needed: only grho
                rowptr_t, colidx_t, vals_t, orders = self.rowptr, self.colidx, g.vals, (None, None)
            default = spec.default_signal and f == 1
            xbar = b_all[0, :self.rows, 0].contiguous() if default else None
            rowsum = g.rowsum_local if default else None
            shards = ((self.rowptr, self.colidx, g.vals), (rowptr_t, colidx_t, vals_t), orders)
            if deltas is None:
                ge, gw, grho = eng.adj_grad_degree(*shards, dinv, iso, self.n, rb, re_, f, k, a, plf, ptf, xbar,
                                                   rowsum)
            else:
                if default:
                    rowsum = self._flipped_rowsum(rowsum, deltas)
                ge, gw, grho, g_flips = eng.adj_grad_degree_flips(*shards, dinv, iso, self.n, rb, re_, f, k, a, plf,
                                                                  ptf, xbar, rowsum, deltas)
                self.launches += 1 if (self.rows and k >= 1) else 0
            pad = torch.zeros(rp, dtype=gw.dtype, device=dev)
            pad[:self.rows] = gw
            gw_full = torch.empty(self.world * rp, dtype=gw.dtype, device=dev)
            self._allgather(gw_full, pad)
            if want_weights:
                ew_grad = eng.adj_grad_entries(self.rowptr, self.colidx, self.n, rb, re_, k, ge if k >= 1 else None,
                                               gw_full, grho, a)
                self.launches += 1 if self.rows else 0
            self.launches += (3 if k >= 1 else 1) if self.rows else 0
            if want_flips:
                mine = eng.adj_grad_flips(deltas, g_flips, gw_full, grho, self.n, rb, re_, a)
                self.launches += 1
                n_delta = len(deltas[0])
                full = torch.empty(self.world * n_delta, dtype=mine.dtype, device=dev)
                self._allgather(full, mine.contiguous())
                full = full.reshape(self.world, n_delta)
                dv_grad = full[0]
                for r in range(1, self.world):
                    dv_grad = dv_grad + full[r]
        if want_lam:
            if k == 0:                # lambda_max does not enter the pass
                lam_grad = torch.zeros((), dtype=torch.float64, device=dev)
            else:
                part = torch.zeros((k, k + 1), dtype=torch.float64, device=dev)
                if self.rows:
                    # <b_i, T_j> for every i in one egnn_cheb_coeff_grad per 8 orders: b_1..b_K take the
                    # place of the scales (row i - 1 of the partials holds b_i against T_0..T_K)
                    for c0 in range(1, k + 1, _COEFF_GRAD_MAX_ROWS):
                        c1 = min(k + 1, c0 + _COEFF_GRAD_MAX_ROWS)
                        part[c0 - 1:c1 - 1] = eng.coeff_grad(b_all[c0:c1, :self.rows].permute(1, 0, 2).contiguous(),
                                                             t_all)
                        self.launches += 2
                full = torch.empty((self.world * k, k + 1), dtype=torch.float64, device=dev)
                self._allgather(full, part)
                parts = full.reshape(self.world, k, k + 1)
                G = parts[0]
                for r in range(1, self.world):
                    G = G + parts[r]
                total = torch.zeros((), dtype=torch.float64, device=dev)
                for i in range(1, k + 1):
                    total = total + G[i - 1, i] + (1.0 if i == 1 else 2.0) * G[i - 1, i - 1] + \
                        (G[i - 1, i - 2] if i >= 2 else 0.0)
                lam_grad = -total / float(spec.lambda_max)
        return ew_grad, lam_grad, dv_grad

    def _flipped_rowsum(self, rowsum_local, deltas):
        """Row sums of the own rows with ``deltas`` applied, rounded as egnn_patch_degrees forms them for
        the signal ``log1p(rowsum)``: each touched row's base sum plus the float32 sum of its flips in list
        order (the sharded analogue of ``wats._flipped_rowsum``)."""
        add = {}
        for r, v in zip(deltas[0], deltas[2]):
            r = int(r)
            if self.row_begin <= r < self.row_end:
                add[r - self.row_begin] = np.float32(add.get(r - self.row_begin, np.float32(0.0)) + np.float32(v))
        rowsum = torch.as_tensor(rowsum_local).clone()
        if add:
            idx = torch.tensor(list(add), dtype=torch.long, device=rowsum.device)
            rowsum[idx] = rowsum[idx] + torch.tensor(list(add.values()), dtype=torch.float32).to(rowsum.device)
        return rowsum

    def _forward_row_order(self):
        """egnn_row_order of the rank's own shard (longest rows first), built once."""
        if self._row_order is None:
            self._row_order = self.engine.row_order(self.rowptr, self.rows)
        return self._row_order


# --------------------------------------------------------------------------- #
# bench.py entry for N > 1 (launched by torch.distributed.run)                   #
# --------------------------------------------------------------------------- #
def _bench_graph(args, dev, world):
    """The named synthetic graph, optionally renumbered: ``--node-order degree`` sorts the nodes
    by degree (the worst case for equal-rows shards; the generators' own ids are random),
    ``--balance`` applies :class:`BalancedOrder` on top.  Returns the CSR and a record of the
    entries per rank before / after."""
    from . import synth
    rp, ci, n = synth.synth_csr(args.workload, self_loops=True, device=dev)
    info = {"node_order": getattr(args, "node_order", "random"), "balance": bool(getattr(args, "balance", False))}
    if info["node_order"] == "degree":
        deg = (rp[1:] - rp[:-1]).long()
        by_deg = BalancedOrder(torch.argsort(deg, descending=True, stable=True), world)
        rp, ci, _ = by_deg.relabel_csr(rp, ci)
    info["shard_entries"] = BalancedOrder.shard_entries(rp, world)
    if info["balance"]:
        rp, ci, _ = BalancedOrder.from_rowptr(rp, world).relabel_csr(rp, ci)
        info["shard_entries_balanced"] = BalancedOrder.shard_entries(rp, world)
    return rp, ci, n, info


def bench_entry(args, rank, local_rank, world, metric, unit, algorithmic_bytes, clock_sampler_cls,
                physical_gpu_index, scale_list, workload_config, make_flips):
    from . import synth
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    f = args.f or {"reddit": 1, "arxiv": 128, "physics": 1, "pubmed": 1, "cora": 1}[args.workload]
    k_max, n_scales = args.order, args.scales
    scales = scale_list(n_scales)
    sh = synth.SHAPES[args.workload]
    # every rank generates the same seeded graph in its own HBM and keeps its rows
    rp_full, ci_full, n, ordering = _bench_graph(args, dev, world)
    nnz = int(ci_full.numel())
    part = RowPartition(n, world)
    rp_loc, ci_loc = part.slice_csr(rp_full, ci_full, rank)
    del rp_full, ci_full
    torch.cuda.empty_cache()
    sw = ShardedWavelet(rp_loc, ci_loc, n, device=dev)
    x0 = None
    if f > 1:
        gen = torch.Generator(device=dev).manual_seed(sh.seed)
        x0 = torch.randn(n, f, device=dev, generator=gen)[sw.row_begin:sw.row_end].contiguous()
    work = float(nnz) * k_max * f
    use_graph = not getattr(args, "no_graph", False)
    from .wats import WaveletSession
    session = WaveletSession(sw, k=k_max, s=scales, f=f, cuda_graph=use_graph)
    if x0 is not None:
        session.x0.copy_(x0)

    def step():
        return session()

    warm = max(3, args.warmup)
    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    sampler = clock_sampler_cls(physical_gpu_index(local_rank))
    sampler.start()
    sw.launches = 0
    if use_graph:                 # count the launches of one uncaptured pass
        sw.features(k=k_max, s=scales, X0_local=x0)
        per_step_launches = sw.launches
        torch.cuda.synchronize()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    dist.barrier()
    start.record()
    for _ in range(args.steps):
        step()
    stop.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join()
    ms = torch.tensor([start.elapsed_time(stop) / args.steps], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dist.barrier()
    ms_per_step = float(ms.item())
    peer_error = sw.exchange_error()

    # phase breakdown of one eager step from the kernel's own timestamps (rank 0's CTA 0, and the
    # per-CTA trace reduced to min / mean / max), outside the timed region
    phase_us = None
    if sw.plan is not None and f == 1:
        from .graph import enable_phase_stamps, read_phase_stamps
        enable_phase_stamps(sw.plan, True, trace=True)
        sw.features(k=k_max, s=scales)
        torch.cuda.synchronize()
        in_kernel_y0 = sw.peer is None or sw.y0_full is None
        phase_us = read_phase_stamps(sw.plan, k_max, first_operand_in_kernel=in_kernel_y0)
        st = sw.plan._keepalive["stamps"].cpu().numpy().astype(np.int64)
        glob, per = st[:64], st[64:].reshape(sw.plan.n_cta, 64)
        o0 = 1 if in_kernel_y0 else 0
        trace = []
        for order in range(1, k_max + 1):
            opened = glob[o0 + 2 * (order - 1)]
            stage, done, rows = (per[:, 3 * (order - 1) + j] - opened for j in range(3))
            trace.append({"stage_done": [float(stage.min()) / 1e3, float(stage.mean()) / 1e3, float(stage.max()) / 1e3],
                          "slices_done": [float(done.min()) / 1e3, float(done.mean()) / 1e3, float(done.max()) / 1e3],
                          "rows_done": [float(rows.min()) / 1e3, float(rows.mean()) / 1e3, float(rows.max()) / 1e3]})
        phase_us["per_cta_us_after_order_opened_min_mean_max"] = trace
        enable_phase_stamps(sw.plan, False)
        dist.barrier()

    # UGCA per-perturbation recompute on the SHARDED graph (BASELINE config 5): the same global flip
    # list on every rank, applied on top of the shards' plans; device-timed, max over ranks
    ugca = None
    if f == 1 and not getattr(args, "no_ugca", False):
        budget = 5
        cands = [make_flips(n, budget, 100 + i) for i in range(32)]
        for i in range(3):
            sw.features(k=k_max, s=scales, deltas=cands[i])
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        u_steps = 64
        for i in range(u_steps):
            sw.features(k=k_max, s=scales, deltas=cands[i % len(cands)])
        b.record()
        torch.cuda.synchronize()
        u_ms = torch.tensor([a.elapsed_time(b) / u_steps], device=dev, dtype=torch.float64)
        dist.all_reduce(u_ms, op=dist.ReduceOp.MAX)
        ugca = {"flips": budget, "recompute_ms": float(u_ms.item()), "value": work / (float(u_ms.item()) * 1e-3),
                "unperturbed_ms": ms_per_step, "steps": u_steps,
                "entry": "ShardedWavelet.features(deltas=(rows, cols, vals)) on every rank: replicated degree patch + "
                         "one step kernel per rank with the flips as kernel arguments; eager launches"}
        peer_error |= sw.exchange_error()

    # self-check (outside the timed region): every rank also runs the single-GPU path on the whole graph
    check = None
    if not getattr(args, "no_check", False):
        from .graph import CsrGraph
        from .wats import graph_wavelet_features
        rp_full, ci_full, _, _ = _bench_graph(args, dev, world)
        gfull = CsrGraph(rp_full, ci_full, None, n)
        x_full = None
        if f > 1:
            x_full = torch.randn(n, f, device=dev, generator=torch.Generator(device=dev).manual_seed(sh.seed))
        want = graph_wavelet_features(gfull, k=k_max, s=scales, X0=x_full, normalize=False)[sw.row_begin:sw.row_end]
        got = sw.features(k=k_max, s=scales, X0_local=x0, normalize=False)
        scale_ref = torch.tensor([float(want.abs().max().item()) if sw.rows else 0.0], device=dev, dtype=torch.float64)
        diff = torch.tensor([float((got - want).abs().max().item()) if sw.rows else 0.0], device=dev,
                            dtype=torch.float64)
        dist.all_reduce(diff, op=dist.ReduceOp.MAX)
        dist.all_reduce(scale_ref, op=dist.ReduceOp.MAX)
        check = {"max_abs_diff_vs_single_gpu": float(diff.item()), "max_abs_single_gpu": float(scale_ref.item()),
                 "quantity": "un-normalised combination S of every rank's rows (the normalised F=1 feature is sign(S))"}
        if ugca is not None:          # and the sharded recompute against the single-GPU recompute of the same flips
            want_d = graph_wavelet_features(gfull, k=k_max, s=scales, deltas=cands[0], normalize=False)[sw.row_begin:sw.row_end]
            got_d = sw.features(k=k_max, s=scales, deltas=cands[0], normalize=False)
            dd = torch.tensor([float((got_d - want_d).abs().max().item()) if sw.rows else 0.0], device=dev,
                              dtype=torch.float64)
            dist.all_reduce(dd, op=dist.ReduceOp.MAX)
            check["ugca_max_abs_diff_vs_single_gpu"] = float(dd.item())
        del gfull, rp_full, ci_full, want, got

    # end to end: pinned host shard -> device -> features -> host, every step
    e2e = None
    if not args.no_e2e:
        rp_h, ci_h = sw.rowptr.cpu().pin_memory(), sw.colidx.cpu().pin_memory()
        x0_h = None if x0 is None else x0.cpu().pin_memory()
        out_h = torch.empty((max(1, sw.rows), n_scales * f), dtype=torch.float32).pin_memory()

        def e2e_step():
            g = ShardedWavelet(rp_h.to(dev, non_blocking=True), ci_h.to(dev, non_blocking=True), n, device=dev,
                               peer_exchange=sw)
            xx = None if x0_h is None else x0_h.to(dev, non_blocking=True)
            feats = g.features(k=k_max, s=scales, X0_local=xx)
            out_h[:sw.rows].copy_(feats, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for _ in range(2):
            e2e_step()
        torch.cuda.synchronize()
        dist.barrier()
        e_steps = max(3, min(args.steps, 10))
        t0 = time.perf_counter()
        for _ in range(e_steps):
            e2e_step()
        torch.cuda.synchronize()
        dt = torch.tensor([(time.perf_counter() - t0) / e_steps], device=dev, dtype=torch.float64)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        h2d = torch.tensor([rp_h.numel() * 4 + ci_h.numel() * 4 + (0 if x0_h is None else x0_h.numel() * 4)],
                           device=dev, dtype=torch.float64)
        dist.all_reduce(h2d)
        e2e = {"value": work / float(dt.item()), "unit": unit, "h2d_bytes_per_step": int(h2d.item()),
               "d2h_bytes_per_step": int(n * n_scales * f * 4), "ms_per_step": float(dt.item()) * 1e3,
               "steps": e_steps,
               "entry": "ShardedWavelet(pinned host row shard) + features -> pinned host, per rank"}

    launches = torch.tensor([per_step_launches * args.steps if use_graph else sw.launches], device=dev,
                            dtype=torch.float64)
    dist.all_reduce(launches)
    own_all = torch.zeros(1, device=dev, dtype=torch.float64)
    if sw.plan is not None and f == 1:    # the kernels' own stream (2-byte indices), summed over the ranks' plans
        own_all += float(2 * sw.plan.n_entries + 4 * (sw.plan.n_slices + 1) + 4 * sw.plan.n_vrows + 8 * sw.plan.n_rowv)
    dist.all_reduce(own_all)
    if rank == 0:
        b_k = algorithmic_bytes(n, nnz, f, k_max, n_scales)
        peaks = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")
        peak = float(json.load(open(peaks))["hbm_gbs"]) if os.path.isfile(peaks) else 6650.0
        narrow = sw.plan is not None and f == 1
        fused = (sw.peer is not None and f == 1) or (sw.fused_wide and f >= WIDE_MIN_F)
        if narrow:
            own = float(own_all.item()) * k_max
            achieved = own / (ms_per_step * 1e-3) / 1e9
            model = "own stream of the step kernels (every rank's plan x K), whole step incl. exchange"
        else:
            achieved = sum(b_k) / (ms_per_step * 1e-3) / 1e9
            model = "SURVEY 8d contract bytes, whole step incl. exchange"
        line = {
            "metric": metric, "value": work / (ms_per_step * 1e-3), "unit": unit, "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, n, nnz, k_max, n_scales, f, 0),
            "run": {"parallelism": (f"{world} row shards; one persistent step kernel per rank: the epilogue stores the "
                                    "next operand into every rank's window over NVLink, one CTA raises the flags, the "
                                    "next order waits per column block on the ranks that own it (no collective launch)"
                                    if (fused and narrow) else
                                    f"{world} row shards, operand pushed into peer windows over NVLink by the epilogue, "
                                    "flag wait in the next order's kernel (no collective launch)" if fused else
                                    f"{world} row shards, all_gather of the order operand per order (NCCL)"),
                    "path": ("sell-step" if narrow else "wide-fused" if (sw.fused_wide and f >= WIDE_MIN_F)
                             else "csr-split-overlap"),
                    "exchange": "peer-window" if fused else "nccl-allgather", "cuda_graph": bool(use_graph),
                    "phase_us_rank0": phase_us,
                    "per_rank_index_stream_mb": (2 * sw.plan.n_entries / 1e6) if narrow else 4 * nnz / world / 1e6,
                    "ordering": ordering},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                         "frac": achieved / (peak * world), "traffic": None,
                         "achieved_contract": sum(b_k) / (ms_per_step * 1e-3) / 1e9, "bytes_model": model},
            "ugca": ugca, "cpu_baseline": None, "e2e": e2e, "gpu_launches": int(launches.item()),
            "exchange_error": int(peer_error), "check": check,
            "clocks": sampler.summary(),
        }
        print(json.dumps(line), flush=True)
    # A captured graph keeps NCCL work objects alive; tearing the communicator
    # down underneath it can block.  Drop the graph first, and leave through
    # os._exit after a last barrier so no destructor can stall the launcher.
    del session
    import gc
    import sys
    gc.collect()
    torch.cuda.synchronize()
    dist.barrier()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)
