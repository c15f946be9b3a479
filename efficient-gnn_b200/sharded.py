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
from .wats import WIDE_MIN_F, _needs_grad, heat_coefficients

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


def split_columns(rowptr: torch.Tensor, colidx: torch.Tensor, col_begin: int, col_end: int):
    """Split a row shard into (local-column CSR, remote-column CSR); entry
    order inside each row is preserved.  Index plumbing only (torch ops)."""
    n_rows = rowptr.numel() - 1
    counts = (rowptr[1:] - rowptr[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(n_rows, device=rowptr.device), counts)
    is_local = (colidx >= col_begin) & (colidx < col_end)
    out = []
    for mask in (is_local, ~is_local):
        ptr = torch.zeros(n_rows + 1, dtype=torch.int64, device=rowptr.device)
        ptr[1:] = torch.cumsum(torch.bincount(rows[mask], minlength=n_rows), 0)
        out.append((ptr.to(torch.int32), colidx[mask].contiguous()))
    return out[0], out[1]


def _stream():
    return _cabi.current_stream()


def _delta_args(deltas):
    """(rows, cols, vals) -> the four delta arguments of the C ABI (host arrays + count)."""
    d_rows, d_cols, d_vals = ([], [], []) if deltas is None else deltas
    return (_cabi.host_array(C.c_int32, [int(v) for v in d_rows]), _cabi.host_array(C.c_int32, [int(v) for v in d_cols]),
            _cabi.host_array(C.c_float, [float(v) for v in d_vals]), len(d_rows))


class CudaEngine:
    """Device side of the sharded path: thin calls into libegnn_b200."""

    SELL_MIN_SEGMENT = 8.0

    def __init__(self, device):
        _cabi.require_device()
        self.device = torch.device(device)
        self.lib = _cabi.load()
        self.comm_stream = torch.cuda.Stream(device=self.device)

    # -- degree vectors -----------------------------------------------------
    def prep(self, rowptr, colidx, n_global, row_begin, n_rows, allreduce):
        dev, lib = self.device, self.lib
        colsum = torch.empty(n_global, dtype=torch.float64, device=dev)
        diag = torch.empty(n_global, dtype=torch.float32, device=dev)
        rowsum = torch.empty(max(1, n_rows), dtype=torch.float32, device=dev)
        dinv = torch.empty(n_global, dtype=torch.float32, device=dev)
        iso = torch.empty(n_global, dtype=torch.uint8, device=dev)
        x0 = torch.empty(max(1, n_rows), dtype=torch.float32, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        w = torch.empty(n_global, dtype=torch.float32, device=dev)
        args = (_cabi.ptr(rowptr), _cabi.ptr(colidx), None, n_global, row_begin, n_rows)
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
        d_rows, d_cols, d_vals = deltas
        dinv2, iso2 = torch.empty_like(dinv), torch.empty_like(iso)
        x02 = torch.empty(max(1, n_rows), dtype=torch.float32, device=self.device)
        _cabi.check(self.lib.egnn_patch_degrees(
            _cabi.ptr(self.w_full), _cabi.ptr(self.rowsum_local), _cabi.ptr(dinv), _cabi.ptr(iso), _cabi.ptr(x0_local),
            n_global, *_delta_args(deltas), _cabi.ptr(dinv2), _cabi.ptr(iso2), _cabi.ptr(x02), row_begin, n_rows,
            _stream()), "egnn_patch_degrees")
        return dinv2, iso2, x02[:n_rows]

    # -- generic CSR kernel, one order ---------------------------------------
    def order(self, phase, local, remote, dinv, iso, t_prev_full, t_prev_local, t_prev2_local, t_out_local,
              out_local, acc_ws, n_global, nnz_hint, row_begin, row_end, f, order, k_max, n_scales, coeffs,
              op_scale, op_shift, normalize, deltas=None):
        lp, lc = (None, None) if local is None else local
        rp, rc = (None, None) if remote is None else remote
        _cabi.check(self.lib.egnn_cheb_order_sharded(
            _cabi.ptr(lp), _cabi.ptr(lc), _cabi.ptr(rp), _cabi.ptr(rc), _cabi.ptr(dinv), _cabi.ptr(iso),
            _cabi.ptr(t_prev_full), _cabi.ptr(t_prev_local), _cabi.ptr(t_prev2_local), _cabi.ptr(t_out_local),
            _cabi.ptr(out_local), _cabi.ptr(acc_ws), n_global, nnz_hint, row_begin, row_end, f, order, k_max,
            n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift), 1 if normalize else 0,
            phase, *_delta_args(deltas), _stream()), "egnn_cheb_order_sharded")

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
            float(op_shift), 1 if normalize else 0, *_delta_args(deltas),
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
                   order, k_max, n_scales, coeffs, op_scale, op_shift, normalize, window, deltas=None):
        _cabi.check(self.lib.egnn_wide_order_sharded(
            _cabi.ptr(rowptr), _cabi.ptr(colidx), None, _cabi.ptr(row_order), _cabi.ptr(dinv), _cabi.ptr(iso),
            _cabi.ptr(x0_local), _cabi.ptr(t_out), _cabi.ptr(out), n_global, row_begin, row_end, f, order, k_max,
            n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift), 1 if normalize else 0,
            *_delta_args(deltas), C.byref(window), _stream()), "egnn_wide_order_sharded")

    # -- backward ------------------------------------------------------------------
    def adjoint(self, phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local, b_out_local, cbar,
                tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs, op_scale,
                op_shift, deltas_t=None):
        """Application ``app`` of the adjoint on the rank's rows (include/egnn_b200.h
        ``egnn_cheb_adjoint_sharded``); ``deltas_t``: the forward's flips, rows and columns swapped."""
        lp, lc = (None, None) if local is None else local
        rp, rc = (None, None) if remote is None else remote
        _cabi.check(self.lib.egnn_cheb_adjoint_sharded(
            _cabi.ptr(lp), _cabi.ptr(lc), _cabi.ptr(rp), _cabi.ptr(rc), _cabi.ptr(dinv), _cabi.ptr(iso),
            _cabi.ptr(b_prev_full), _cabi.ptr(b_prev_local), _cabi.ptr(b_prev2_local), _cabi.ptr(b_out_local),
            _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(acc_ws), n_global, nnz_hint, row_begin, row_end, f, app,
            k_max, n_scales, coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift), phase,
            *_delta_args(deltas_t), _stream()), "egnn_cheb_adjoint_sharded")

    def wide_adjoint(self, rowptr, colidx, row_order, dinv, iso, cbar, tbar, xbar, n_global, row_begin, row_end, f,
                     app, k_max, n_scales, coeffs, op_scale, op_shift, window, deltas_t=None):
        _cabi.check(self.lib.egnn_wide_adjoint_sharded(
            _cabi.ptr(rowptr), _cabi.ptr(colidx), _cabi.ptr(row_order), _cabi.ptr(dinv), _cabi.ptr(iso),
            _cabi.ptr(cbar), _cabi.ptr(tbar), _cabi.ptr(xbar), n_global, row_begin, row_end, f, app, k_max, n_scales,
            coeffs.ctypes.data_as(C.c_void_p), float(op_scale), float(op_shift), *_delta_args(deltas_t),
            C.byref(window), _stream()), "egnn_wide_adjoint_sharded")

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


class _ShardedSpec:
    """Everything of one sharded pass but its differentiable inputs: ``s`` holds the scales' values."""

    def __init__(self, k, s, lambda_max, want_orders, deltas):
        self.k, self.s, self.lambda_max, self.want_orders, self.deltas = k, s, lambda_max, want_orders, deltas


class _ShardedPass(torch.autograd.Function):
    """``(C [rows, S, F], T [K+1, rows, F])`` of the rank's rows of one un-normalised pass as a function
    of the local signal ``x0`` (None: the default signal) and the scales ``s`` (None when they need no
    gradient).  ``T`` is empty unless the orders are wanted or ``s`` needs a gradient.  Backward: the
    adjoint pass over the transposed shard (:meth:`ShardedWavelet._adjoint`) and the scale gradient from
    every rank's float64 partials (:meth:`ShardedWavelet._scale_grad`); both are collective."""

    @staticmethod
    def forward(ctx, x0, s, sw, spec):
        ctx.set_materialize_grads(False)
        s_grad = s is not None and ctx.needs_input_grad[1]
        want = spec.want_orders or s_grad
        res = sw._pass(spec.k, spec.s, None if x0 is None else x0.detach(), spec.lambda_max, False, want, spec.deltas)
        f = 1 if (x0 is None or x0.dim() == 1) else int(x0.shape[1])
        if want:
            _, orders, comb = res
            t_all = torch.stack([o.reshape(sw.rows, f) for o in orders])
        else:
            comb = res
            t_all = comb.new_empty((0,))
            ctx.mark_non_differentiable(t_all)
        comb = comb.reshape(sw.rows, -1, f)
        ctx.sw, ctx.spec, ctx.f = sw, spec, f
        ctx.x_shape = None if x0 is None else x0.shape
        ctx.s_meta = None if s is None else (s.shape, s.device, s.dtype)
        ctx.save_for_backward(t_all if s_grad else None)
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
        x_grad = s_grad = None
        if ctx.needs_input_grad[0]:
            x_grad = sw._adjoint(spec, cbar, tbar, f).reshape(ctx.x_shape)
        if ctx.needs_input_grad[1]:
            shape, dev, dtype = ctx.s_meta
            s_grad = sw._scale_grad(spec, cbar, t_all).to(device=dev, dtype=dtype).reshape(shape)
        return x_grad, s_grad, None, None


class ShardedWavelet:
    """Wavelet features of a row-sharded graph.

    ``rowptr_local`` / ``colidx_local``: the rank's rows (global column ids),
    rows assigned by :class:`RowPartition`.  ``engine`` defaults to the CUDA
    engine; tests inject a CPU engine to drive this logic over gloo.

    :meth:`features` is differentiable w.r.t. ``X0_local`` and a tensor ``s``
    (DESIGN.md section 12).  The backward is collective, like DDP's: every rank
    calls ``backward`` on a loss of its own rows, and the gradients are those of
    the sum of the ranks' losses.  The adjacency and ``lambda_max`` get no
    gradient here (single-GPU ``graph_wavelet_features`` gives those).
    """

    def __init__(self, rowptr_local, colidx_local, n_global: int, *, group=None, engine=None, device=None,
                 use_sell: Optional[bool] = None, comm=None, peer_exchange: Optional[bool] = None):
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
        self.dinv, self.iso, self.x0, unsorted = self.engine.prep(self.rowptr, self.colidx, self.n, self.row_begin,
                                                                  self.rows, self._allreduce)
        self.local_half, self.remote_half = split_columns(self.rowptr, self.colidx, self.row_begin, self.row_end)
        self.plan = None
        if use_sell is not False:
            self.plan = self.engine.sell_plan(self.rowptr, self.colidx, self.rows, self.n, self.row_begin, unsorted)
        # The narrow path exchanges the PRE-SCALED operand dinv * T, the generic path plain T:
        # every rank must run the same one.  A rank whose shard does not qualify for the plan
        # (unsorted rows, too sparse, no rows) takes the plan away from all of them.
        if self.world > 1:
            have = torch.tensor([1.0 if self.plan is not None else 0.0], dtype=torch.float64, device=self.device)
            self._allreduce(have)
            if int(round(float(have.item()))) != self.world:
                self.plan = None
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
        self.launches = 0

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
    def features(self, k=3, s=0.8, *, X0_local=None, lambda_max: float = 2.0, normalize: bool = True,
                 return_parts: bool = False, deltas=None):
        """Features of the local rows ``[rows, S*F]`` (reference defaults
        k=3, s=0.8, X0 = log1p(degree)); with ``return_parts`` also the local
        slabs of every order and the un-normalised combination.

        ``deltas=(rows, cols, vals)``: edge flips with GLOBAL node ids applied
        on top of the sharded graph without rebuilding it - the UGCA
        per-perturbation recompute (calib_attack/calib_fga.py:868,908,952) on a
        graph that spans several GPUs.  Every rank passes the same list; each
        patches its replicated dinv/iso and the x0 of its own rows, and the
        order kernels add the flipped entries of the rows they own.

        Differentiable w.r.t. ``X0_local`` and a 0-d / 1-d tensor ``s`` when
        grad mode is on and one of them requires grad: every output then
        carries a ``grad_fn`` (``deltas=`` is supported).  ``X0_local.grad``
        receives this rank's rows of the gradient and ``s.grad`` the full scale
        gradient, identical bits on every rank.  The backward is collective:
        every rank must call ``backward`` (once per call of ``features``, in
        the same order on every rank), with the same inputs requiring grad."""
        x_in = None if X0_local is None else torch.as_tensor(X0_local)
        if _needs_grad(self.x0 if x_in is None else x_in, s):
            return self._features_grad(int(k), s, x_in, lambda_max, normalize, return_parts, deltas)
        return self._pass(k, s, X0_local, lambda_max, normalize, return_parts, deltas)

    def _features_grad(self, k, s, x_in, lambda_max, normalize, return_parts, deltas):
        """The differentiable pass: un-normalised combination (and the orders when wanted) through
        :class:`_ShardedPass`, then the out-of-place normalisation (as ``graph_wavelet_features``)."""
        s_vals = s.detach().cpu().numpy() if isinstance(s, torch.Tensor) else s
        if deltas is None or len(deltas[0]) == 0:
            deltas = None
        x0 = x_in
        if x0 is not None:
            x0 = x0.to(device=self.device, dtype=torch.float32)
        spec = _ShardedSpec(k, s_vals, float(lambda_max), return_parts, deltas)
        s_in = s if (isinstance(s, torch.Tensor) and s.requires_grad) else None
        comb, t_all = _ShardedPass.apply(x0, s_in, self, spec)
        feats = self.engine.l1_normalize(comb) if normalize else comb
        feats = feats.reshape(self.rows, -1)
        if return_parts:
            return feats, [t_all[i] for i in range(k + 1)], comb
        return feats

    def _pass(self, k, s, X0_local, lambda_max, normalize, return_parts, deltas):
        eng, dev = self.engine, self.device
        k = int(k)
        coeffs = np.ascontiguousarray(heat_coefficients(k, s), dtype=np.float32)
        n_scales = coeffs.shape[0]
        dinv, iso, x0_default = self.dinv, self.iso, self.x0
        base_rowsum = None
        if deltas is not None and len(deltas[0]) > 0:
            x_in = None if X0_local is None else torch.as_tensor(X0_local)
            f_in = 1 if (x_in is None or x_in.dim() == 1) else int(x_in.shape[1])
            if k >= 1 and f_in == 1 and self.plan is not None and self.peer is not None and self._rowsum_full is not None:
                # fused narrow path: the step kernel gets the base graph's vectors plus the row sums of every
                # node and re-derives the nodes the flips touch itself (same arithmetic on every rank) - a
                # perturbed pass is one launch, and the first operand dinv * x0 stays known everywhere
                base_rowsum = self._rowsum_full
            else:
                dinv, iso, x0_default = eng.patch_degrees(self.dinv, self.iso, self.x0, self.n, self.row_begin,
                                                          self.rows, deltas)
        else:
            deltas = None
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

        def finish(out, orders):
            out = out[:self.rows]
            if k == 0 and fused_norm:
                out = out / (out.abs().sum(dim=2, keepdim=True) + 1e-8)
            if return_parts:
                comb = out
                feats = comb / (comb.abs().sum(dim=2, keepdim=True) + 1e-8) if normalize else comb
                return feats.reshape(self.rows, -1), orders, comb
            return out.reshape(self.rows, -1)

        # order 1 writes every (row, scale, column) of out, so it is not cleared either
        out = torch.empty((max(1, self.rows), n_scales, f), dtype=torch.float32, device=dev)
        orders = [x0]
        if k == 0:
            out[:self.rows] = torch.from_numpy(coeffs[:, 0]).to(dev).reshape(1, -1, 1) * x0.unsqueeze(1)
            return finish(out, orders)
        use_plan = self.plan is not None and f == 1
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
                               k, n_scales, coeffs, op_scale, op_shift, fused_norm, win, deltas)
                self.launches += 1
                if return_parts:
                    orders.append(t_out)
            return finish(out, orders)
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
            return finish(out, orders)
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
                eng.order(0, self.local_half, None, *common, None, t_prev, t_prev2, t_out, out, acc_ws, *tail)
            eng.join()
            if self.rows:
                eng.order(1, None, self.remote_half, *common, full, t_prev, t_prev2, t_out, out, acc_ws, *tail,
                          deltas=deltas)
                self.launches += 2
            if return_parts:
                orders.append(t_out[:self.rows])
            t_prev2, t_prev = t_prev, t_out
        return finish(out, orders)

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
            key = ((recv[:, 0] - self.row_begin) * n + recv[:, 1]).sort().values
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

    def _adjoint(self, spec, cbar, tbar, f):
        """This rank's rows of the signal's gradient ``[rows, F]`` from its rows of ``cbar`` ``[rows, S, F]``
        and ``tbar`` ``[K+1, rows, F]`` (collective: the operand of every application is exchanged).  The
        forward's flips are applied transposed, with the forward's patched ``dinv`` / ``iso``."""
        eng, dev, k = self.engine, self.device, spec.k
        coeffs = np.ascontiguousarray(heat_coefficients(k, spec.s), dtype=np.float32)
        n_scales = coeffs.shape[0]
        op_scale, op_shift = 2.0 / spec.lambda_max, -1.0
        dinv, iso, deltas_t = self.dinv, self.iso, None
        if spec.deltas is not None:
            dinv, iso, _ = eng.patch_degrees(self.dinv, self.iso, self.x0, self.n, self.row_begin, self.rows,
                                             spec.deltas)
            d_rows, d_cols, d_vals = spec.deltas
            deltas_t = (d_cols, d_rows, d_vals)
        if self.rows == 0:            # the fused kernels still take part in the exchange: valid pointers
            cbar = torch.zeros((1, n_scales, f), dtype=torch.float32, device=dev)
        xbar = torch.empty((max(1, self.rows), f), dtype=torch.float32, device=dev)
        coef = (k, n_scales, coeffs, op_scale, op_shift)
        if k == 0:                    # xbar = v_0: no operator application, nothing exchanged
            if self.rows:
                eng.adjoint(2, None, None, dinv, iso, None, None, None, xbar, cbar, tbar, None, self.n, 1,
                            self.row_begin, self.row_end, f, 0, *coef)
                self.launches += 1
            return xbar[:self.rows]
        rowptr_t, colidx_t, local, remote = self._adjoint_csr()
        if self.fused_wide and f >= WIDE_MIN_F:
            # exchange fused: the operand dinv (.) b travels through the forward's window and flags
            win = self._wide_window((f + 3) // 4 * 4).window
            order = self._adjoint_row_order()
            for app in range(k + 1):
                eng.wide_adjoint(rowptr_t, colidx_t, order, dinv, iso, cbar, tbar, xbar, self.n, self.row_begin,
                                 self.row_end, f, app, *coef, win, deltas_t)
                self.launches += 1
            return xbar[:self.rows]
        # generic CSR kernel, local / remote column halves around the exchange of b_{m+1} (as the forward)
        rp = self.part.rows_per

        def slab():
            return torch.empty((rp, f), dtype=torch.float32, device=dev)

        tail = (self.n, max(1, int(colidx_t.numel())), self.row_begin, self.row_end, f)
        b_prev = slab()
        if self.rows:
            eng.adjoint(2, None, None, dinv, iso, None, None, None, b_prev, cbar, tbar, None, *tail, 0, *coef)
            self.launches += 1
        b_prev2 = None
        full = torch.empty((self.world * rp, f), dtype=torch.float32, device=dev)
        acc_ws = slab()
        for app in range(1, k + 1):
            m = k - app
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
        return xbar[:self.rows]

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
        alpha = torch.from_numpy(coeffs).to(self.device)
        kk = torch.arange(k1, dtype=torch.float64, device=self.device)
        return -(kk * alpha * total).sum(dim=1)


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
