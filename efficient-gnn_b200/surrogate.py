"""Sparse structure-gradient surrogate for the UGCA attack (SURVEY 8f.3).

The attack (calib_attack/calib_fga.py:864-890) evaluates the calibrated
surrogate on a dense ``[N,N]`` adjacency leaf and calls
``torch.autograd.grad(loss, adj)``, although it only reads row and column
``target_node`` of the result (:881).  That dense forward/backward through
``CompatibleGCN`` (src/gnn/model.py:43-52) is what caps the reference at
20,000 nodes (exp/ablation/ugca_full_multi_dataset.py:575-590).

:class:`SparseGCNSurrogate` restates the same two-layer row-normalised GCN on
the device CSR graph of this package (plus the attack's edge flips as a delta
list, exactly like the wavelet recompute) and produces

* the logits of ONE target node, as a tensor that autograd can differentiate
  (so the attack's own loss functions run unchanged on it), and
* row and column ``target`` of ``dLoss/dA`` - two ``[N]`` vectors - from one
  CSR product and O(N * hidden) dot products, in libegnn_b200 kernels
  (csrc/surrogate.cuh).

``X W1^T`` is computed once per model with a library GEMM (torch): neither the
features nor the weights change during an attack.
"""
from __future__ import annotations

import torch

from . import _cabi
from .graph import CsrGraph, as_graph, deltas_from_dense

__all__ = ["SparseGCNSurrogate", "StructureGradient"]

CTX_FLOATS = 136


def _stream():
    return _cabi.current_stream()


class StructureGradient:
    """Row and column ``target`` of ``dLoss/dA`` (``[N]`` each) and the score the
    attack ranks candidate flips by: ``(row + col) * (1 - 2 A[target, :])``
    (calib_fga.py:880-881)."""

    def __init__(self, row, col):
        self.row, self.col = row, col

    def flip_scores(self, adj_row):
        return (self.row + self.col) * (-2.0 * adj_row + 1.0)


class _TargetLogits(torch.autograd.Function):
    """logits[target] as a function of an ``anchor`` scalar that stands in for the
    adjacency: backward turns the upstream gradient into the structure gradient
    (stored on the surrogate) instead of materialising an [N,N] tensor."""

    @staticmethod
    def forward(ctx, anchor, sur, target, deltas):
        logits, gcn_ctx = sur._target_logits(target, deltas)
        ctx.sur, ctx.target, ctx.deltas, ctx.gcn_ctx = sur, target, deltas, gcn_ctx
        return logits.reshape(1, -1)

    @staticmethod
    def backward(ctx, upstream):
        sur = ctx.sur
        sur.last_gradient = sur._structure_grad(ctx.target, upstream.reshape(-1).contiguous(), ctx.deltas, ctx.gcn_ctx)
        return torch.zeros((), device=upstream.device), None, None, None


class SparseGCNSurrogate:
    """``CompatibleGCN`` (src/gnn/model.py:7-53, eval mode) on a CSR graph.

    ``gcn``: a module with ``gc1`` / ``gc2`` ``nn.Linear`` layers (the
    reference's ``CompatibleGCN`` or an equivalent); ``features`` ``[N, F]``;
    ``adj``: anything :func:`as_graph` accepts.  The hidden width must be a
    multiple of 4, at most 128 (the reference default is 64).
    """

    def __init__(self, gcn, features, adj):
        _cabi.require_device()
        self.graph: CsrGraph = as_graph(adj)
        dev = self.graph.device
        self.lib = _cabi.load()
        w1 = gcn.gc1.weight.detach().to(dev, torch.float32)
        self.b1 = _cabi.vec_ready(gcn.gc1.bias.detach().to(dev))     # read with 16-byte vector loads
        self.w2 = gcn.gc2.weight.detach().to(dev, torch.float32).contiguous()
        self.b2 = gcn.gc2.bias.detach().to(dev, torch.float32).contiguous()
        self.h = int(w1.shape[0])
        self.n_classes = int(self.w2.shape[0])
        if self.h % 4 or self.h > 128:
            raise ValueError("hidden width must be a multiple of 4, at most 128")
        x = torch.as_tensor(features).to(dev, torch.float32)
        if x.shape[0] != self.graph.n:
            raise ValueError("features and adjacency disagree on the number of nodes")
        self.xw = (x @ w1.t()).contiguous()              # [N, H]: library GEMM, once per model
        self.last_gradient = None
        self._state = None                               # (deltas key, Z1, deg) of the last propagate

    # -- forward pieces -------------------------------------------------------
    def propagate(self, deltas=None):
        """``Z1 = A_n X W1^T + b1`` ``[N, H]`` and the raw row sums ``[N]`` of the
        (flipped) adjacency; cached for the delta list it was computed with."""
        key = None if deltas is None else tuple(map(tuple, deltas))
        if self._state is not None and self._state[0] == key:
            return self._state[1], self._state[2]
        g, dev = self.graph, self.graph.device
        with torch.cuda.device(dev):
            z1 = torch.empty((g.n, self.h), dtype=torch.float32, device=dev)
            deg = torch.empty(g.n, dtype=torch.float32, device=dev)
            _cabi.check(self.lib.egnn_gcn_propagate(
                _cabi.ptr(g.rowptr), _cabi.ptr(g.colidx), _cabi.ptr(g.vals), _cabi.ptr(self.xw), _cabi.ptr(self.b1),
                _cabi.ptr(z1), _cabi.ptr(deg), g.n, self.h, *_cabi.delta_args(deltas), _stream()), "egnn_gcn_propagate")
        self._state = (key, z1, deg)
        return z1, deg

    def _target_logits(self, target, deltas):
        g, dev = self.graph, self.graph.device
        z1, _ = self.propagate(deltas)
        with torch.cuda.device(dev):
            logits = torch.empty(self.n_classes, dtype=torch.float32, device=dev)
            gcn_ctx = torch.empty(CTX_FLOATS, dtype=torch.float32, device=dev)
            _cabi.check(self.lib.egnn_gcn_target_logits(
                _cabi.ptr(g.rowptr), _cabi.ptr(g.colidx), _cabi.ptr(g.vals), _cabi.ptr(z1), _cabi.ptr(self.w2),
                _cabi.ptr(self.b2), int(target), g.n, self.h, self.n_classes, _cabi.ptr(logits), _cabi.ptr(gcn_ctx),
                *_cabi.delta_args(deltas), _stream()), "egnn_gcn_target_logits")
        return logits, gcn_ctx

    def _structure_grad(self, target, upstream, deltas, gcn_ctx):
        g, dev = self.graph, self.graph.device
        z1, deg = self.propagate(deltas)
        with torch.cuda.device(dev):
            row = torch.empty(g.n, dtype=torch.float32, device=dev)
            col = torch.empty(g.n, dtype=torch.float32, device=dev)
            _cabi.check(self.lib.egnn_gcn_structure_grad(
                _cabi.ptr(g.rowptr), _cabi.ptr(g.colidx), _cabi.ptr(g.vals), _cabi.ptr(upstream.to(torch.float32)),
                _cabi.ptr(self.w2), _cabi.ptr(z1), _cabi.ptr(self.xw), _cabi.ptr(self.b1), _cabi.ptr(deg),
                _cabi.ptr(gcn_ctx), int(target), g.n, self.h, self.n_classes, _cabi.ptr(row), _cabi.ptr(col),
                *_cabi.delta_args(deltas), _stream()), "egnn_gcn_structure_grad")
        return StructureGradient(row, col)

    # -- what the attack calls ----------------------------------------------------
    def target_logits(self, target, deltas=None):
        """``base_model(x, adj)[[target]]`` (``[1, C]``) on the graph with the
        flips applied.  Differentiable: after ``loss.backward()`` (or
        ``torch.autograd.grad(loss, surrogate.anchor)``) the structure gradient
        of that loss is in :attr:`last_gradient`."""
        self.anchor = torch.zeros((), device=self.graph.device, requires_grad=True)
        return _TargetLogits.apply(self.anchor, self, int(target), deltas)

    def flips_of(self, base_adj_dense, adj_dense):
        """The delta list of a dense perturbed adjacency against the dense base the
        surrogate was built from (``None`` if more than 64 entries differ) - for callers
        that, like the reference attack, carry the perturbed graph as a dense matrix."""
        return deltas_from_dense(base_adj_dense, adj_dense)

    def structure_gradient(self, loss, retain_graph=False):
        """Row / column ``target`` of ``dLoss/dA`` for a scalar ``loss`` computed from
        the output of the last :meth:`target_logits` call - the sparse stand-in for
        ``torch.autograd.grad(loss, adj_leaf)`` (calib_fga.py:877,889-890)."""
        torch.autograd.grad(loss, self.anchor, retain_graph=retain_graph)
        return self.last_gradient

    def all_logits(self, deltas=None):
        """The full ``[N, C]`` forward (second propagation through the same kernel)."""
        g, dev = self.graph, self.graph.device
        z1, _ = self.propagate(deltas)
        h1 = torch.relu(z1)
        with torch.cuda.device(dev):
            h2 = torch.empty_like(h1)
            _cabi.check(self.lib.egnn_gcn_propagate(
                _cabi.ptr(g.rowptr), _cabi.ptr(g.colidx), _cabi.ptr(g.vals), _cabi.ptr(h1), None, _cabi.ptr(h2), None,
                g.n, self.h, *_cabi.delta_args(deltas), _stream()), "egnn_gcn_propagate")
        return h2 @ self.w2.t() + self.b2
