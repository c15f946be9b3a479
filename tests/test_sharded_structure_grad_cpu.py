"""Host logic of the row-sharded edge-weight and ``lambda_max`` gradients on CPU: world 2 and 3 over gloo,
with a NumPy engine whose new methods restate the weighted orders, the weighted adjoint applications and
the gradient terms in float64.  What is under test is the weighted prep, the values through the column
split and the transpose (its ``all_to_all`` carries them), the exchange of the pre-scaled stacks and of
``gw``, and the rank-order sum of the ``lambda_max`` partials.

Two bars: the gradient terms are checked to 1e-10 against a float64 restatement from every rank's
Clenshaw vectors and orders as the pass computed them (float32 values, so this pins the plumbing
exactly), and the whole gradient against ``adjacency_vjp`` at section 10's norm-wise bar (the pass
itself stores its orders in float32).  Also: the ABI's argument errors of the new entry points."""
import ctypes as C
import os
import socket
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from test_sharded_backward_cpu import AdjointNumpyEngine, RecordingComm  # noqa: E402


def _spmv_half(half, rows, row_begin, d, src, off):
    """sum_{j != i} A_ij d_j src[j - off] over a (weighted) half, float64 [rows, f]."""
    rp, ci = half[0].numpy(), half[1].numpy()
    v = half[2].numpy().astype(np.float64) if len(half) == 3 else np.ones(ci.size)
    acc = np.zeros((rows, src.shape[1]))
    r = np.repeat(np.arange(rows), np.diff(rp))
    keep = ci != (r + row_begin)
    np.add.at(acc, r[keep], (v[keep] * d[ci[keep]])[:, None] * src[ci[keep] - off])
    return acc


class WeightedNumpyEngine(AdjointNumpyEngine):
    """AdjointNumpyEngine for weighted shards plus float64 restatements of the gradient methods of
    CudaEngine (tests only)."""

    def __init__(self):
        super().__init__()
        self.seen = {}

    def prep(self, rowptr, colidx, n_global, row_begin, n_rows, allreduce, vals=None):
        rp, ci = rowptr.numpy(), colidx.numpy()
        v = np.ones(ci.size) if vals is None else vals.numpy().astype(np.float64)
        rows = np.repeat(np.arange(n_rows), np.diff(rp)) + row_begin
        colsum = torch.zeros(n_global, dtype=torch.float64)
        diag = torch.zeros(n_global, dtype=torch.float64)
        np.add.at(colsum.numpy(), ci, v)
        on = rows == ci
        np.add.at(diag.numpy(), rows[on], v[on])
        rowsum = np.zeros(n_rows)
        np.add.at(rowsum, rows - row_begin, v)
        allreduce(colsum)
        allreduce(diag)
        w = colsum.numpy() - diag.numpy()
        iso = w == 0
        dinv = np.where(iso, 1.0, 1.0 / np.sqrt(np.where(iso, 1.0, w)))
        self.w_full, self.rowsum_local = w.copy(), rowsum.copy()
        return torch.from_numpy(dinv), torch.from_numpy(iso.astype(np.uint8)), torch.from_numpy(np.log1p(rowsum)), False

    def row_order(self, rowptr, n_rows):
        return None

    def order(self, phase, local, remote, dinv, iso, t_prev_full, t_prev_local, t_prev2_local, t_out_local,
              out_local, acc_ws, n_global, nnz_hint, row_begin, row_end, f, order, k_max, n_scales, coeffs,
              op_scale, op_shift, normalize, deltas=None):
        half = local if phase == 0 else remote
        if len(half) == 2:
            return super().order(phase, local, remote, dinv, iso, t_prev_full, t_prev_local, t_prev2_local,
                                 t_out_local, out_local, acc_ws, n_global, nnz_hint, row_begin, row_end, f, order,
                                 k_max, n_scales, coeffs, op_scale, op_shift, normalize, deltas)
        self.calls.append(f"order{order}.phase{phase}.w")
        # the binary restatement with the half's weights folded into dinv of each entry
        rows = row_end - row_begin
        d = dinv.numpy().astype(np.float64)
        if phase == 0:
            acc_ws.numpy()[:rows] = _spmv_half(half, rows, row_begin, d, t_prev_local.numpy().astype(np.float64),
                                               row_begin)
            return
        acc = _spmv_half(half, rows, row_begin, d, t_prev_full.numpy().astype(np.float64), 0)
        src = t_prev_full.numpy().astype(np.float64)
        for dr, dc, dv in zip(*(deltas or ([], [], []))):
            if row_begin <= dr < row_end and dr != dc:
                acc[dr - row_begin] += dv * d[dc] * src[dc]
        acc += acc_ws.numpy()[:rows]
        di = d[row_begin:row_end, None]
        theta = (op_scale * (1 - iso.numpy()[row_begin:row_end]) + op_shift)[:, None]
        xprev = t_prev_local.numpy()[:rows].astype(np.float64)
        lap = theta * xprev - op_scale * di * acc
        tk = lap if order == 1 else 2 * lap - t_prev2_local.numpy()[:rows]
        if t_out_local is not None:
            t_out_local.numpy()[:rows] = tk
        o = out_local.numpy()
        for s in range(n_scales):
            ck, cp = coeffs[s, order], coeffs[s, order - 1]
            val = cp * xprev + ck * tk if order == 1 else o[:rows, s, :] + ck * tk
            if normalize and order == k_max:
                val = val / (np.abs(val).sum(axis=1, keepdims=True) + 1e-8)
            o[:rows, s, :] = val

    def adjoint(self, phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local, b_out_local, cbar,
                tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs, op_scale,
                op_shift, deltas_t=None):
        half = local if phase == 0 else remote
        if app == 0 or len(half) == 2:
            return super().adjoint(phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local,
                                   b_out_local, cbar, tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app,
                                   k_max, n_scales, coeffs, op_scale, op_shift, deltas_t)
        self.calls.append(f"adj{app}.phase{phase}.w")
        rows, m = row_end - row_begin, k_max - app
        d = dinv.numpy().astype(np.float64)
        if phase == 0:
            acc_ws.numpy()[:rows] = _spmv_half(half, rows, row_begin, d, b_prev_local.numpy().astype(np.float64),
                                               row_begin)
            return
        assert deltas_t is None
        cb = cbar.numpy()[:rows].astype(np.float64)
        v = sum(float(coeffs[s, m]) * cb[:, s, :] for s in range(n_scales))
        if tbar is not None:
            v = v + tbar.numpy()[m, :rows]
        acc = _spmv_half(half, rows, row_begin, d, b_prev_full.numpy().astype(np.float64), 0) + acc_ws.numpy()[:rows]
        di = d[row_begin:row_end, None]
        theta = (op_scale * (1 - iso.numpy()[row_begin:row_end]) + op_shift)[:, None]
        own = b_prev_local.numpy()[:rows].astype(np.float64)
        b2 = 0.0 if b_prev2_local is None else b_prev2_local.numpy()[:rows]
        b_out_local.numpy()[:rows] = (1.0 if m == 0 else 2.0) * (theta * own - op_scale * di * acc) + v - b2

    # -- the gradient terms, float64 ---------------------------------------------------
    def adj_grad_stacks(self, b_all, t_all, dinv, n_global, row_begin, row_end, rows_per, f, k):
        rows = row_end - row_begin
        self.seen["b_all"], self.seen["t_all"] = b_all[:, :rows].clone(), t_all.clone()
        d = dinv.numpy()[row_begin:row_end, None].astype(np.float64)
        pl = np.zeros((rows_per, k * f))
        pt = np.zeros((rows_per, k * f))
        for i in range(k):
            pl[:rows, i * f:(i + 1) * f] = (1.0 if i == 0 else 2.0) * d * b_all.numpy()[i + 1, :rows]
            pt[:rows, i * f:(i + 1) * f] = d * t_all.numpy()[i]
        return torch.from_numpy(pl), torch.from_numpy(pt)

    def adj_grad_degree(self, shard, shard_t, row_orders, dinv, iso, n_global, row_begin, row_end, f, k, op_scale,
                        pl_full, pt_full, xbar, rowsum):
        rows = row_end - row_begin

        def dots(csr, own, gath):
            rp, ci, v = csr
            v = np.ones(ci.numel()) if v is None else v.numpy().astype(np.float64)
            r = np.repeat(np.arange(rows), np.diff(rp.numpy()))
            ci = ci.numpy()
            if k == 0:
                g = np.zeros(ci.size)
            else:
                g = (own.numpy()[r + row_begin] * gath.numpy()[ci]).sum(axis=1)
            g[ci == r + row_begin] = 0.0
            out = np.zeros(rows)
            np.add.at(out, r, v * g)
            return g, out

        g, R = dots(shard, pl_full, pt_full)
        _, Q = dots(shard_t, pt_full, pl_full)
        d = dinv.numpy()[row_begin:row_end].astype(np.float64)
        is_iso = iso.numpy()[row_begin:row_end] != 0
        gw = np.where(is_iso, 0.0, 0.5 * op_scale * d * d * (R + Q))
        grho = np.zeros(rows) if xbar is None else xbar.numpy().astype(np.float64) / (1.0 + np.asarray(rowsum))
        return torch.from_numpy(g), torch.from_numpy(gw), torch.from_numpy(grho)

    def adj_grad_entries(self, rowptr, colidx, n_global, row_begin, row_end, k, g, gw_full, grho, op_scale):
        rows = row_end - row_begin
        r = np.repeat(np.arange(rows), np.diff(rowptr.numpy()))
        ci = colidx.numpy()
        gv = np.zeros(ci.size) if g is None else g.numpy()
        out = grho.numpy()[r] + np.where(ci != r + row_begin, -op_scale * gv + gw_full.numpy()[ci], 0.0)
        self.seen["entries"] = out.copy()
        return torch.from_numpy(out)


def weighted_graph(n, seed):
    """Weighted directed graph with an in-star hub on node 0 (its transpose differs from the shard),
    an isolated node, stored self loops, explicit zero weights and a column (node 5) whose only
    entries are explicit zeros."""
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=5.0 / n, random_state=rng, format="lil")
    a[:, 0] = 0
    a[rng.choice(np.arange(6, n), size=n // 3, replace=False), 0] = 1.0
    a[3, :] = 0
    a[:, 3] = 0
    a[:, 5] = 0
    a[2, 8] = 0                       # free the positions of the explicit zeros below, so that
    a[4, 1] = 0                       # sum_duplicates keeps them zero
    a = sp.csr_matrix(a)
    a.data[:] = rng.uniform(0.2, 2.0, a.data.size)
    pat = a.tolil()
    for i in (7, 11):
        pat[i, i] = 0.7
    pat = sp.csr_matrix(pat)
    # explicit zeros: two ordinary entries and both entries of column 5
    rows, cols = list(pat.nonzero()[0]), list(pat.nonzero()[1])
    vals = list(np.asarray(pat[rows, cols]).ravel())
    for (i, j) in [(1, 5), (9, 5), (2, 8), (4, 1)]:
        rows.append(i); cols.append(j); vals.append(0.0)
    m = sp.coo_matrix((np.array(vals, np.float32), (rows, cols)), shape=(n, n)).tocsr()
    m.sum_duplicates()
    m.sort_indices()
    return m


def tiny_graph():
    """4 nodes, weighted and directed: with 3 ranks the last one owns no rows."""
    d = np.array([[0.0, 1.5, 0.0, 0.5], [0.0, 0.7, 2.0, 0.0], [1.0, 0.0, 0.0, 0.0], [0.0, 0.0, 3.0, 0.0]], np.float32)
    return sp.csr_matrix(d)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, case, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from adjacency_reference import adjacency_vjp
        from efficient_gnn_b200 import sharded
        graph, f, k, scales, normalize, lam_val, stored_weights = case
        adj = tiny_graph() if graph == "tiny" else weighted_graph(301, 4)
        n = adj.shape[0]
        rp = torch.from_numpy(adj.indptr.astype(np.int32))
        ci = torch.from_numpy(adj.indices.astype(np.int32))
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        b, e = part.begin(rank), part.end(rank)
        w_loc = adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)
        comm = RecordingComm()
        eng = WeightedNumpyEngine()
        # either the shard stores the weights and they come in again as edge_weight, or a binary shard
        # gets all of them per call
        sw = sharded.ShardedWavelet(rpl, cil, n, engine=eng, device="cpu", comm=comm,
                                    vals_local=torch.from_numpy(w_loc) if stored_weights else None)
        rng = np.random.default_rng(17)
        x_full = rng.standard_normal((n, f)).astype(np.float32) if f > 1 else None
        n_s = len(scales)
        hbar = rng.standard_normal((n, n_s * f))
        cbar = rng.standard_normal((n, n_s, f))
        ew = torch.from_numpy(w_loc.astype(np.float64)).requires_grad_(True)
        lam = torch.tensor(lam_val, dtype=torch.float64, requires_grad=True)
        x0 = None if x_full is None else torch.from_numpy(x_full[b:e].copy()).requires_grad_(True)
        feats, orders, comb = sw.features(k=k, s=scales, X0_local=x0, lambda_max=lam, normalize=normalize,
                                          return_parts=True, edge_weight=ew)
        loss = (feats.double() * torch.from_numpy(hbar[b:e])).sum() + (comb.double() * torch.from_numpy(cbar[b:e])).sum()
        loss.backward()
        dA, dlam = adjacency_vjp(adj, k, scales, x_full, lam_val, normalize, hbar, cbar)
        # every rank's entry gradients, reassembled
        every = [None] * world
        dist.all_gather_object(every, (b, e, ew.grad.numpy().copy(), eng.seen.get("entries"),
                                       {kk: v.numpy() for kk, v in eng.seen.items() if kk != "entries"},
                                       sw.dinv.numpy() if not stored_weights else None))
        coo = adj.tocoo()
        ref = dA[coo.row, coo.col]
        got = np.concatenate([v[2] for v in every])
        assert np.linalg.norm(got - ref) <= 1e-5 * np.linalg.norm(ref), np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert abs(float(lam.grad) - dlam) <= 1e-5 * max(1.0, abs(dlam)), (float(lam.grad), dlam)
        # the plumbing, to 1e-10: the same terms from every rank's b_k and T_k in float64
        if k >= 1:
            b_full = np.concatenate([v[4]["b_all"] for v in every], axis=1).astype(np.float64)
            t_full = np.concatenate([v[4]["t_all"] for v in every], axis=1).astype(np.float64)
            A = adj.toarray().astype(np.float64)
            off = A - np.diag(np.diag(A))
            w = off.sum(axis=0)
            iso = w == 0
            d = np.where(iso, 1.0, 1.0 / np.sqrt(np.where(iso, 1.0, w)))
            a = 2.0 / lam_val
            G = sum((1.0 if i == 1 else 2.0) * (d[:, None] * b_full[i]) @ (d[:, None] * t_full[i - 1]).T
                    for i in range(1, k + 1))
            gw = np.where(iso, 0.0, 0.5 * a * d * d * ((off * G).sum(axis=1) + (off * G).sum(axis=0)))
            grho = b_full[0][:, 0] / (1.0 + A.sum(axis=1)) if f == 1 else np.zeros(n)
            dA2 = -a * G + gw[None, :]
            np.fill_diagonal(dA2, 0.0)
            dA2 += grho[:, None]
            want = dA2[coo.row, coo.col]
            ent = np.concatenate([v[3] for v in every])
            assert np.abs(ent - want).max() <= 1e-10 * np.abs(want).max(), np.abs(ent - want).max()
            zero = np.zeros((n, f))
            dl = -sum(float((b_full[i] * (t_full[i] + (t_full[i - 2] if i >= 2 else zero) +
                                          (1.0 if i == 1 else 2.0) * t_full[i - 1])).sum())
                      for i in range(1, k + 1)) / lam_val
            assert abs(float(lam.grad) - dl) <= 1e-10 * max(1.0, abs(dl))
        else:
            assert float(lam.grad) == 0.0
        if x0 is not None:
            assert x0.grad is not None and x0.grad.shape == x0.shape
        # identical bits of lambda_max.grad on every rank, the same collectives in the same order
        bits = [None] * world
        dist.all_gather_object(bits, lam.grad.numpy().tobytes())
        assert all(v == bits[0] for v in bits)
        logs = [None] * world
        dist.all_gather_object(logs, comm.log)
        assert all(lg == logs[0] for lg in logs)
        # the weighted kernels ran, and flips refuse a weight gradient
        assert any(c.endswith(".w") for c in eng.calls) or sw.rows == 0 or k == 0
        with pytest.raises(ValueError):
            sw.features(k=k, s=scales, edge_weight=ew, deltas=([0], [1], [1.0]))
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


CASES = {
    # graph, f, k, scales, normalize, lambda_max, weights stored in the shard
    "default_signal_k3": ("dir", 1, 3, [0.8, 1.6], True, 2.0, True),
    "custom_f3_k1": ("dir", 3, 1, [0.8], False, 1.7, False),
    "custom_f3_k4": ("dir", 3, 4, [0.8, 1.2], True, 2.0, True),
    "default_signal_k0": ("dir", 1, 0, [0.8], False, 2.0, True),
    "tiny_empty_rank": ("tiny", 1, 3, [0.8], True, 2.3, True),
}


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", sorted(CASES))
def test_sharded_structure_grad_gloo(world, name):
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, CASES[name], ret), nprocs=world, join=True)
    assert [ret.get(r) for r in range(world)] == ["ok"] * world


def _mixed_worker(rank, world, port, ret):
    """Rank 0 stores weights, the other ranks pass a binary shard: every rank then runs the weighted
    path (unit weights on the binary ranks) and the same collectives."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from adjacency_reference import adjacency_vjp
        from efficient_gnn_b200 import sharded
        from vjp_reference import wavelet_vjp
        adj = weighted_graph(301, 4)
        n, f, k, scales = adj.shape[0], 3, 3, [0.8, 1.6]
        part = sharded.RowPartition(n, world)
        ref = adj.copy()
        ref.data[ref.indptr[part.end(0)]:] = 1.0         # what the binary ranks' rows mean
        rp = torch.from_numpy(adj.indptr.astype(np.int32))
        ci = torch.from_numpy(adj.indices.astype(np.int32))
        rpl, cil = part.slice_csr(rp, ci, rank)
        b, e = part.begin(rank), part.end(rank)
        vals = torch.from_numpy(adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)) if rank == 0 else None
        comm = RecordingComm()
        eng = WeightedNumpyEngine()
        eng.fake_plan = object()                          # every rank would take the plan when binary
        sw = sharded.ShardedWavelet(rpl, cil, n, engine=eng, device="cpu", comm=comm, vals_local=vals)
        assert sw.plan is None and sw.vals is not None
        if rank:
            assert torch.equal(sw.vals, torch.ones(cil.numel()))
        rng = np.random.default_rng(17)
        x_full = rng.standard_normal((n, f)).astype(np.float32)
        hbar = rng.standard_normal((n, len(scales) * f))
        x0 = torch.from_numpy(x_full[b:e].copy()).requires_grad_(True)
        lam = torch.tensor(2.0, dtype=torch.float64, requires_grad=True)
        feats = sw.features(k=k, s=scales, X0_local=x0, lambda_max=lam)
        (feats.double() * torch.from_numpy(hbar[b:e])).sum().backward()
        xw, _ = wavelet_vjp(ref, k, scales, x_full, 2.0, True, hbar)
        _, dlam = adjacency_vjp(ref, k, scales, x_full, 2.0, True, hbar)
        every = [None] * world
        dist.all_gather_object(every, (b, e, x0.grad.numpy().copy()))
        got = np.zeros((n, f))
        for bb, ee, g in every:
            got[bb:ee] = g
        assert np.abs(got - xw).max() <= 1e-5 * np.abs(xw).max(), np.abs(got - xw).max()
        assert abs(float(lam.grad) - dlam) <= 1e-5 * max(1.0, abs(dlam)), (float(lam.grad), dlam)
        logs = [None] * world
        dist.all_gather_object(logs, comm.log)
        assert all(lg == logs[0] for lg in logs)
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_mixed_weighted_binary_gloo(world):
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_mixed_worker, args=(world, port, ret), nprocs=world, join=True)
    assert [ret.get(r) for r in range(world)] == ["ok"] * world


# ---- argument errors of the new entry points (no GPU: nothing is launched) ------------------------
BASE = 1 << 20


def ok(i):
    return BASE + 4096 * i               # 16-byte aligned fakes


def test_order_and_adjoint_vals_argument_errors():
    from efficient_gnn_b200 import _cabi
    lib = _cabi.load()
    coeffs = np.ones(16, dtype=np.float32)

    def order(vl=ok(3), vr=ok(6), rows=(0, 4), tprev=ok(10)):
        return lib.egnn_cheb_order_sharded_vals(ok(1), ok(2), vl, ok(4), ok(5), vr, ok(7), ok(8), ok(9), tprev, None,
                                                ok(12), ok(13), ok(14), 8, 4, rows[0], rows[1], 4, 1, 3, 1,
                                                coeffs.ctypes.data, 1.0, -1.0, 0, 0, None, None, None, 0, None)

    assert order(tprev=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert order(rows=(3, 9)) == -1 and b"row range" in lib.egnn_last_error()
    assert order(vr=None) == -1 and b"come together" in lib.egnn_last_error()

    def adj(vl=ok(3), vr=ok(6), cbar=ok(15), rows=(0, 4)):
        return lib.egnn_cheb_adjoint_sharded_vals(ok(1), ok(2), vl, ok(4), ok(5), vr, ok(7), ok(8), ok(9), ok(10),
                                                  None, ok(12), cbar, None, ok(16), 8, 4, rows[0], rows[1], 4, 1, 3,
                                                  1, coeffs.ctypes.data, 1.0, -1.0, 0, None, None, None, 0, None)

    assert adj(cbar=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert adj(rows=(5, 4)) == -1 and b"row range" in lib.egnn_last_error()
    assert adj(vl=None) == -1 and b"come together" in lib.egnn_last_error()
    assert adj(cbar=ok(15) + 4) == -1 and b"16-byte aligned" in lib.egnn_last_error()


def test_wide_adjoint_all_argument_errors():
    from efficient_gnn_b200 import _cabi
    lib = _cabi.load()
    coeffs = np.ones(16, dtype=np.float32)
    w = _cabi.PeerWindowStruct()
    w.rank, w.world, w.rows_per, w.f = 0, 2, 4, 8
    w.base[0], w.base[1] = ok(20), ok(30)

    def wide(b_out=ok(9), cbar=ok(6), win=True, rows=(0, 4)):
        return lib.egnn_wide_adjoint_sharded_all(ok(1), ok(2), ok(3), None, ok(4), ok(5), cbar, None, ok(8), b_out, 8,
                                                 rows[0], rows[1], 8, 1, 3, 1, coeffs.ctypes.data, 1.0, -1.0, None,
                                                 None, None, 0, C.byref(w) if win else None, None)

    assert wide(win=False) == -1 and b"null pointer" in lib.egnn_last_error()
    assert wide(rows=(2, 9)) == -1 and b"row range" in lib.egnn_last_error()
    assert wide(b_out=ok(9) + 4) == -1 and b"16-byte aligned" in lib.egnn_last_error()
    assert wide(cbar=ok(6) + 8) == -1 and b"16-byte aligned" in lib.egnn_last_error()


def test_structure_grad_sharded_argument_errors():
    from efficient_gnn_b200 import _cabi
    lib = _cabi.load()
    assert lib.egnn_adj_grad_stacks_sharded(ok(1), 4, ok(2), 4, ok(3), 8, 2, 1, 4, 3, ok(4), ok(5), None) == -1
    assert b"row range" in lib.egnn_last_error()
    assert lib.egnn_adj_grad_stacks_sharded(ok(1), 2, ok(2), 4, ok(3), 8, 0, 4, 4, 3, ok(4), ok(5), None) == -1
    assert b"shorter" in lib.egnn_last_error()
    assert lib.egnn_adj_grad_stacks_sharded(None, 4, ok(2), 4, ok(3), 8, 0, 4, 4, 3, ok(4), ok(5), None) == -1
    assert b"null pointer" in lib.egnn_last_error()
    ws = lib.egnn_adj_grad_degree_sharded_ws_bytes(4)

    def degree(pl=ok(10), g=ok(13), rows=(0, 4), f=4, vals=None, vals_t=None, wsb=ws):
        return lib.egnn_adj_grad_degree_sharded(ok(1), ok(2), vals, None, ok(4), ok(5), vals_t, None, ok(7), ok(8), 8,
                                                rows[0], rows[1], f, 3, 1.0, pl, ok(11), None, None, g, ok(14),
                                                ok(15), ok(16), wsb, None)

    assert degree(g=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert degree(rows=(4, 10)) == -1 and b"row range" in lib.egnn_last_error()
    assert degree(vals=ok(3)) == -1 and b"come together" in lib.egnn_last_error()
    assert degree(pl=None) == -1 and b"stacks" in lib.egnn_last_error()
    assert degree(pl=ok(10) + 4) == -1 and b"16-byte aligned" in lib.egnn_last_error()
    assert degree(wsb=ws - 1) != 0 and b"too small" in lib.egnn_last_error()
    assert degree(pl=ok(10) + 4, f=3, rows=(4, 4)) == 0     # K*F = 9: scalar loads; no rows: nothing to do

    def entries(gw=ok(5), rows=(0, 4)):
        return lib.egnn_adj_grad_entries_sharded(ok(1), ok(2), 8, rows[0], rows[1], 3, ok(4), gw, ok(6), 1.0, ok(7),
                                                 None)

    assert entries(gw=None) == -1 and b"null pointer" in lib.egnn_last_error()
    assert entries(rows=(6, 9)) == -1 and b"row range" in lib.egnn_last_error()
    assert entries(gw=None, rows=(4, 4)) == 0          # a rank without rows: nothing to write
