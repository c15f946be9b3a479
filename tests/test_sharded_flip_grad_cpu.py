"""Gradients through edge flips on the row-sharded pass (DESIGN.md section 15) on CPU: world 2 and 3 over
gloo, with the NumPy engine of ``test_sharded_structure_grad_cpu`` extended by float64 restatements of the
two flip methods of CudaEngine (and the weighted adjoint with transposed flips).  What is under test is
the host logic: the flip values as an autograd input, the degree vectors patched once for the adjoint and
the gradient terms, the flipped row sums of the default signal, the flips' part of ``R`` / ``Q`` on the
ranks that own their rows and columns, and the rank-order sum of the ranks' flip values.

Bars: the flip values and ``lambda_max`` to 1e-10 against a dense float64 restatement from every rank's
Clenshaw vectors and orders as the pass computed them; norm-wise 1e-5 against ``adjacency_vjp`` of the
dense ``A + delta``; identical ``v.grad`` / ``lambda_max.grad`` bits and collective logs on every rank."""
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

from test_sharded_backward_cpu import RecordingComm  # noqa: E402
from test_sharded_structure_grad_cpu import WeightedNumpyEngine, _spmv_half, tiny_graph, weighted_graph  # noqa: E402


class FlipNumpyEngine(WeightedNumpyEngine):
    """WeightedNumpyEngine plus the flip methods of CudaEngine, in float64 (tests only)."""

    def patch_degrees(self, dinv, iso, x0_local, n_global, row_begin, n_rows, deltas):
        # the base engine's patch, with dinv kept in float64 like this engine's prep
        w, rowsum = self.w_full.copy(), self.rowsum_local.copy()
        for r, c, v in zip(*deltas):
            if r != c:
                w[c] += v
            if row_begin <= r < row_begin + n_rows:
                rowsum[r - row_begin] += v
        is_iso = w == 0
        d2 = np.where(is_iso, 1.0, 1.0 / np.sqrt(np.where(is_iso, 1.0, w)))
        self.calls.append("patch")
        return torch.from_numpy(d2), torch.from_numpy(is_iso.astype(np.uint8)), torch.from_numpy(np.log1p(rowsum))

    def adjoint(self, phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local, b_out_local, cbar,
                tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs, op_scale,
                op_shift, deltas_t=None):
        if phase != 1 or app == 0 or len(remote) == 2 or deltas_t is None:
            return super().adjoint(phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local,
                                   b_out_local, cbar, tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app,
                                   k_max, n_scales, coeffs, op_scale, op_shift, deltas_t)
        # a weighted application with the forward's flips transposed
        self.calls.append(f"adj{app}.phase1.w.flips")
        rows, m = row_end - row_begin, k_max - app
        d = dinv.numpy().astype(np.float64)
        cb = cbar.numpy()[:rows].astype(np.float64)
        v = sum(float(coeffs[s, m]) * cb[:, s, :] for s in range(n_scales))
        if tbar is not None:
            v = v + tbar.numpy()[m, :rows]
        src = b_prev_full.numpy().astype(np.float64)
        acc = _spmv_half(remote, rows, row_begin, d, src, 0) + acc_ws.numpy()[:rows]
        for dr, dc, dv in zip(*deltas_t):
            if row_begin <= dr < row_end and dr != dc:
                acc[dr - row_begin] += dv * d[dc] * src[dc]
        di = d[row_begin:row_end, None]
        theta = (op_scale * (1 - iso.numpy()[row_begin:row_end]) + op_shift)[:, None]
        own = b_prev_local.numpy()[:rows].astype(np.float64)
        b2 = 0.0 if b_prev2_local is None else b_prev2_local.numpy()[:rows]
        b_out_local.numpy()[:rows] = (1.0 if m == 0 else 2.0) * (theta * own - op_scale * di * acc) + v - b2

    def adj_grad_degree_flips(self, shard, shard_t, row_orders, dinv, iso, n_global, row_begin, row_end, f, k,
                              op_scale, pl_full, pt_full, xbar, rowsum, deltas):
        self.calls.append("degree_flips")
        rows = row_end - row_begin

        def dots(csr, own, gath):
            rp, ci, v = csr
            v = np.ones(ci.numel()) if v is None else v.numpy().astype(np.float64)
            r = np.repeat(np.arange(rows), np.diff(rp.numpy()))
            ci = ci.numpy()
            g = np.zeros(ci.size) if k == 0 else (own.numpy()[r + row_begin] * gath.numpy()[ci]).sum(axis=1)
            g[ci == r + row_begin] = 0.0
            out = np.zeros(rows)
            np.add.at(out, r, v * g)
            return g, out

        g, R = dots(shard, pl_full, pt_full)
        _, Q = dots(shard_t, pt_full, pl_full)
        rs, cs, vs = deltas
        g_flips = np.zeros(len(rs)) if k == 0 else \
            np.array([float((pl_full.numpy()[r] * pt_full.numpy()[c]).sum()) for r, c in zip(rs, cs)])
        for p, (r, c, v) in enumerate(zip(rs, cs, vs)):
            if r == c:
                continue
            if row_begin <= r < row_end:
                R[r - row_begin] += v * g_flips[p]
            if row_begin <= c < row_end:
                Q[c - row_begin] += v * g_flips[p]
        d = dinv.numpy()[row_begin:row_end].astype(np.float64)
        is_iso = iso.numpy()[row_begin:row_end] != 0
        gw = np.where(is_iso, 0.0, 0.5 * op_scale * d * d * (R + Q))
        grho = np.zeros(rows) if xbar is None else xbar.numpy().astype(np.float64) / (1.0 + np.asarray(rowsum))
        self.seen["rowsum"] = None if rowsum is None else np.asarray(rowsum, dtype=np.float64).copy()
        return torch.from_numpy(g), torch.from_numpy(gw), torch.from_numpy(grho), torch.from_numpy(g_flips)

    def adj_grad_flips(self, deltas, g_flips, gw_full, grho, n_global, row_begin, row_end, op_scale):
        self.calls.append("flip_values")
        out = np.zeros(len(deltas[0]))
        for p, (r, c) in enumerate(zip(deltas[0], deltas[1])):
            if row_begin <= r < row_end:
                out[p] = grho.numpy()[r - row_begin] + \
                    (0.0 if r == c else -op_scale * g_flips.numpy()[p] + gw_full.numpy()[c])
        self.seen["flip_values"] = out.copy()
        return torch.from_numpy(out)


def binary_graph(n, seed):
    """The pattern of ``weighted_graph`` made binary and symmetric (self loops kept)."""
    a = weighted_graph(n, seed)
    a.data[:] = 1.0
    a.eliminate_zeros()
    s = ((a + a.T) > 0).astype(np.float32)
    s = sp.csr_matrix(s, dtype=np.float32)
    s.sort_indices()
    return s


def make_flips(adj, zero_only=False):
    """Flips of every kind on ``adj`` (global ids): an added entry and a removed stored entry whose rows
    and columns belong to different ranks, a re-weighted entry, two diagonal flips (one on a stored self
    loop), a flip that isolates a column, two flips on one entry and zero-valued candidates on a stored
    and an unstored entry.  Values are sums of few powers of two (the float32 sums of a row's flips are
    exact), except the removals, which are the stored values negated."""
    A = adj.toarray().astype(np.float64)
    n = A.shape[0]
    if n < 10:                       # the tiny graph: one flip of several kinds
        return [0, 3, 1, 2, 0], [2, 3, 2, 0, 1], [1.0, 0.5, -float(A[1, 2]), 0.0, 0.25]
    off = A - np.diag(np.diag(A))
    nz = off != 0
    indeg = nz.sum(axis=0)
    used = set()
    rows, cols, vals = [], [], []

    def add(r, c, v):
        rows.append(int(r)); cols.append(int(c)); vals.append(float(v))
        used.add(int(c))

    # the column with the fewest stored off-diagonal values (one on the weighted graph, unit values on the
    # binary one, so that the removals cancel its in-degree exactly): removing them isolates it
    c_iso = min((c for c in range(n - 1, 5, -1) if indeg[c] >= 1), key=lambda c: indeg[c])
    for r_iso in np.nonzero(nz[:, c_iso])[0]:
        add(r_iso, c_iso, -A[r_iso, c_iso])
    # added entry, row on the first rank, column on the last
    r, c = 10, next(c for c in range(n - 1, n // 2, -1) if A[10, c] == 0 and indeg[c] >= 2)
    add(r, c, 1.0)
    # removed stored entry, row on the last ranks, column on the first, column keeps other entries
    r = next(i for i in range(n - 1, n // 2, -1) if any(nz[i, j] and indeg[j] >= 2 and j not in used and j < n // 3
                                                         for j in range(n)))
    c = next(j for j in range(n // 3) if nz[r, j] and indeg[j] >= 2 and j not in used)
    add(r, c, -A[r, c])
    # re-weighted stored entry
    r, c = next((i, j) for i, j in zip(*np.nonzero(nz)) if indeg[j] >= 2 and j not in used and 100 < i < 200)
    add(r, c, 0.5)
    # diagonal flips: a new self loop and a stored one
    add(20, 20, 0.75)
    add(7, 7, -0.25)
    # two flips on one unstored entry
    c = next(j for j in range(n // 2, n) if A[40, j] == 0 and j not in used and j != 40)
    add(40, c, 0.25)
    add(40, c, 0.5)
    # zero-valued candidates: a stored entry and an unstored one
    r, c = next((i, j) for i, j in zip(*np.nonzero(nz)) if j not in used and i > 200)
    add(r, c, 0.0)
    c = next(j for j in range(n // 3, n) if A[150, j] == 0 and j not in used and j != 150)
    add(150, c, 0.0)
    assert sum(1 for cc in cols if cc == c_iso) == indeg[c_iso]
    assert indeg[c_iso] == 1 or np.all(A[:, c_iso][nz[:, c_iso]] == 1.0)
    return rows, cols, vals


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
        graph, f, k, scales, normalize, lam_val, want = case
        adj = {"weighted": lambda: weighted_graph(301, 4), "binary": lambda: binary_graph(301, 4),
               "tiny": tiny_graph}[graph]()
        n = adj.shape[0]
        rp = torch.from_numpy(adj.indptr.astype(np.int32))
        ci = torch.from_numpy(adj.indices.astype(np.int32))
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        b, e = part.begin(rank), part.end(rank)
        weighted = graph != "binary"
        w_loc = adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)
        comm = RecordingComm()
        eng = FlipNumpyEngine()
        sw = sharded.ShardedWavelet(rpl, cil, n, engine=eng, device="cpu", comm=comm,
                                    vals_local=torch.from_numpy(w_loc) if weighted else None)
        assert (sw.vals is None) == (not weighted)
        rows, cols, vals = make_flips(adj)
        rng = np.random.default_rng(17)
        x_full = rng.standard_normal((n, f)).astype(np.float32) if f > 1 else None
        n_s = len(scales)
        hbar = rng.standard_normal((n, n_s * f))
        cbar = rng.standard_normal((n, n_s, f))
        v = torch.tensor(vals, dtype=torch.float64, requires_grad="v" in want)
        lam = torch.tensor(lam_val, dtype=torch.float64, requires_grad="lam" in want)
        x0 = None if x_full is None else torch.from_numpy(x_full[b:e].copy()).requires_grad_(True)
        eng.calls.clear()
        feats, orders, comb = sw.features(k=k, s=scales, X0_local=x0, lambda_max=lam, normalize=normalize,
                                          return_parts=True, deltas=(rows, cols, v if "v" in want else vals))
        loss = (feats.double() * torch.from_numpy(hbar[b:e])).sum() + \
            (comb.double() * torch.from_numpy(cbar[b:e])).sum()
        loss.backward()
        # the degree vectors are patched once in the backward (and once in the forward)
        assert eng.calls.count("patch") == 2, eng.calls
        assert ("degree_flips" in eng.calls) == ("v" in want)
        assert ("flip_values" in eng.calls) == ("v" in want)
        Ap = adj.toarray().astype(np.float64)
        for r, c, dv in zip(rows, cols, vals):
            Ap[r, c] += np.float64(np.float32(dv))
        dA, dlam = adjacency_vjp(Ap, k, scales, x_full, lam_val, normalize, hbar, cbar)
        ref_v = dA[rows, cols]
        if "v" in want:
            got_v = v.grad.numpy()
            assert v.grad.shape == (len(rows),)
            assert np.linalg.norm(got_v - ref_v) <= 1e-5 * np.linalg.norm(ref_v), \
                np.linalg.norm(got_v - ref_v) / np.linalg.norm(ref_v)
        else:
            assert v.grad is None
        if "lam" in want:
            assert abs(float(lam.grad) - dlam) <= 1e-5 * max(1.0, abs(dlam)), (float(lam.grad), dlam)
        else:
            assert lam.grad is None
        if x0 is not None:
            assert x0.grad is not None and x0.grad.shape == x0.shape
        # the plumbing, to 1e-10: the same terms of A' from every rank's b_k and T_k in float64
        every = [None] * world
        dist.all_gather_object(every, (b, e, {kk: vv.numpy() for kk, vv in eng.seen.items()
                                               if kk in ("b_all", "t_all")}, eng.seen.get("rowsum"),
                                       eng.seen.get("flip_values")))
        if k >= 1 and "v" in want:
            b_full = np.concatenate([x[2]["b_all"] for x in every], axis=1).astype(np.float64)
            t_full = np.concatenate([x[2]["t_all"] for x in every], axis=1).astype(np.float64)
            off = Ap - np.diag(np.diag(Ap))
            w = off.sum(axis=0)
            iso = w == 0
            d = np.where(iso, 1.0, 1.0 / np.sqrt(np.where(iso, 1.0, w)))
            a = 2.0 / lam_val
            G = sum((1.0 if i == 1 else 2.0) * (d[:, None] * b_full[i]) @ (d[:, None] * t_full[i - 1]).T
                    for i in range(1, k + 1))
            gw = np.where(iso, 0.0, 0.5 * a * d * d * ((off * G).sum(axis=1) + (off * G).sum(axis=0)))
            if f == 1 and x_full is None:
                # the flipped row sums as the library rounds them: base sum + float32 sum of the row's flips
                rho = adj.toarray().astype(np.float64).sum(axis=1)
                add = {}
                for r, dv in zip(rows, vals):
                    add[r] = np.float32(add.get(r, np.float32(0.0)) + np.float32(dv))
                for r, s_ in add.items():
                    rho[r] += np.float64(s_)
                got_rho = np.concatenate([x[3] for x in every])
                assert np.abs(got_rho - rho).max() <= 1e-12 * np.abs(rho).max()
                grho = b_full[0][:, 0] / (1.0 + rho)
            else:
                grho = np.zeros(n)
            want_v = np.array([grho[r] + (0.0 if r == c else -a * G[r, c] + gw[c]) for r, c in zip(rows, cols)])
            # every rank's values (the owner's, 0 elsewhere) added in rank order; the float32 pass input
            # hands them back rounded to float32
            got_v = every[0][4]
            for x in every[1:]:
                got_v = got_v + x[4]
            assert np.abs(got_v - want_v).max() <= 1e-10 * np.abs(want_v).max(), np.abs(got_v - want_v).max()
            assert np.array_equal(v.grad.numpy(), got_v.astype(np.float32).astype(np.float64))
            # a repeated entry gives each of its flips the entry's value
            for p in range(len(rows)):
                for q in range(p):
                    if (rows[p], cols[p]) == (rows[q], cols[q]):
                        assert got_v[p] == got_v[q]
            if "lam" in want:
                zero = np.zeros((n, f))
                dl = -sum(float((b_full[i] * (t_full[i] + (t_full[i - 2] if i >= 2 else zero) +
                                              (1.0 if i == 1 else 2.0) * t_full[i - 1])).sum())
                          for i in range(1, k + 1)) / lam_val
                assert abs(float(lam.grad) - dl) <= 1e-10 * max(1.0, abs(dl))
        if k == 0 and "lam" in want:
            assert float(lam.grad) == 0.0
        # identical bits on every rank, the same collectives in the same order
        bits = [None] * world
        dist.all_gather_object(bits, (None if v.grad is None else v.grad.numpy().tobytes(),
                                      None if lam.grad is None else lam.grad.numpy().tobytes()))
        assert all(x == bits[0] for x in bits)
        logs = [None] * world
        dist.all_gather_object(logs, comm.log)
        assert all(lg == logs[0] for lg in logs)
        # an edge weight that requires grad still refuses flips
        if weighted:
            with pytest.raises(ValueError):
                sw.features(k=k, s=scales, edge_weight=torch.from_numpy(w_loc).requires_grad_(True),
                            deltas=(rows, cols, v))
        # a flip-value tensor of the wrong shape is refused
        with pytest.raises(ValueError):
            sw.features(k=k, s=scales, deltas=(rows, cols, torch.zeros(len(rows) + 1, requires_grad=True)))
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


CASES = {
    # graph, f, k, scales, normalize, lambda_max, inputs requiring grad
    "weighted_default_k3": ("weighted", 1, 3, [0.8, 1.6], True, 2.0, ("v", "lam")),
    "binary_default_k3": ("binary", 1, 3, [0.8], False, 1.9, ("v", "lam")),
    "weighted_f3_k1": ("weighted", 3, 1, [0.8], False, 1.7, ("v", "lam")),
    "binary_f3_k3": ("binary", 3, 3, [0.8, 1.2], True, 2.0, ("v", "lam")),
    "weighted_default_k0": ("weighted", 1, 0, [0.8], False, 2.0, ("v", "lam")),
    "binary_f3_k0": ("binary", 3, 0, [0.8], True, 2.0, ("v",)),
    "weighted_f3_k3_lam_only": ("weighted", 3, 3, [0.8], True, 2.0, ("lam",)),
    "binary_default_k3_v_only": ("binary", 1, 3, [0.8, 1.6], True, 2.0, ("v",)),
    "tiny_empty_rank": ("tiny", 1, 3, [0.8], True, 2.3, ("v", "lam")),
}


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", sorted(CASES))
def test_sharded_flip_grad_gloo(world, name):
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, CASES[name], ret), nprocs=world, join=True)
    assert [ret.get(r) for r in range(world)] == ["ok"] * world
