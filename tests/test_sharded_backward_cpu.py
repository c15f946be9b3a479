"""Host logic of the row-sharded backward on CPU: world 2 and 3 over gloo, with a NumPy engine whose
adjoint methods restate one application of ``M^T`` (and the coefficient gradient) in float64.  What
is under test is the transposed-shard build, symmetric-shard detection, the transposed flips, the
exchange order of the adjoint and the rank-order sum of the scale gradient - the arithmetic is the
reference's, so any mismatch with ``wavelet_vjp`` is plumbing."""
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

from test_sharded_cpu import NumpyEngine  # noqa: E402


class AdjointNumpyEngine(NumpyEngine):
    """NumpyEngine plus the backward methods of CudaEngine (tests only)."""

    def adjoint(self, phase, local, remote, dinv, iso, b_prev_full, b_prev_local, b_prev2_local, b_out_local, cbar,
                tbar, acc_ws, n_global, nnz_hint, row_begin, row_end, f, app, k_max, n_scales, coeffs, op_scale,
                op_shift, deltas_t=None):
        self.calls.append(f"adj{app}.phase{phase}")
        rows, m = row_end - row_begin, k_max - app
        cb = cbar.numpy()[:rows].astype(np.float64)
        v = sum(float(coeffs[s, m]) * cb[:, s, :] for s in range(n_scales))
        if tbar is not None:
            v = v + tbar.numpy()[m, :rows]
        if app == 0:
            b_out_local.numpy()[:rows] = v
            return
        d = dinv.numpy().astype(np.float64)
        if phase == 0:
            rp, ci = local[0].numpy(), local[1].numpy()
            src, off = b_prev_local.numpy().astype(np.float64), row_begin
        else:
            rp, ci = remote[0].numpy(), remote[1].numpy()
            src, off = b_prev_full.numpy().astype(np.float64), 0
        acc = np.zeros((rows, f))
        r = np.repeat(np.arange(rows), np.diff(rp))
        keep = ci != (r + row_begin)
        np.add.at(acc, r[keep], d[ci[keep], None] * src[ci[keep] - off])
        if phase == 0:
            assert deltas_t is None
            acc_ws.numpy()[:rows] = acc
            return
        for dr, dc, dv in zip(*(deltas_t or ([], [], []))):
            if row_begin <= dr < row_end and dr != dc:
                acc[dr - row_begin] += dv * d[dc] * src[dc]
        acc += acc_ws.numpy()[:rows]
        di = d[row_begin:row_end, None]
        theta = (op_scale * (1 - iso.numpy()[row_begin:row_end]) + op_shift)[:, None]
        own = b_prev_local.numpy()[:rows].astype(np.float64)
        b2 = 0.0 if b_prev2_local is None else b_prev2_local.numpy()[:rows]
        b_out_local.numpy()[:rows] = (1.0 if m == 0 else 2.0) * (theta * own - op_scale * di * acc) + v - b2

    def coeff_grad(self, cbar, t_all):
        cb, t = cbar.numpy().astype(np.float64), t_all.numpy().astype(np.float64)
        return torch.from_numpy(np.einsum("rsf,krf->sk", cb, t))

    def l1_normalize(self, comb):
        return comb / (comb.abs().sum(dim=2, keepdim=True) + 1e-8)


class RecordingComm:
    """DistComm that logs every collective (name and shape) it runs."""

    def __init__(self):
        from efficient_gnn_b200 import sharded
        self.inner = sharded.DistComm()
        self.rank, self.world = self.inner.rank, self.inner.world
        self.log = []

    def allreduce(self, t):
        self.log.append(("allreduce", tuple(t.shape)))
        self.inner.allreduce(t)

    def allgather(self, full, slab):
        self.log.append(("allgather", tuple(full.shape)))
        self.inner.allgather(full, slab)

    def alltoall(self, out, inp, out_splits, in_splits):
        self.log.append(("alltoall", inp.dim()))
        self.inner.alltoall(out, inp, out_splits, in_splits)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def directed_graph(n, seed, symmetric):
    """Binary graph with an in-star hub (node 0 is the column of a long column, a short row), isolated
    nodes and self loops; ``symmetric`` mirrors it."""
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=6.0 / n, random_state=rng, format="lil")
    a[:, 0] = 0
    a[rng.choice(np.arange(5, n), size=n // 3, replace=False), 0] = 1.0       # in-star on node 0
    a[3, :] = 0
    a[:, 3] = 0                                                            # node 3 isolated
    for i in (7, 11):
        a[i, i] = 1.0
    a = sp.csr_matrix(a)
    a.data[:] = 1.0
    if symmetric:
        a = ((a + a.T) > 0).astype(np.float32)
    a = sp.csr_matrix(a, dtype=np.float32)
    a.sort_indices()
    return a


def _worker(rank, world, port, case, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from efficient_gnn_b200 import sharded
        from vjp_reference import wavelet_vjp
        n, f, k, scales, symmetric, normalize, custom, flips = case
        adj = directed_graph(n, 5, symmetric)
        deltas = None
        ref_adj = adj
        if flips:
            dense = adj.toarray()
            rows, cols, vals = [], [], []
            for u, v in [(1, 0), (n - 1, 2), (4, n // 2), (9, 9), (n // 3, n - 2)]:
                w = float(1 - 2 * dense[u, v])
                dense[u, v] += w
                rows.append(u); cols.append(v); vals.append(w)
            # remove node 20's last in-edge: column 20 becomes empty
            for u in np.nonzero(dense[:, 20])[0]:
                if u != 20:
                    rows.append(int(u)); cols.append(20); vals.append(-1.0)
                    dense[u, 20] = 0.0
            deltas = (rows, cols, vals)
            ref_adj = sp.csr_matrix(dense.astype(np.float32))
        rp = torch.from_numpy(adj.indptr.astype(np.int32))
        ci = torch.from_numpy(adj.indices.astype(np.int32))
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        comm = RecordingComm()
        eng = AdjointNumpyEngine()
        sw = sharded.ShardedWavelet(rpl, cil, n, engine=eng, device="cpu", comm=comm)
        b, e = sw.row_begin, sw.row_end
        rng = np.random.default_rng(11)
        x_full = rng.standard_normal((n, f)).astype(np.float32) if custom else None
        n_s = len(scales)
        hbar = rng.standard_normal((n, n_s * f))
        cbar = rng.standard_normal((n, n_s, f))
        tbar = rng.standard_normal((k + 1, n, f))
        s_t = torch.tensor(scales, dtype=torch.float64, requires_grad=True)
        x0 = None
        if custom:
            x0 = torch.from_numpy(x_full[b:e].copy()).requires_grad_(True)
        feats, orders, comb = sw.features(k=k, s=s_t, X0_local=x0, normalize=normalize, return_parts=True,
                                          deltas=deltas)
        assert feats.grad_fn is not None and comb.grad_fn is not None and all(o.grad_fn for o in orders)
        loss = (feats.double() * torch.from_numpy(hbar[b:e])).sum() + (comb.double() * torch.from_numpy(cbar[b:e])).sum()
        for i, o in enumerate(orders):
            loss = loss + (o.double() * torch.from_numpy(tbar[i, b:e])).sum()
        loss.backward()
        xw, sw_ref = wavelet_vjp(ref_adj, k, scales, x_full, 2.0, normalize, hbar, cbar, tbar)
        if custom:
            g = torch.zeros((part.rows_per, f))
            g[:sw.rows] = x0.grad
            full = torch.empty((world * part.rows_per, f))
            dist.all_gather_into_tensor(full, g)
            got = full[:n].numpy()
            assert np.abs(got - xw).max() <= 1e-5 * np.abs(xw).max(), np.abs(got - xw).max()
        np.testing.assert_allclose(s_t.grad.numpy(), sw_ref, rtol=1e-5, atol=1e-6 * np.abs(sw_ref).max())
        # identical bits of s.grad on every rank
        every = [None] * world
        dist.all_gather_object(every, s_t.grad.numpy().tobytes())
        assert all(v == every[0] for v in every)
        # the transposed shard: built once, dropped when every shard equals its transpose
        if not custom or k == 0:
            assert sw._adjoint_shard is None          # no application of M^T: nothing built, nothing exchanged
        elif symmetric:
            assert sw._adjoint_shard is False
        else:
            assert sw._adjoint_shard is not False
            rpt, cit = sw._adjoint_shard[:2]
            at = adj.T.tocsr()
            at.sort_indices()
            assert np.array_equal(rpt.numpy(), at.indptr[b:e + 1] - at.indptr[b])
            assert np.array_equal(cit.numpy(), at.indices[at.indptr[b]:at.indptr[e]])
        # the same collectives in the same order on every rank
        logs = [None] * world
        dist.all_gather_object(logs, comm.log)
        assert all(lg == logs[0] for lg in logs)
        # the adjoint's exchange runs between the two halves of every application
        adj_calls = [c for c in eng.calls if c.startswith("adj") or c in ("fork", "join")]
        if k >= 1 and sw.rows and custom:
            i = adj_calls.index("adj1.phase0")
            assert adj_calls[i - 1] == "fork" and adj_calls[i + 1] == "join" and adj_calls[i + 2] == "adj1.phase1"
        ret[rank] = "ok"
    finally:
        dist.destroy_process_group()


CASES = {
    # n, f, k, scales, symmetric, normalize, custom signal, flips
    "directed": (1003, 3, 4, [0.8, 1.6], False, True, True, False),
    "symmetric": (1003, 2, 3, [0.8], True, False, True, False),
    "directed_flips": (1003, 3, 3, [0.8, 1.6], False, True, True, True),
    "default_signal_s_only": (1003, 1, 3, [0.8, 1.2, 2.0], False, False, False, False),
    "k0": (1003, 2, 0, [0.8], False, True, True, False),
}


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", sorted(CASES))
def test_sharded_backward_gloo(world, name):
    port = _free_port()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, port, CASES[name], ret), nprocs=world, join=True)
    assert [ret.get(r) for r in range(world)] == ["ok"] * world
