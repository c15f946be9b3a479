"""Backward of the row-sharded pass on ONE GPU: the ranks of a 1/2/3/4-way partition run as processes
sharing the device, with a gloo exchange staged through host memory standing in for NCCL.  (Host
threads, as in tests/test_gpu_sharded.py, cannot drive a collective backward: torch runs the backward
of every CUDA graph on one worker thread per device, so one rank's node waiting in a collective
would block the other ranks' nodes behind it.)  This covers the generic path, the adjoint
instantiations of cheb_order_kernel over the local and remote halves of the (transposed) shard,
against the float64 ``wavelet_vjp`` at the DESIGN.md section 10 bars; the fused peer exchange needs
one GPU per rank (tests/test_gpu_sharded_backward_peer.py)."""
import os
import socket
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import elementwise_ratio, rel_max_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


class StagedComm:
    """Collectives of ShardedWavelet over gloo, staged through host memory (tests only)."""

    def __init__(self):
        self.rank, self.world = dist.get_rank(), dist.get_world_size()

    def allreduce(self, t):
        c = t.cpu()
        dist.all_reduce(c)
        t.copy_(c)

    def allgather(self, full, slab):
        c = torch.empty(full.shape, dtype=full.dtype)
        dist.all_gather_into_tensor(c, slab.contiguous().cpu())
        full.copy_(c)

    def alltoall(self, out, inp, out_splits, in_splits):
        c = torch.empty(out.shape, dtype=out.dtype)
        dist.all_to_all_single(c, inp.contiguous().cpu(), out_splits, in_splits)
        out.copy_(c)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def graph(n, directed, seed=5):
    """Binary graph, mean row length ~8, self loops on a few nodes, nodes 3 and n-4 isolated.  Directed:
    an in-star on node 0 (about n/2 rows point at it, node 0 itself has a short row), so the long
    row of the backward exists only in the transpose; otherwise the graph is mirrored."""
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=8.0 / n, random_state=rng, format="lil")
    if directed:
        a[:, 0] = 0
        a[rng.choice(np.arange(5, n), size=n // 2, replace=False), 0] = 1.0
    for i in (3, n - 4):
        a[i, :] = 0
        a[:, i] = 0
    for i in (7, 11):
        a[i, i] = 1.0
    a = sp.csr_matrix(a)
    a.data[:] = 1.0
    if not directed:
        a = (a + a.T) > 0
    a = sp.csr_matrix(a, dtype=np.float32)
    a.sort_indices()
    return a


def flips64(adj):
    """64 flips with global ids: adds, removals, one on the diagonal, and the removal of every in-edge
    of one node (its column empties)."""
    n = adj.shape[0]
    dense = adj.toarray()
    rng = np.random.default_rng(17)
    col = 40
    while not 0 < int((dense[:, col] != 0).sum() - dense[col, col]) <= 6:
        col += 1
    rows, cols, vals = [], [], []
    for u in np.nonzero(dense[:, col])[0]:
        if u != col:
            rows.append(int(u)); cols.append(col); vals.append(-1.0)
    rows.append(9); cols.append(9); vals.append(1.0 - 2 * float(dense[9, 9]))
    while len(rows) < 64:
        u, v = (int(x) for x in rng.integers(0, n, 2))
        if (u, v) in zip(rows, cols) or u == col or v == col:
            continue
        rows.append(u); cols.append(v); vals.append(1.0 - 2 * float(dense[u, v]))
    for u, v, w in zip(rows, cols, vals):
        dense[u, v] += w
    return (rows, cols, vals), sp.csr_matrix(dense.astype(np.float32))


# name: n, f, k, scales, directed, normalize, custom signal (False: only s requires grad), flips, return_parts
CASES = {
    "f1_sym_k3": (3001, 1, 3, [0.8], False, False, True, False, True),
    "f3_dir_k3_s3": (3001, 3, 3, [0.8, 1.2, 2.0], True, True, True, False, True),
    "f8_sym_k1": (3001, 8, 1, [0.8], False, True, True, False, False),
    "f37_dir_k20": (3001, 37, 20, [0.8, 1.6, 2.4], True, True, True, False, False),
    "f130_dir_k3_flips": (3001, 130, 3, [0.8], True, False, True, True, True),
    "f8_dir_k0": (3001, 8, 0, [0.8, 1.6, 2.4], True, True, True, False, True),
    "f1_dir_k20_flips": (3001, 1, 20, [0.8], True, False, True, True, False),
    "default_signal_s_only": (3001, 1, 3, [0.8, 1.6, 2.4], True, False, False, False, True),
}


def order_instance(f):
    """The adjoint instantiation of cheb_order_kernel egnn_cheb_adjoint_sharded picks for width f."""
    vec, u = (4, 1) if f % 4 == 0 else ((1, 1) if f <= 32 else (1, 4))
    return f"cheb_order_kernel<{vec}, {u}, false, false, true>"


def run_case(sw, case, x_full, deltas, dev, profile):
    n, f, k, scales, directed, normalize, custom, flips, parts = case
    b, e = sw.row_begin, sw.row_end
    rng = np.random.default_rng(11)
    n_s = len(scales)
    hbar = torch.from_numpy(rng.standard_normal((n, n_s * f)).astype(np.float32)).to(dev)
    cbar = torch.from_numpy(rng.standard_normal((n, n_s, f)).astype(np.float32)).to(dev)
    tbar = torch.from_numpy(rng.standard_normal((k + 1, n, f)).astype(np.float32)).to(dev)

    def once():
        s_t = torch.tensor(scales, dtype=torch.float64, requires_grad=True)
        x0 = torch.from_numpy(x_full[b:e].copy()).to(dev).requires_grad_(True) if custom else None
        out = sw.features(k=k, s=s_t, X0_local=x0, normalize=normalize, return_parts=parts, deltas=deltas)
        if parts:
            feats, orders, comb = out
            assert feats.grad_fn is not None and comb.grad_fn is not None and all(o.grad_fn for o in orders)
            loss = (feats * hbar[b:e]).sum() + (comb * cbar[b:e]).sum()
            for i, o in enumerate(orders):
                loss = loss + (o * tbar[i, b:e]).sum()
        else:
            assert out.grad_fn is not None
            loss = (out * hbar[b:e]).sum()
        loss.backward()
        torch.cuda.synchronize()
        return (None if x0 is None else x0.grad.cpu().numpy()), s_t.grad.numpy().copy()

    names = []
    if profile:
        from torch.profiler import ProfilerActivity, profile as prof
        with prof(activities=[ProfilerActivity.CUDA]) as p:
            g1 = once()
        names = sorted({ev.name for ev in p.events() if ev.device_type == torch.autograd.DeviceType.CUDA})
    else:
        g1 = once()
    g2 = once()
    same = (g1[0] is None or np.array_equal(g1[0], g2[0])) and np.array_equal(g1[1], g2[1])
    return {"b": b, "e": e, "x": g1[0], "s": g1[1].tobytes(), "repeat_bits": same, "kernels": names}


def _worker(rank, world, port, names, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(0)
        dev = torch.device("cuda", 0)
        from efficient_gnn_b200 import sharded
        import efficient_gnn_b200 as egnn
        for name in names:
            case = CASES[name]
            n, f, k, scales, directed, normalize, custom, flips, parts = case
            adj = graph(n, directed)
            deltas = flips64(adj)[0] if flips else None
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(n, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            sw = sharded.ShardedWavelet(rpl, cil, n, device=dev, comm=StagedComm())
            x_full = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)
            xl = torch.from_numpy(x_full[sw.row_begin:sw.row_end].copy()).to(dev) if custom else None
            # a no-grad call before and after the differentiable ones: same launches, same bits, no grad_fn
            sw.launches = 0
            before = sw.features(k=k, s=scales, X0_local=xl, deltas=deltas)
            launches_before = sw.launches
            res = run_case(sw, case, x_full, deltas, dev, profile=True)
            sw.launches = 0
            after = sw.features(k=k, s=scales, X0_local=xl, deltas=deltas)
            res["nograd_same"] = (sw.launches == launches_before and after.grad_fn is None
                                  and torch.equal(before, after))
            if world == 1:            # the single-GPU pass on the same graph, same loss
                g = egnn.CsrGraph(rp, ci, None, n)
                s_t = torch.tensor(scales, dtype=torch.float64, requires_grad=True)
                x0 = torch.from_numpy(x_full).to(dev).requires_grad_(True) if custom else None
                rng = np.random.default_rng(11)
                n_s = len(scales)
                hbar = torch.from_numpy(rng.standard_normal((n, n_s * f)).astype(np.float32)).to(dev)
                cbar = torch.from_numpy(rng.standard_normal((n, n_s, f)).astype(np.float32)).to(dev)
                tbar = torch.from_numpy(rng.standard_normal((k + 1, n, f)).astype(np.float32)).to(dev)
                out = egnn.graph_wavelet_features(g, k=k, s=s_t, X0=x0, normalize=normalize, return_parts=parts,
                                                  deltas=deltas)
                if parts:
                    loss = (out.features * hbar).sum() + (out.combined * cbar).sum()
                    for i, o in enumerate(out.orders):
                        loss = loss + (o * tbar[i]).sum()
                else:
                    loss = (out * hbar).sum()
                loss.backward()
                res["single_x"] = None if x0 is None else x0.grad.cpu().numpy()
                res["single_s"] = s_t.grad.numpy()
                res["symmetric_dropped"] = sw._adjoint_shard is False
            ret[(rank, name)] = res
    finally:
        dist.destroy_process_group()


def _reference(name):
    from vjp_reference import wavelet_vjp
    n, f, k, scales, directed, normalize, custom, flips, parts = CASES[name]
    adj = graph(n, directed)
    ref_adj = flips64(adj)[1] if flips else adj
    rng = np.random.default_rng(11)
    n_s = len(scales)
    hbar = rng.standard_normal((n, n_s * f)).astype(np.float32)
    cbar = rng.standard_normal((n, n_s, f)).astype(np.float32)
    tbar = rng.standard_normal((k + 1, n, f)).astype(np.float32)
    x_full = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32) if custom else None
    if not parts:
        cbar = tbar = None
    return wavelet_vjp(ref_adj, k, scales, x_full, 2.0, normalize, hbar, cbar, tbar)


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_sharded_backward_matches_vjp(world):
    names = sorted(CASES)
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), names, ret), nprocs=world, join=True)
    for name in names:
        n, f, k, scales, directed, normalize, custom, flips, parts = CASES[name]
        xw, sbar = _reference(name)
        tol = 1e-5 if k <= 16 else 1e-4
        res = [ret[(r, name)] for r in range(world)]
        assert all(r["repeat_bits"] for r in res), f"{name}: two backward passes differ"
        assert all(r["nograd_same"] for r in res), f"{name}: the no-grad call changed"
        assert all(r["s"] == res[0]["s"] for r in res), f"{name}: s.grad differs between ranks"
        s_got = np.frombuffer(res[0]["s"], dtype=np.float64)
        assert rel_max_err(s_got, sbar) <= tol, (name, s_got, sbar)
        msg = f"world {world} {name}: s.grad rel err {rel_max_err(s_got, sbar):.2e}"
        if custom:
            got = np.zeros((n, f))
            for r in res:
                got[r["b"]:r["e"]] = r["x"].reshape(r["e"] - r["b"], f)
            nw, el = rel_max_err(got, xw), elementwise_ratio(got, xw, tol)
            el3 = elementwise_ratio(got, xw, tol, floor=1e-3)
            msg += f", X0.grad norm-wise {nw:.2e}, element-wise {el:.2f} (1e-3 floor {el3:.2f})"
            assert nw <= tol and el <= 1.0, msg
            if world == 1:
                d = np.abs(got - res[0]["single_x"]).max()
                msg += f", max |diff| to graph_wavelet_features {d:.2e}"
                assert rel_max_err(got, res[0]["single_x"]) <= tol, msg
        if world == 1:
            assert rel_max_err(s_got, res[0]["single_s"]) <= tol, msg
            assert res[0]["symmetric_dropped"] == (custom and k >= 1 and not directed)
        # the instantiation each case names ran in its backward
        kernels = " ".join(n_ for r in res for n_ in r["kernels"])
        assert not custom or "adjoint_prologue_kernel" in kernels, (name, kernels)
        if custom and k >= 1:
            assert order_instance(f) in kernels, (name, order_instance(f), kernels)
        print(msg)
