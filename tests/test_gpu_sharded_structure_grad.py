"""Edge-weight and ``lambda_max`` gradients of the row-sharded pass on ONE GPU: the ranks of a 1/2/3/4-way
partition run as processes sharing the device, with the staged gloo exchange of
tests/test_gpu_sharded_backward.py.  Weighted directed graphs (an in-star hub, so the transpose differs
from the shard; an isolated node; stored self loops; explicit zero weights including a column of only
zeros; a rank without rows on the tiny graph) against the float64 ``adjacency_vjp`` / ``forward64`` /
``wavelet_vjp`` at the bars of DESIGN.md sections 10 and 11, and against one-GPU
``graph_wavelet_features`` on the equivalent sparse COO tensor.  Two GPUs: the fused wide exchange and
``EGNN_EXCHANGE=nccl``."""
import os
import re
import socket
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import elementwise_ratio, rel_max_err
from test_gpu_sharded_backward import StagedComm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def weighted_graph(n, seed=4):
    """Directed, weights in [0.2, 2]: in-star on node 0, node 3 isolated, self loops on 7 and 11,
    explicit zeros at (2, 8) and (4, 1), and column 5 holding only explicit zeros."""
    if n == 4:
        return sp.csr_matrix(np.array([[0.0, 1.5, 0.0, 0.5], [0.0, 0.7, 2.0, 0.0], [1.0, 0.0, 0.0, 0.0],
                                       [0.0, 0.0, 3.0, 0.0]], np.float32))
    rng = np.random.default_rng(seed)
    a = sp.random(n, n, density=6.0 / n, random_state=rng, format="lil")
    a[:, 0] = 0
    a[rng.choice(np.arange(6, n), size=n // 2, replace=False), 0] = 1.0
    a[3, :] = 0
    a[:, 3] = 0
    a[:, 5] = 0
    a[2, 8] = 0                       # free the positions of the explicit zeros below, so that
    a[4, 1] = 0                       # sum_duplicates keeps them zero
    for i in (7, 11):
        a[i, i] = 1.0
    a = sp.coo_matrix(a)
    a.eliminate_zeros()
    vals = rng.uniform(0.2, 2.0, a.nnz)
    rows = np.concatenate([a.row, [1, 9, 2, 4]])
    cols = np.concatenate([a.col, [5, 5, 8, 1]])
    vals = np.concatenate([vals, [0.0, 0.0, 0.0, 0.0]]).astype(np.float32)
    m = sp.coo_matrix((vals, (rows, cols)), shape=(n, n)).tocsr()
    m.sum_duplicates()
    m.sort_indices()
    return m


N = 1001
# name: n, f, k, scales, normalize, lambda_max, weights stored in the shard (else passed per call)
CASES = {
    "f1_default_k3_s3": (N, 1, 3, [0.8, 1.6, 2.4], True, 2.0, True),
    "f1_default_k0": (N, 1, 0, [0.8], False, 2.0, True),
    "f1_default_k1_binary_shard": (N, 1, 1, [0.8], False, 1.6, False),
    "f3_k3_s3": (N, 3, 3, [0.8, 1.2, 2.0], True, 2.0, True),
    "f8_k3_binary_shard": (N, 8, 3, [0.8], False, 2.5, False),
    "f37_k17": (N, 37, 17, [0.8], True, 2.0, True),
    "f130_k3_s3": (N, 130, 3, [0.8, 1.6, 2.4], False, 2.0, True),
    "tiny_f1_default_k3": (4, 1, 3, [0.8], True, 2.0, True),
}


def _loss_arrays(n, f, k, n_s):
    rng = np.random.default_rng(11)
    return (rng.standard_normal((n, n_s * f)).astype(np.float32), rng.standard_normal((n, n_s, f)).astype(np.float32))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_case(sw, case, adj, dev, comm_rank):
    n, f, k, scales, normalize, lam_val, stored = case
    b, e = sw.row_begin, sw.row_end
    w_loc = adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)
    hbar, cbar = (torch.from_numpy(a).to(dev) for a in _loss_arrays(n, f, k, len(scales)))
    x_full = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32) if f > 1 else None

    def once():
        ew = torch.from_numpy(w_loc).to(dev).requires_grad_(True)
        lam = torch.tensor(lam_val, dtype=torch.float64, requires_grad=True)
        x0 = None if x_full is None else torch.from_numpy(x_full[b:e].copy()).to(dev).requires_grad_(True)
        feats, orders, comb = sw.features(k=k, s=scales, X0_local=x0, lambda_max=lam, normalize=normalize,
                                          return_parts=True, edge_weight=ew)
        loss = (feats * hbar[b:e]).sum() + (comb * cbar[b:e]).sum()
        loss.backward()
        torch.cuda.synchronize()
        return (ew.grad.cpu().numpy(), float(lam.grad), None if x0 is None else x0.grad.cpu().numpy(),
                comb.detach().cpu().numpy())

    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        g1 = once()
    kernels = sorted({ev.name for ev in p.events() if ev.device_type == torch.autograd.DeviceType.CUDA})
    g2 = once()
    same = np.array_equal(g1[0], g2[0]) and g1[1] == g2[1] and (g1[2] is None or np.array_equal(g1[2], g2[2]))
    return {"b": b, "e": e, "ew": g1[0], "lam": g1[1], "x": g1[2], "comb": g1[3], "repeat_bits": same,
            "kernels": kernels}


def _worker(rank, world, port, names, ret):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.cuda.set_device(0)
        dev = torch.device("cuda", 0)
        import efficient_gnn_b200 as egnn
        from efficient_gnn_b200 import sharded
        for name in names:
            case = CASES[name]
            n, f, k, scales, normalize, lam_val, stored = case
            adj = weighted_graph(n)
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(n, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            b, e = part.begin(rank), part.end(rank)
            w_loc = torch.from_numpy(adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)).to(dev)
            sw = sharded.ShardedWavelet(rpl, cil, n, device=dev, comm=StagedComm(),
                                        vals_local=w_loc if stored else None)
            xl = None
            if f > 1:
                xl = torch.from_numpy(np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)[b:e]).to(dev)
            # a no-grad call before and after the differentiable ones: same launches, same bits
            sw.launches = 0
            before = sw.features(k=k, s=scales, X0_local=xl)
            launches_before = sw.launches
            res = run_case(sw, case, adj, dev, rank)
            sw.launches = 0
            after = sw.features(k=k, s=scales, X0_local=xl)
            res["nograd_same"] = sw.launches == launches_before and after.grad_fn is None and torch.equal(before, after)
            res["weighted_plan"] = sw.plan is not None and stored
            if world == 1:            # one GPU on the equivalent sparse COO tensor, same loss
                coo = adj.tocoo()
                idx = torch.from_numpy(np.stack([coo.row, coo.col]).astype(np.int64)).to(dev)
                vals = torch.from_numpy(coo.data.astype(np.float32)).to(dev).requires_grad_(True)
                lam = torch.tensor(lam_val, dtype=torch.float64, device=dev, requires_grad=True)
                a_t = torch.sparse_coo_tensor(idx, vals, (n, n))
                x0 = None if f == 1 else torch.from_numpy(
                    np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)).to(dev)
                hbar, cbar = (torch.from_numpy(x).to(dev) for x in _loss_arrays(n, f, k, len(scales)))
                out = egnn.graph_wavelet_features(a_t, k=k, s=scales, X0=x0, lambda_max=lam, normalize=normalize,
                                                  return_parts=True)
                ((out.features * hbar).sum() + (out.combined * cbar).sum()).backward()
                res["single_ew"] = vals.grad.cpu().numpy()
                res["single_lam"] = float(lam.grad)
            ret[(rank, name)] = res
    finally:
        dist.destroy_process_group()


def _check(name, res, world, tag):
    from adjacency_reference import adjacency_vjp, forward64
    from vjp_reference import wavelet_vjp
    n, f, k, scales, normalize, lam_val, stored = CASES[name]
    adj = weighted_graph(n)
    hbar, cbar = _loss_arrays(n, f, k, len(scales))
    x_full = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32) if f > 1 else None
    dA, dlam, size = adjacency_vjp(adj, k, scales, x_full, lam_val, normalize, hbar, cbar, with_scale=True)
    coo = adj.tocoo()
    ref = dA[coo.row, coo.col]
    tol = 1e-5 if k <= 16 else 1e-4
    got = np.concatenate([r["ew"] for r in res]).astype(np.float64)
    nw, el = rel_max_err(got, ref), elementwise_ratio(got, ref, tol)
    el3 = elementwise_ratio(got, ref, tol, floor=1e-3)
    lam_err = abs(res[0]["lam"] - dlam) / max(size, 1e-30)
    msg = (f"{tag} world {world} {name}: edge_weight.grad norm-wise {nw:.2e}, element-wise {el:.2f} (1e-3 floor "
           f"{el3:.2f}), lambda_max.grad size-relative {lam_err:.2e} (plain {abs(res[0]['lam'] - dlam) / max(abs(dlam), 1e-30):.2e})")
    assert all(r["repeat_bits"] for r in res), f"{name}: two backward passes differ"
    assert all(r["lam"] == res[0]["lam"] for r in res), f"{name}: lambda_max.grad differs between ranks"
    assert all(r.get("nograd_same", True) for r in res), f"{name}: the no-grad call changed"
    assert not any(r.get("weighted_plan") for r in res), f"{name}: a weighted shard kept the SELL plan"
    assert nw <= tol and el <= 1.0, msg
    if k == 0:
        assert res[0]["lam"] == 0.0
    else:
        assert lam_err <= tol, msg
    # the weighted forward against the float64 restatement
    p = forward64(adj, k, scales, x_full, lam_val)
    comb = np.zeros((n, len(scales), f))
    for r in res:
        comb[r["b"]:r["e"]] = r["comb"]
    want = np.stack(p["S"], axis=1)
    assert rel_max_err(comb, want) <= tol, (msg, rel_max_err(comb, want))
    msg += f", forward {rel_max_err(comb, want):.2e}"
    if f > 1:                         # the signal's gradient on the weighted shard
        xw, _ = wavelet_vjp(adj, k, scales, x_full, lam_val, normalize, hbar, cbar)
        gx = np.zeros((n, f))
        for r in res:
            gx[r["b"]:r["e"]] = r["x"]
        nwx, elx = rel_max_err(gx, xw), elementwise_ratio(gx, xw, tol)
        msg += f", X0.grad norm-wise {nwx:.2e}, element-wise {elx:.2f}"
        assert nwx <= tol and elx <= 1.0, msg
    if "single_ew" in res[0]:
        d1 = rel_max_err(got, res[0]["single_ew"].astype(np.float64))
        msg += f", vs graph_wavelet_features {d1:.2e}"
        assert d1 <= tol, msg
        if k >= 1:
            assert abs(res[0]["lam"] - res[0]["single_lam"]) / max(size, 1e-30) <= tol, msg
    return msg


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_sharded_structure_grad_matches_vjp(world):
    names = sorted(CASES)
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), names, ret), nprocs=world, join=True)
    for name in names:
        n, f, k, scales, normalize, lam_val, stored = CASES[name]
        res = [ret[(r, name)] for r in range(world)]
        print(_check(name, res, world, "staged"))
        kernels = " ".join(n_ for r in res for n_ in r["kernels"])
        assert "shard_grad_entries_kernel" in kernels and "adj_grad_finish_kernel" in kernels, (name, kernels)
        if k >= 1:
            assert "shard_grad_dot_kernel" in kernels and "shard_grad_stacks_kernel" in kernels, (name, kernels)
            assert "cheb_order_kernel" in kernels and ", true, false, true>" in kernels, (name, kernels)  # weighted ADJ


# ---- two GPUs: the fused wide exchange and NCCL --------------------------------------------------------
TWO = [("f8_k3_binary_shard", "peer"), ("f130_k3_s3", "peer"), ("f37_k17", "peer"), ("f3_k3_s3", "nccl"),
       ("f130_k3_s3", "nccl"), ("f1_default_k3_s3", "nccl")]


def _worker2(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from efficient_gnn_b200 import sharded
        for name, exchange in TWO:
            os.environ["EGNN_EXCHANGE"] = exchange
            n, f, k, scales, normalize, lam_val, stored = CASES[name]
            adj = weighted_graph(n)
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(n, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            b, e = part.begin(rank), part.end(rank)
            w_loc = torch.from_numpy(adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)).to(dev)
            sw = sharded.ShardedWavelet(rpl, cil, n, device=dev, vals_local=w_loc if stored else None)
            assert sw.fused_wide == (exchange == "peer")
            res = run_case(sw, CASES[name], adj, dev, rank)
            sw.check_exchange()
            sw.close()
            ret[(rank, name, exchange)] = res
    finally:
        dist.destroy_process_group()


def test_two_rank_structure_grad():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (one process per GPU)")
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker2, args=(world, _free_port(), ret), nprocs=world, join=True)
    for name, exchange in TWO:
        res = [ret[(r, name, exchange)] for r in range(world)]
        print(_check(name, res, world, exchange))
        kernels = " ".join(n_ for r in res for n_ in r["kernels"])
        if exchange == "peer":
            assert "adjoint_prologue_push_kernel" in kernels, (name, kernels)
            assert re.search(r"cheb_wide_kernel<\d, true, (true|false), true, false, true>", kernels), (name, kernels)
