"""Gradients through edge flips on the row-sharded pass on ONE GPU (DESIGN.md section 15): the ranks of a
1/2/3/4-way partition run as processes sharing the device, with the staged gloo exchange of
tests/test_gpu_sharded_backward.py.  Graphs: the weighted directed graph of
tests/test_gpu_sharded_structure_grad.py (an in-star hub, an isolated node, self loops) and its pattern
made binary and symmetric.  Flips of every kind (added, removed, re-weighted, diagonal, isolating,
repeated, zero-valued candidates), 1, 10 and 64 of them.

Checks: the flip values against the float64 ``adjacency_vjp`` of the dense ``A + delta`` at section 10's
bars, scaled by the size of the whole gradient (as section 14); ``lambda_max`` at section 11's
size-relative bar; world 1 against one-GPU ``graph_wavelet_features(coo, deltas=(r, c, v))``; bitwise
repeatable backward passes; ``X0`` / ``s`` gradients bitwise those of the same call without ``v``
requiring grad; the two new kernels run once per backward, only with flip gradients, and a no-grad call
launches no gradient kernel.  Two GPUs: the fused narrow forward with in-kernel patches and the fused
wide adjoint."""
import os
import socket
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from test_gpu_flip_adjacency_grad import flipped, make_flips, report, report_lambda_max
from test_gpu_sharded_backward import StagedComm
from test_gpu_sharded_structure_grad import weighted_graph

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

N = 1001
FLIP_KERNELS = ("shard_grad_flip_terms_kernel", "shard_grad_flip_values_kernel")


def graph(name):
    a = weighted_graph(N)
    if name == "weighted":
        return a
    a = a.copy()
    a.data[:] = 1.0
    a.eliminate_zeros()
    s = sp.csr_matrix(((a + a.T) > 0).astype(np.float32), dtype=np.float32)
    s.sort_indices()
    return s


def flips_of(A, m):
    """:func:`make_flips` with, from 10 flips on, an unstored and a stored entry turned into zero-valued
    candidates (the added entry at 6, the re-weighted one at 8)."""
    rows, cols, vals = make_flips(A, m, seed=m)
    if m >= 10:
        vals[6] = vals[8] = 0.0
    return rows, cols, vals


# name: graph, F (1: default signal), K, S, flips, normalize, lambda_max.  The default signal is not
# normalised here: one column normalised on its own is about sign(S), whose gradient is at rounding level
# (section 14), so it would test nothing.
CASES = {
    "weighted_f1_k3_s3_10": ("weighted", 1, 3, 3, 10, False, 2.0),
    "weighted_f1_k0_10": ("weighted", 1, 0, 1, 10, False, 2.0),
    "binary_f1_k1_1": ("binary", 1, 1, 1, 1, False, 1.7),
    "weighted_f3_k3_64": ("weighted", 3, 3, 1, 64, True, 2.0),
    "binary_f8_k3_s3_10": ("binary", 8, 3, 3, 10, False, 2.2),
    "weighted_f37_k17_10": ("weighted", 37, 17, 1, 10, True, 2.0),
    "binary_f1_k17_64": ("binary", 1, 17, 1, 64, False, 2.0),
}


def _scales(n_s):
    return [0.8] if n_s == 1 else [0.8, 0.4, 1.3]


def _inputs(case):
    gname, f, k, n_s, m, normalize, lam_val = case
    A = graph(gname).toarray().astype(np.float64)
    rng = np.random.default_rng(f + k + m)
    x = None if f == 1 else rng.standard_normal((N, f)).astype(np.float32)
    hb = rng.standard_normal((N, n_s * f)).astype(np.float32)
    return A, flips_of(A, m), x, hb


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _names(prof):
    return [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]


def run_case(sw, case, dev):
    from torch.profiler import ProfilerActivity, profile
    gname, f, k, n_s, m, normalize, lam_val = case
    A, (rows, cols, vals), x, hb = _inputs(case)
    b, e = sw.row_begin, sw.row_end
    hbar = torch.from_numpy(hb[b:e]).to(dev)

    def once(with_v):
        v = torch.tensor(vals, dtype=torch.float32, device=dev, requires_grad=with_v)
        lam = torch.tensor(lam_val, dtype=torch.float64, requires_grad=True)
        s = torch.tensor(_scales(n_s), dtype=torch.float64, requires_grad=True)
        x0 = None if x is None else torch.from_numpy(x[b:e].copy()).to(dev).requires_grad_(True)
        feats = sw.features(k=k, s=s, X0_local=x0, lambda_max=lam, normalize=normalize,
                            deltas=(rows, cols, v if with_v else vals))
        (feats * hbar).sum().backward()
        torch.cuda.synchronize()
        return (None if v.grad is None else v.grad.cpu().numpy(), float(lam.grad), s.grad.numpy().copy(),
                None if x0 is None else x0.grad.cpu().numpy())

    with profile(activities=[ProfilerActivity.CUDA]) as p:
        g1 = once(True)
    with_names = _names(p)
    g2 = once(True)
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        g0 = once(False)
    without_names = _names(p)
    sw.launches = 0
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        with torch.no_grad():
            sw.features(k=k, s=_scales(n_s), X0_local=None if x is None else torch.from_numpy(x[b:e]).to(dev),
                        deltas=(rows, cols, vals))
        torch.cuda.synchronize()
    nograd_names = _names(p)
    return {"b": b, "e": e, "v": g1[0], "lam": g1[1],
            "repeat_bits": np.array_equal(g1[0], g2[0]) and g1[1] == g2[1] and np.array_equal(g1[2], g2[2]),
            "xs_same": np.array_equal(g1[2], g0[2]) and (g1[3] is None or np.array_equal(g1[3], g0[3])),
            "flip_launches": [sum(kn in n_ for n_ in with_names) for kn in FLIP_KERNELS],
            "flip_launches_lam_only": [sum(kn in n_ for n_ in without_names) for kn in FLIP_KERNELS],
            "nograd_grad_kernels": [n_ for n_ in nograd_names if "adj_grad" in n_ or "shard_grad" in n_]}


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
            gname, f, k, n_s, m, normalize, lam_val = case
            adj = graph(gname)
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(N, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            b, e = part.begin(rank), part.end(rank)
            w_loc = torch.from_numpy(adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)).to(dev)
            sw = sharded.ShardedWavelet(rpl, cil, N, device=dev, comm=StagedComm(),
                                        vals_local=w_loc if gname == "weighted" else None)
            res = run_case(sw, case, dev)
            if world == 1:            # one GPU on the equivalent sparse COO tensor, same loss
                A, (rows, cols, vals), x, hb = _inputs(case)
                coo = adj.tocoo()
                idx = torch.from_numpy(np.stack([coo.row, coo.col]).astype(np.int64)).to(dev)
                a_t = torch.sparse_coo_tensor(idx, torch.from_numpy(coo.data.astype(np.float32)).to(dev), (N, N))
                v = torch.tensor(vals, dtype=torch.float32, device=dev, requires_grad=True)
                lam = torch.tensor(lam_val, dtype=torch.float64, device=dev, requires_grad=True)
                out = egnn.graph_wavelet_features(a_t, k=k, s=_scales(n_s), X0=None if x is None else
                                                  torch.from_numpy(x).to(dev), lambda_max=lam, normalize=normalize,
                                                  deltas=(rows, cols, v))
                (out * torch.from_numpy(hb).to(dev)).sum().backward()
                res["single_v"], res["single_lam"] = v.grad.cpu().numpy(), float(lam.grad)
            ret[(rank, name)] = res
    finally:
        dist.destroy_process_group()


def _check(name, res, world, tag):
    from adjacency_reference import adjacency_vjp
    case = CASES[name]
    gname, f, k, n_s, m, normalize, lam_val = case
    A, flips, x, hb = _inputs(case)
    dA, dlam, size = adjacency_vjp(flipped(A, flips), k, _scales(n_s), None if x is None else x.astype(np.float64),
                                   lam_val, normalize, hb, with_scale=True)
    tol = 1e-4 if k > 16 else 1e-5
    rows, cols, _ = flips
    label = f"{tag} world {world} {name}"
    assert all(r["repeat_bits"] for r in res), f"{label}: two backward passes differ"
    assert all(np.array_equal(r["v"], res[0]["v"]) and r["lam"] == res[0]["lam"] for r in res), \
        f"{label}: v.grad / lambda_max.grad differ between ranks"
    assert all(r["xs_same"] for r in res), f"{label}: X0 / s gradients changed with v requiring grad"
    report(f"{label} flip values", res[0]["v"], dA[rows, cols], tol, whole=np.abs(dA))
    report_lambda_max(f"{label} dlambda_max", res[0]["lam"], dlam if k else 0.0, size, tol)
    for r in res:
        assert r["flip_launches"] == [1 if k >= 1 else 0, 1], (label, r["flip_launches"])
        assert r["flip_launches_lam_only"] == [0, 0], (label, r["flip_launches_lam_only"])
        assert r["nograd_grad_kernels"] == [], (label, r["nograd_grad_kernels"])
    if "single_v" in res[0]:
        report(f"{label} vs graph_wavelet_features", res[0]["v"], res[0]["single_v"].astype(np.float64), tol,
               whole=np.abs(dA))
        if k >= 1:
            assert abs(res[0]["lam"] - res[0]["single_lam"]) / max(size, 1e-30) <= tol, label


@pytest.mark.parametrize("world", [1, 2, 3, 4])
def test_sharded_flip_grad_matches_vjp(world):
    names = sorted(CASES)
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), names, ret), nprocs=world, join=True)
    for name in names:
        _check(name, [ret[(r, name)] for r in range(world)], world, "staged")


# ---- two GPUs: the fused narrow forward (in-kernel patches) and the fused wide adjoint ------------------
TWO = ["binary_f1_k1_1", "binary_f1_k17_64", "binary_f8_k3_s3_10", "weighted_f37_k17_10"]


def _worker2(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from efficient_gnn_b200 import sharded
        os.environ["EGNN_EXCHANGE"] = "peer"
        for name in TWO:
            gname, f, k, n_s, m, normalize, lam_val = CASES[name]
            adj = graph(gname)
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(N, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            b, e = part.begin(rank), part.end(rank)
            w_loc = torch.from_numpy(adj.data[adj.indptr[b]:adj.indptr[e]].astype(np.float32)).to(dev)
            sw = sharded.ShardedWavelet(rpl, cil, N, device=dev, vals_local=w_loc if gname == "weighted" else None)
            res = run_case(sw, CASES[name], dev)
            res["in_kernel_patch"] = f == 1 and sw.plan is not None and sw.peer is not None
            res["fused_wide"] = f >= 8 and sw.fused_wide
            sw.check_exchange()
            sw.close()
            ret[(rank, name)] = res
    finally:
        dist.destroy_process_group()


def test_two_rank_flip_grad():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (one process per GPU)")
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker2, args=(world, _free_port(), ret), nprocs=world, join=True)
    for name in TWO:
        res = [ret[(r, name)] for r in range(world)]
        _check(name, res, world, "peer")
        print(f"\n[{name}] in-kernel patches {res[0]['in_kernel_patch']}, fused wide adjoint {res[0]['fused_wide']}")
