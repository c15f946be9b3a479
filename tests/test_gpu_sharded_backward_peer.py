"""Backward of the row-sharded pass with one process per GPU (2 ranks over NCCL; skipped with fewer
GPUs): the fused peer exchange of the wide path (egnn_wide_adjoint_sharded, the adjoint
instantiations of cheb_wide_kernel with PEER) and, with ``EGNN_EXCHANGE=nccl``, the generic path
over NCCL, against the float64 ``wavelet_vjp`` and the single-GPU gradient of the same graph."""
import os
import socket

import numpy as np
import pytest
import torch

from helpers import elementwise_ratio, rel_max_err
from test_gpu_sharded_backward import flips64, graph

pytestmark = pytest.mark.gpu

N = 6001
# f, directed, flips, k, exchange
CASES = [(1, False, False, 20, "peer"), (8, False, False, 3, "peer"), (64, False, True, 20, "peer"),
         (130, True, True, 3, "peer"), (64, True, False, 20, "peer"), (130, False, False, 3, "peer"),
         (8, True, True, 3, "nccl"), (64, False, False, 20, "nccl"), (1, True, True, 20, "nccl"),
         (130, True, False, 3, "nccl")]
SCALES = [0.8, 1.6]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _loss_arrays(f, k):
    rng = np.random.default_rng(11)
    return (rng.standard_normal((N, len(SCALES) * f)).astype(np.float32),
            rng.standard_normal((N, len(SCALES), f)).astype(np.float32))


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import efficient_gnn_b200 as egnn
        from efficient_gnn_b200 import sharded
        from torch.profiler import ProfilerActivity, profile
        for i, (f, directed, flips, k, exchange) in enumerate(CASES):
            os.environ["EGNN_EXCHANGE"] = exchange
            adj = graph(N, directed)
            deltas = flips64(adj)[0] if flips else None
            rp = torch.from_numpy(adj.indptr.astype(np.int32)).to(dev)
            ci = torch.from_numpy(adj.indices.astype(np.int32)).to(dev)
            part = sharded.RowPartition(N, world)
            rpl, cil = part.slice_csr(rp, ci, rank)
            sw = sharded.ShardedWavelet(rpl, cil, N, device=dev)
            assert sw.fused_wide == (exchange == "peer")
            b, e = sw.row_begin, sw.row_end
            x_full = np.random.default_rng(f).standard_normal((N, f)).astype(np.float32)
            hbar, cbar = (torch.from_numpy(a).to(dev) for a in _loss_arrays(f, k))
            s_t = torch.tensor(SCALES, dtype=torch.float64, requires_grad=True)
            x0 = torch.from_numpy(x_full[b:e].copy()).to(dev).requires_grad_(True)
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                feats, orders, comb = sw.features(k=k, s=s_t, X0_local=x0, return_parts=True, deltas=deltas)
                loss = (feats * hbar[b:e]).sum() + (comb * cbar[b:e]).sum()
                loss.backward()
                torch.cuda.synchronize()
            kernels = sorted({ev.name for ev in p.events() if ev.device_type == torch.autograd.DeviceType.CUDA})
            sw.check_exchange()                          # raises if a flag wait timed out
            # the single-GPU gradient of the same graph on this rank's GPU
            g = egnn.CsrGraph(rp, ci, None, N)
            s1 = torch.tensor(SCALES, dtype=torch.float64, requires_grad=True)
            x1 = torch.from_numpy(x_full).to(dev).requires_grad_(True)
            r1 = egnn.graph_wavelet_features(g, k=k, s=s1, X0=x1, return_parts=True, deltas=deltas)
            ((r1.features * hbar).sum() + (r1.combined * cbar).sum()).backward()
            np.savez(os.path.join(out_dir, f"case{i}_rank{rank}.npz"), b=b, e=e, x=x0.grad.cpu().numpy(),
                     s=s_t.grad.numpy(), single_x=x1.grad[b:e].cpu().numpy(), single_s=s1.grad.numpy(),
                     kernels=np.array(kernels, dtype=object), transposed=sw._adjoint_shard is not False)
            sw.close()
    finally:
        dist.destroy_process_group()


def test_two_rank_backward_matches_vjp(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (one process per GPU)")
    import torch.multiprocessing as mp
    from vjp_reference import wavelet_vjp
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for i, (f, directed, flips, k, exchange) in enumerate(CASES):
        adj = graph(N, directed)
        ref_adj = flips64(adj)[1] if flips else adj
        hbar, cbar = _loss_arrays(f, k)
        x_full = np.random.default_rng(f).standard_normal((N, f)).astype(np.float32)
        xw, sbar = wavelet_vjp(ref_adj, k, SCALES, x_full, 2.0, True, hbar, cbar)
        tol = 1e-5 if k <= 16 else 1e-4
        got = np.zeros((N, f))
        zs = [np.load(tmp_path / f"case{i}_rank{r}.npz", allow_pickle=True) for r in range(world)]
        for z in zs:
            got[int(z["b"]):int(z["e"])] = z["x"]
        assert np.array_equal(zs[0]["s"], zs[1]["s"])
        nw, el = rel_max_err(got, xw), elementwise_ratio(got, xw, tol)
        el3 = elementwise_ratio(got, xw, tol, floor=1e-3)
        d1 = max(float(np.abs(z["x"] - z["single_x"]).max()) for z in zs)
        msg = (f"{exchange} f={f} directed={directed} flips={flips} K={k}: X0.grad norm-wise {nw:.2e}, element-wise "
               f"{el:.2f} (1e-3 floor {el3:.2f}), s.grad {rel_max_err(zs[0]['s'], sbar):.2e}, "
               f"max |diff| to single GPU {d1:.2e}")
        print(msg)
        assert nw <= tol and el <= 1.0, msg
        assert rel_max_err(zs[0]["s"], sbar) <= tol, msg
        kernels = " ".join(str(n) for z in zs for n in z["kernels"])
        assert bool(zs[0]["transposed"]) == directed
        if exchange == "peer" and f >= 8:
            assert "adjoint_prologue_push_kernel" in kernels, msg
            assert ", true, false, true>" in kernels.replace("(egnn::WideParams)", ""), msg   # PEER, static rows, ADJ
            if not directed:          # same sums in the same order as one GPU (DESIGN.md section 12)
                assert all(np.array_equal(z["x"], z["single_x"]) for z in zs), msg
        else:
            assert "cheb_order_kernel" in kernels and "adjoint_prologue_kernel" in kernels, msg
