"""Cost of the edge-weight gradient of the row-sharded wavelet pass (DESIGN.md section 13): forward
without grad, forward + backward w.r.t. the signal, forward + backward w.r.t. the edge weights, and,
from one backward's saved vectors, the gradient terms alone (stacks, degree and entry kernels) and
the exchange of the pre-scaled stacks, per rank count.

Launch one process per GPU:

    python -m torch.distributed.run --nproc_per_node N scripts/time_sharded_structure_grad.py [--out DIR]

Workloads: the arxiv shape made directed (one direction of every other edge pair dropped) at F = 128
with a custom signal, and the Reddit shape at F = 1 with the default signal; both with weights drawn
uniformly from [0.5, 1.5].  K = 3, one scale.  CUDA events, warm-up first, medians of the timed
repeats, the maximum over the ranks.  Prints the card and its power limit beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from efficient_gnn_b200 import sharded, synth  # noqa: E402

K, SCALES = 3, [0.8]
# workload, F (1: the default signal log1p(weighted degree)), directed
WORKLOADS = [("arxiv", 128, True), ("reddit", 1, False)]


def card(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def directed(rp, ci, n):
    """Keep entry (i, j) unless i > j and (i + j) is even: a directed graph with long rows kept."""
    rows = torch.repeat_interleave(torch.arange(n, device=rp.device), (rp[1:] - rp[:-1]).long())
    keep = ~((rows > ci.long()) & ((rows + ci.long()) % 2 == 0))
    rp2 = torch.zeros(n + 1, dtype=torch.int64, device=rp.device)
    rp2[1:] = torch.cumsum(torch.bincount(rows[keep], minlength=n), 0)
    return rp2.to(torch.int32), ci[keep].contiguous()


def timed(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    dist.barrier()
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def worst(ms, dev):
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    name, limit = card(dev)
    rows_out = []
    for workload, f, is_directed in WORKLOADS:
        rp, ci, n = synth.synth_csr(workload, self_loops=True, device=dev)
        if is_directed:
            rp, ci = directed(rp, ci, n)
        gen = torch.Generator(device=dev).manual_seed(5)
        w_full = torch.rand(ci.numel(), device=dev, generator=gen) + 0.5
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        b, e = part.begin(rank), part.end(rank)
        wl = w_full[int(rp[b]):int(rp[e])].contiguous()
        nnz = int(ci.numel())
        del rp, ci, w_full
        sw = sharded.ShardedWavelet(rpl, cil, n, device=dev, vals_local=wl)
        x0 = None
        if f > 1:
            x0 = torch.randn(n, f, device=dev, generator=gen)[b:e].contiguous()
        hbar = torch.randn(n, len(SCALES) * f, device=dev, generator=gen)[b:e].contiguous()
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        sw._adjoint_csr()
        sw._adjoint_vals(sw._base)
        torch.cuda.synchronize()
        build_ms = worst((time.perf_counter() - t0) * 1e3, dev)
        # the signal whose gradient is timed: a custom width-F signal.  At F = 1 the default signal has no
        # X0 input, so the X0 column uses a random width-1 signal, and its no-grad forward is timed beside it
        xs = x0 if x0 is not None else torch.randn(e - b, 1, device=dev, generator=gen)

        def fwd():
            sw.features(k=K, s=SCALES, X0_local=x0)

        xg = xs.clone().requires_grad_(True)

        def fwd_bwd_x():
            (sw.features(k=K, s=SCALES, X0_local=xg) * hbar).sum().backward()

        ew = wl.clone().requires_grad_(True)

        def fwd_bwd_w():
            (sw.features(k=K, s=SCALES, X0_local=x0, edge_weight=ew) * hbar).sum().backward()

        fwd_ms = worst(timed(fwd, args.repeats), dev)
        fwd_x_ms = fwd_ms if x0 is not None else worst(timed(lambda: sw.features(k=K, s=SCALES, X0_local=xs),
                                                             args.repeats), dev)
        bx_ms = worst(timed(fwd_bwd_x, args.repeats), dev)
        bw_ms = worst(timed(fwd_bwd_w, args.repeats), dev)

        # the gradient terms alone, from one backward's Clenshaw vectors and orders
        saved = {}
        orig = sw._structure_grad

        def grab(spec, b_all, t_all, f_, *wants, **kw):
            saved.update(spec=spec, b_all=b_all, t_all=t_all)
            return orig(spec, b_all, t_all, f_, *wants, **kw)

        sw._structure_grad = grab
        fwd_bwd_w()
        sw._structure_grad = orig
        spec, b_all, t_all = saved["spec"], saved["b_all"], saved["t_all"]
        eng, g = sw.engine, spec.graph
        rp_ = sw.part.rows_per
        a = 2.0 / spec.lambda_max
        pl, pt = eng.adj_grad_stacks(b_all, t_all, g.dinv, n, b, e, rp_, f, K)
        plf = torch.empty((world * rp_, K * f), device=dev)
        ptf = torch.empty_like(plf)
        sw._allgather(plf, pl)
        sw._allgather(ptf, pt)
        rpt, cit = sw._adjoint_csr()[:2]
        vt = sw._adjoint_vals(g)[0]
        orders = (sw._forward_row_order(), sw._adjoint_row_order())
        default = f == 1 and x0 is None
        xbar = b_all[0, :sw.rows, 0].contiguous() if default else None
        gw_full = torch.zeros(world * rp_, device=dev)

        def terms():
            eng.adj_grad_stacks(b_all, t_all, g.dinv, n, b, e, rp_, f, K)
            ge, gw, grho = eng.adj_grad_degree((sw.rowptr, sw.colidx, g.vals), (rpt, cit, vt), orders, g.dinv, g.iso,
                                               n, b, e, f, K, a, plf, ptf, xbar, g.rowsum_local if default else None)
            eng.adj_grad_entries(sw.rowptr, sw.colidx, n, b, e, K, ge, gw_full, grho, a)

        def exchange():
            sw._allgather(plf, pl)
            sw._allgather(ptf, pt)

        terms_ms = worst(timed(terms, args.repeats), dev)
        exch_ms = worst(timed(exchange, args.repeats), dev)
        if sw.peer is not None or sw._wide_peers:
            sw.check_exchange()
        path = "wide-fused" if (sw.fused_wide and f >= 8) else "generic-allgather"
        row = {"workload": workload, "f": f, "signal": "default" if x0 is None else "custom", "directed": is_directed,
               "weighted": True, "n_gpus": world, "nnz": nnz, "k": K, "path": path,
               "transposed_copy": sw._adjoint_shard is not False,
               "fwd_nograd_ms": fwd_ms, "x0_grad_signal": "custom" if x0 is not None else "custom width 1",
               "fwd_nograd_x0_signal_ms": fwd_x_ms, "fwd_bwd_x0_ms": bx_ms, "fwd_bwd_edge_weight_ms": bw_ms,
               "grad_terms_ms": terms_ms, "stack_exchange_ms": exch_ms, "transpose_build_ms": build_ms,
               "card": name, "power_limit": limit}
        rows_out.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
        sw.close()
        del sw, x0, xg, ew, hbar, rpl, cil, b_all, t_all, pl, pt, plf, ptf, saved, spec
        torch.cuda.empty_cache()
    if rank == 0 and args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"sharded_structure_grad_n{world}.json"), "w") as fh:
            json.dump(rows_out, fh, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
