"""Cost of gradients through edge flips on the row-sharded wavelet pass (DESIGN.md section 15): forward +
backward with the flip values and ``lambda_max`` requiring grad, the same pass with only ``lambda_max``,
and the device time of each of the two flip kernels, per rank count.

Launch one process per GPU:

    python -m torch.distributed.run --nproc_per_node N scripts/time_sharded_flip_structure_grad.py [--out DIR]

Workloads: the Reddit shape at F = 1 (the default signal) and the arxiv shape made directed (one direction
of every other edge pair dropped) at F = 128 with a custom signal; binary shards, K = 3, one scale, 10
flips (added entries, removed stored entries, diagonal flips, zero-valued candidates) spread over the
graph.  CUDA events, warm-up first, medians of the timed repeats, the maximum over the ranks; the kernel
times come from torch.profiler in separate passes (mean device time per launch).  Prints the card and its
power limit beside the numbers.
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from efficient_gnn_b200 import sharded, synth  # noqa: E402
from time_sharded_structure_grad import card, directed, timed, worst  # noqa: E402

K, SCALES, N_FLIPS = 3, [0.8], 10
# workload, F (1: the default signal log1p(degree)), directed
WORKLOADS = [("reddit", 1, False), ("arxiv", 128, True)]
KERNELS = ("shard_grad_flip_terms_kernel", "shard_grad_flip_values_kernel")


def flips_for(rp, ci, n):
    """Ten flips with global ids, the same on every rank: removed stored entries and zero-valued candidates
    on stored entries of rows spread over the graph, added entries, and diagonal flips."""
    rows, cols, vals = [], [], []
    for t in range(N_FLIPS):
        i = (t * 7919 + 13) % n
        lo, hi = int(rp[i]), int(rp[i + 1])
        j = int(ci[lo]) if hi > lo else (i + 1) % n
        if t % 5 == 0:
            rows.append(i), cols.append(j), vals.append(-1.0 if hi > lo else 1.0)
        elif t % 5 == 1:
            rows.append(i), cols.append(j), vals.append(0.0)
        elif t % 5 == 2:
            rows.append(i), cols.append((i + n // 2) % n), vals.append(1.0)
        elif t % 5 == 3:
            rows.append(i), cols.append(i), vals.append(0.5)
        else:
            rows.append(i), cols.append((i * 31 + 7) % n), vals.append(0.0)
    return rows, cols, vals


def kernel_us(fn, repeats):
    """Mean device time per launch of each flip kernel over ``repeats`` calls of ``fn``, and launches per
    call."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        for _ in range(repeats):
            fn()
        torch.cuda.synchronize()
    out = {}
    for kn in KERNELS:
        ts = [ev.time_range.elapsed_us() for ev in p.events()
              if ev.device_type == torch.autograd.DeviceType.CUDA and kn in ev.name]
        out[kn] = {"us": sum(ts) / len(ts) if ts else None, "launches_per_call": len(ts) / repeats}
    return out


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
        deltas = flips_for(rp.cpu(), ci.cpu(), n)
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        b, e = part.begin(rank), part.end(rank)
        nnz = int(ci.numel())
        del rp, ci
        sw = sharded.ShardedWavelet(rpl, cil, n, device=dev)
        gen = torch.Generator(device=dev).manual_seed(5)
        x0 = None if f == 1 else torch.randn(n, f, device=dev, generator=gen)[b:e].contiguous()
        hbar = torch.randn(n, len(SCALES) * f, device=dev, generator=gen)[b:e].contiguous()
        d_rows, d_cols, d_vals = deltas
        v = torch.tensor(d_vals, device=dev, requires_grad=True)
        lam = torch.tensor(2.0, dtype=torch.float64, requires_grad=True)

        def fwd_bwd_v_lam():
            (sw.features(k=K, s=SCALES, X0_local=x0, lambda_max=lam, deltas=(d_rows, d_cols, v)) * hbar).sum() \
                .backward()

        def fwd_bwd_lam():
            (sw.features(k=K, s=SCALES, X0_local=x0, lambda_max=lam, deltas=deltas) * hbar).sum().backward()

        def fwd_nograd():
            sw.features(k=K, s=SCALES, X0_local=x0, deltas=deltas)

        fwd_ms = worst(timed(fwd_nograd, args.repeats), dev)
        v_lam_ms = worst(timed(fwd_bwd_v_lam, args.repeats), dev)
        lam_ms = worst(timed(fwd_bwd_lam, args.repeats), dev)
        v_lam_ms2 = worst(timed(fwd_bwd_v_lam, args.repeats), dev)      # alternated: the spread of the pair
        lam_ms2 = worst(timed(fwd_bwd_lam, args.repeats), dev)
        kern = kernel_us(fwd_bwd_v_lam, args.repeats)
        kern_lam = kernel_us(fwd_bwd_lam, 2)
        if sw.peer is not None or sw._wide_peers:
            sw.check_exchange()
        us = {kn: worst(kern[kn]["us"] or 0.0, dev) for kn in KERNELS}
        path = ("sell-fused" if sw.peer is not None and f == 1 else
                "wide-fused" if (sw.fused_wide and f >= 8) else "sell" if (sw.plan is not None and f == 1)
                else "generic")
        row = {"workload": workload, "f": f, "signal": "default" if x0 is None else "custom",
               "directed": is_directed, "n_gpus": world, "nnz": nnz, "k": K, "n_flips": N_FLIPS, "path": path,
               "fwd_nograd_flips_ms": fwd_ms,
               "fwd_bwd_v_lam_ms": [v_lam_ms, v_lam_ms2], "fwd_bwd_lam_only_ms": [lam_ms, lam_ms2],
               "flip_grad_overhead": min(v_lam_ms, v_lam_ms2) / min(lam_ms, lam_ms2) - 1.0,
               "flip_terms_kernel_us": us[KERNELS[0]], "flip_values_kernel_us": us[KERNELS[1]],
               "flip_kernel_launches_per_backward": [kern[kn]["launches_per_call"] for kn in KERNELS],
               "flip_kernel_launches_lam_only": [kern_lam[kn]["launches_per_call"] for kn in KERNELS],
               "card": name, "power_limit": limit}
        rows_out.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
        sw.close()
        del sw, x0, hbar, rpl, cil, v
        torch.cuda.empty_cache()
    if rank == 0 and args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"sharded_flip_structure_grad_n{world}.json"), "w") as fh:
            json.dump(rows_out, fh, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
