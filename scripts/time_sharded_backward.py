"""Forward (no grad) against forward + backward of the row-sharded wavelet pass, one adjoint
application against one forward order, and the one-time transposed-shard build, per rank count.

Launch one process per GPU:

    python -m torch.distributed.run --nproc_per_node N scripts/time_sharded_backward.py [--out DIR]

CUDA events, warm-up first, medians of the timed repeats, the maximum over the ranks.  Prints the
card and its power limit beside the numbers; the table in DESIGN.md section 12 comes from this script.
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
# workload, F, directed (arxiv: the synthetic graph with one direction of every other edge dropped)
WORKLOADS = [("reddit", 64, False), ("arxiv", 128, True), ("reddit", 1, False)]


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
        part = sharded.RowPartition(n, world)
        rpl, cil = part.slice_csr(rp, ci, rank)
        del rp, ci
        sw = sharded.ShardedWavelet(rpl, cil, n, device=dev)
        gen = torch.Generator(device=dev).manual_seed(7)
        x_full = torch.randn(n, f, device=dev, generator=gen)
        x0 = x_full[sw.row_begin:sw.row_end].contiguous()
        hbar = torch.randn(n, len(SCALES) * f, device=dev, generator=gen)[sw.row_begin:sw.row_end]
        del x_full
        # one-time transposed-shard build (collective), then the steady state
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        sw._adjoint_csr()
        torch.cuda.synchronize()
        build_ms = worst((time.perf_counter() - t0) * 1e3, dev)

        def fwd():
            sw.features(k=K, s=SCALES, X0_local=x0)

        xg = x0.clone().requires_grad_(True)

        def fwd_bwd():
            (sw.features(k=K, s=SCALES, X0_local=xg) * hbar).sum().backward()

        state = {}

        def bwd_only():
            state["loss"].backward()

        fwd_ms = worst(timed(fwd, args.repeats), dev)
        both_ms = worst(timed(fwd_bwd, args.repeats), dev)
        # backward alone: forward queued and finished outside the window
        times = []
        for i in range(args.repeats + 3):
            state["loss"] = (sw.features(k=K, s=SCALES, X0_local=xg) * hbar).sum()
            torch.cuda.synchronize()
            dist.barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            bwd_only()
            b.record()
            b.synchronize()
            if i >= 3:
                times.append(a.elapsed_time(b))
        bwd_ms = worst(sorted(times)[len(times) // 2], dev)
        if sw.peer is not None or sw._wide_peers:
            sw.check_exchange()
        path = ("wide-fused" if (sw.fused_wide and f >= 8) else "generic-allgather")
        row = {"workload": workload, "f": f, "directed": is_directed, "n_gpus": world, "k": K,
               "transposed_copy": sw._adjoint_shard is not False, "backward_path": path,
               "forward_path": "sell-step" if (sw.plan is not None and f == 1) else path,
               "fwd_nograd_ms": fwd_ms, "fwd_bwd_ms": both_ms, "bwd_ms": bwd_ms,
               "bwd_over_fwd": bwd_ms / fwd_ms, "per_order_ms": fwd_ms / K, "per_app_ms": bwd_ms / K,
               "transpose_build_ms": build_ms, "card": name, "power_limit": limit}
        rows_out.append(row)
        if rank == 0:
            print(json.dumps(row), flush=True)
        sw.close()
        del sw, x0, xg, hbar, rpl, cil
        torch.cuda.empty_cache()
    if rank == 0 and args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, f"sharded_backward_n{world}.json"), "w") as fh:
            json.dump(rows_out, fh, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
