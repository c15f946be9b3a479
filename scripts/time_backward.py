"""Forward (no grad) against forward + backward of the wavelet pass, and one
adjoint application against one forward order, on the benchmark's graph shapes.

CUDA events, warm-up first, medians of the timed repeats.  Prints the card and
its power limit beside the numbers; the figures in DESIGN.md section 10 come
from this script.

    python scripts/time_backward.py [--repeats 10] [--out DIR]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import efficient_gnn_b200 as egnn  # noqa: E402
from efficient_gnn_b200 import synth  # noqa: E402
from efficient_gnn_b200.wats import _PassSpec, _run_adjoint  # noqa: E402

K = 3
WORKLOADS = [("reddit", 1, [0.8]), ("reddit", 64, [0.8]), ("arxiv", 128, [0.8]),
             ("arxiv", 128, [0.3, 0.8, 1.6, 2.4]), ("physics", 8415, [0.8])]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def timed(fn, repeats, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return sorted(times)[len(times) // 2]


def per_launch(run, n_launches, repeats, used=None, warmup=3):
    """Median over repeats of the mean time between the event pairs (2j, 2j+1), j < used (default
    n_launches), of a call that records 2 * n_launches events (ms per launch)."""
    used = n_launches if used is None else used
    res = []
    for it in range(warmup + repeats):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * n_launches)]
        for e in ev:
            e.record()                            # creates the CUDA event behind each handle
        torch.cuda.synchronize()
        run((ctypes.c_void_p * (2 * n_launches))(*[e.cuda_event for e in ev]))
        torch.cuda.synchronize()
        if it >= warmup:
            res.append(sum(ev[2 * j].elapsed_time(ev[2 * j + 1]) for j in range(used)) / used)
    return sorted(res)[len(res) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print(f"card: {name}, power limit {limit}")
    rows = []
    for shape, f, scales in WORKLOADS:
        rp, ci, n = synth.synth_csr(shape, self_loops=True, device="cuda")
        g = egnn.CsrGraph(rp, ci, None, n)
        gen = torch.Generator(device="cuda").manual_seed(1)
        x = torch.randn(n, f, device="cuda", generator=gen)
        up = torch.randn(n, len(scales) * f, device="cuda", generator=gen)
        xg = x.clone().requires_grad_()

        def fwd():
            with torch.no_grad():
                egnn.graph_wavelet_features(g, k=K, s=scales, X0=x)

        def fwd_bwd():
            xg.grad = None
            (up * egnn.graph_wavelet_features(g, k=K, s=scales, X0=xg)).sum().backward()

        t_fwd = timed(fwd, args.repeats)          # F = 1: the warm-up calls build the SELL plan (second call)
        t_fb = timed(fwd_bwd, args.repeats)
        # per order of the default forward path (F = 1: one SELL launch for all orders, shared evenly)
        sell = f == 1 and g.has_sell_plan()

        def fwd_orders(ev):
            with torch.no_grad():
                egnn.graph_wavelet_features(g, k=K, s=scales, X0=x, _order_events=ev)
        # with the SELL plan events 0 and 1 bracket the whole step
        t_order = per_launch(fwd_orders, K, args.repeats, used=1) / K if sell else per_launch(fwd_orders, K, args.repeats)
        spec = _PassSpec(g, g.adjoint, K, egnn.heat_coefficients(K, scales), 2.0, -1.0, False)
        cbar = torch.randn(n, len(scales), f, device="cuda", generator=gen)
        t_app = per_launch(lambda ev: _run_adjoint(spec, cbar, app_events=ev), K, args.repeats)
        row = dict(shape=shape, n=n, nnz=g.nnz, f=f, S=len(scales), k=K, forward_ms=t_fwd, forward_backward_ms=t_fb,
                   backward_over_forward=(t_fb - t_fwd) / t_fwd, forward_order_ms=t_order,
                   forward_order_kernel="sell_step (per order)" if sell else ("wide" if f >= 8 else "generic"),
                   adjoint_application_ms=t_app, application_over_order=t_app / t_order)
        rows.append(row)
        print(json.dumps(row))
        del g, spec, x, xg, up, cbar
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_backward.json"), "w") as fh:
            json.dump(dict(card=name, power_limit=limit, rows=rows), fh, indent=1)


if __name__ == "__main__":
    main()
