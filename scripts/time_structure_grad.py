"""Cost of the adjacency gradient of the wavelet pass (DESIGN.md section 11).

For each workload: the forward alone (no grad), forward + backward with a signal gradient,
forward + backward with an adjacency gradient (all three from the same adjacency input, graph
construction included), and on a graph built once: the forward kernels with every order kept, the
adjoint pass that keeps every Clenshaw vector, and each new kernel on its own (the degree terms,
the pattern or dense gradient, the lambda_max reduction).  CUDA events, warm-up first, medians of
the timed repeats; the card and its power limit are read in the same run.

    python scripts/time_structure_grad.py [--repeats 10] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import efficient_gnn_b200 as egnn  # noqa: E402
from efficient_gnn_b200 import synth  # noqa: E402
from efficient_gnn_b200.wats import (_PassSpec, _adjacency_grad, _lambda_max_grad, _run_adjoint,  # noqa: E402
                                     _run_cheb)

K = 3
# shape, F (None: default signal), adjacency layout
WORKLOADS = [("arxiv", 128, "coo"), ("reddit", None, "coo"), ("n20k", None, "dense"), ("n20k", 16, "dense")]


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


def adjacency(shape, layout):
    """(adjacency input builder, n): a COO tensor over the shape's CSR or a dense [N, N] matrix of a
    20,000-node hub-skewed directed weighted graph."""
    if shape == "n20k":
        n = 20_000
        e = synth.synth_edges(n, 10 * n, seed=6, device="cuda")
        e = e[:, torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(8), device="cuda") < 0.6]
        dense = torch.zeros((n, n), device="cuda")
        dense[e[0], e[1]] = 0.5 + torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(9),
                                             device="cuda")
        return (lambda grad: dense.clone().requires_grad_() if grad else dense), n
    rp, ci, n = synth.synth_csr(shape, self_loops=True, device="cuda")
    rows = torch.repeat_interleave(torch.arange(n, device="cuda"), (rp[1:] - rp[:-1]).long())
    idx = torch.stack([rows, ci.long()])
    w = torch.ones(ci.numel(), device="cuda")
    return (lambda grad: torch.sparse_coo_tensor(idx, w.clone().requires_grad_() if grad else w, (n, n))), n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print(f"card: {name}, power limit {limit}")
    rows = []
    for shape, f, layout in WORKLOADS:
        make, n = adjacency(shape, layout)
        fw = 1 if f is None else f
        gen = torch.Generator(device="cuda").manual_seed(1)
        x = None if f is None else torch.randn(n, f, device="cuda", generator=gen)
        up = torch.randn(n, fw, device="cuda", generator=gen)
        kw = dict(k=K, s=0.8, normalize=False)

        def fwd():
            with torch.no_grad():
                egnn.graph_wavelet_features(make(False), X0=x, **kw)

        def fwd_bwd_x():
            xg = (torch.zeros(n, 1, device="cuda") if x is None else x).clone().requires_grad_()
            (up * egnn.graph_wavelet_features(make(False), X0=xg, **kw)).sum().backward()

        def fwd_bwd_adj():
            (up * egnn.graph_wavelet_features(make(True), X0=x, **kw)).sum().backward()

        row = dict(shape=shape, n=n, f=fw, k=K, layout=layout, default_signal=f is None)
        row["forward_ms"] = timed(fwd, args.repeats)
        row["forward_backward_x0_ms"] = timed(fwd_bwd_x, args.repeats)
        row["forward_backward_adjacency_ms"] = timed(fwd_bwd_adj, args.repeats)
        # the pieces on a graph built once
        a = make(False)
        g = egnn.as_graph(a)
        x0 = g.x0 if x is None else x
        coeffs = egnn.heat_coefficients(K, 0.8)
        op_scale = 1.0
        state = {}

        def forward_kernels():
            state["t"] = _run_cheb(g, x0, K, coeffs, op_scale, -1.0, False, True)[1]

        cbar = up.reshape(n, 1, fw).contiguous()

        def adjoint_all():
            state["b"] = _run_adjoint(g.adjoint(), (g.dinv, g.iso), K, coeffs, op_scale, -1.0, cbar, keep_all=True)[1]

        row["forward_kernels_ms"] = timed(forward_kernels, args.repeats)
        row["adjoint_all_ms"] = timed(adjoint_all, args.repeats)
        pattern = None
        if layout == "coo":
            c = a.coalesce().indices().to(torch.int32)
            pattern = (c[0].contiguous(), c[1].contiguous())
        spec = _PassSpec(g, g.adjoint, K, coeffs, op_scale, -1.0, True, default_signal=f is None, lambda_max=2.0,
                         pattern=pattern)
        lib = egnn._cabi.load()
        gw = torch.empty(n, device="cuda")
        grho = torch.empty(n, device="cuda")
        ws_bytes = int(lib.egnn_adj_grad_degree_ws_bytes(n))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        P = egnn._cabi.ptr
        lam, t = state["b"][1:], state["t"][:K]

        def degree():
            egnn._cabi.check(lib.egnn_adj_grad_degree(
                P(g.rowptr), P(g.colidx), P(g.vals), P(g.adjoint().rowptr), P(g.adjoint().colidx), P(g.adjoint().vals),
                P(g.dinv), P(g.iso), n, g.nnz, fw, K, op_scale, P(lam), P(t),
                P(state["b"][0]) if f is None else None, P(g.rowsum) if f is None else None, P(gw), P(grho), P(ws),
                ws_bytes, egnn._cabi.current_stream()), "egnn_adj_grad_degree")

        row["degree_ms"] = timed(degree, args.repeats)
        if layout == "coo":
            out = torch.empty(pattern[0].numel(), device="cuda")

            def pairs():
                egnn._cabi.check(lib.egnn_adj_grad_pairs(P(pattern[0]), P(pattern[1]), out.numel(), P(g.dinv), P(lam),
                                                         P(t), P(gw), P(grho), n, fw, K, op_scale, P(out),
                                                         egnn._cabi.current_stream()), "egnn_adj_grad_pairs")
            row["pairs_ms"] = timed(pairs, args.repeats)
            row["pairs"] = out.numel()
        else:
            out = torch.empty((n, n), device="cuda")

            def dense():
                egnn._cabi.check(lib.egnn_adj_grad_dense(P(g.dinv), P(lam), P(t), P(gw), P(grho), n, fw, K, op_scale,
                                                         P(out), n, egnn._cabi.current_stream()), "egnn_adj_grad_dense")
            row["dense_ms"] = timed(dense, args.repeats)
            row["dense_write_TBps"] = 4.0 * n * n / (row["dense_ms"] * 1e-3) / 1e12
        row["lambda_max_ms"] = timed(lambda: _lambda_max_grad(state["b"], state["t"], 2.0), args.repeats)
        row["whole_adjacency_backward_ms"] = timed(lambda: _adjacency_grad(spec, state["b"], state["t"]), args.repeats)
        row["degree_plus_pattern_over_forward_plus_adjoint"] = (
            (row["degree_ms"] + row.get("pairs_ms", 0.0)) / (row["forward_kernels_ms"] + row["adjoint_all_ms"]))
        rows.append(row)
        print(json.dumps(row))
        del make, a, g, out, state, spec
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_structure_grad.json"), "w") as fh:
            json.dump(dict(card=name, power_limit=limit, rows=rows), fh, indent=1)


if __name__ == "__main__":
    main()
