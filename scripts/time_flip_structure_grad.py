"""Cost of adjacency gradients through edge flips (DESIGN.md section 14).

Two workloads, K = 3, three scales, F = 1 default signal, 10 flips (added and removed entries):

* ``n20k``: the attack's shape, a 20,000-node directed weighted graph held as a dense ``[N, N]``
  matrix.  ``flips``: what ``WATS(recompute_on_forward=True, adjacency_grad=True)`` runs, the dense
  leaf ``A'`` as the gradient input, the resident graph of ``A`` with the flips for the pass.
  ``rebuilt``: ``A'`` passed as a fresh adjacency (dense -> CSR, degree pass, then the pass).
* ``reddit``: the Reddit shape as a sparse COO pattern with a value leaf.  ``flips``: the resident
  graph with the flips and a flip-value leaf (gradient at the flips).  ``rebuilt``: the COO pattern of
  ``A'`` with a value leaf (gradient at every entry).

Forward + backward of each (CUDA events, warm-up first, medians of the timed repeats), and the
flip-terms kernel alone from a ``torch.profiler`` run of its own (mean device time over the repeats).
The card and its power limit are read in the same run.

    python scripts/time_flip_structure_grad.py [--repeats 10] [--out DIR]
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
from efficient_gnn_b200.graph import deltas_from_dense  # noqa: E402
from efficient_gnn_b200.wats import _graph_features  # noqa: E402

K = 3
SCALES = [0.8, 0.4, 1.3]
N_FLIPS = 10


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


def flips_on(rows_of, cols_of, is_stored, n, seed):
    """Five added and five removed entries (distinct, off the diagonal)."""
    g = torch.Generator().manual_seed(seed)
    rows, cols, vals = [], [], []
    while len(rows) < N_FLIPS:
        want_stored = len(rows) % 2 == 1
        if want_stored:
            q = int(torch.randint(0, rows_of.numel(), (1,), generator=g))
            r, c = int(rows_of[q]), int(cols_of[q])
        else:
            r, c = (int(v) for v in torch.randint(0, n, (2,), generator=g))
        if r == c or (r, c) in zip(rows, cols) or is_stored(r, c) != want_stored:
            continue
        rows.append(r)
        cols.append(c)
        vals.append(-1.0 if want_stored else 1.0)
    return rows, cols, vals


def kernel_us(fn, name, repeats):
    """Mean device time (us) of the kernels whose name contains ``name`` per call of ``fn``."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(repeats):
            fn()
        torch.cuda.synchronize()
    hits = [e for e in prof.events() if e.device_type.name == "CUDA" and name in e.name]
    return sum(e.device_time for e in hits) / repeats, len(hits) // repeats


def dense_workload(repeats):
    n = 20_000
    e = synth.synth_edges(n, 10 * n, seed=6, device="cuda")
    e = e[:, torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(8), device="cuda") < 0.6]
    base = torch.zeros((n, n), device="cuda")
    base[e[0], e[1]] = 0.5 + torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(9),
                                        device="cuda")
    ec = e.cpu()
    stored = set(zip(ec[0].tolist(), ec[1].tolist()))
    rows, cols, vals = flips_on(ec[0], ec[1], lambda r, c: (r, c) in stored, n, seed=1)
    pert = base.clone()
    for r, c, v in zip(rows, cols, vals):
        pert[r, c] += v if v > 0 else -float(pert[r, c])
    g = egnn.as_graph(base)                        # the resident graph
    up = torch.randn(n, len(SCALES), device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))

    def flip_path():                               # as WATS.features_for: find the flips, run them on g
        leaf = pert.clone().requires_grad_()
        d = deltas_from_dense(base, leaf.detach())
        (up * _graph_features(g, K, SCALES, None, 2.0, False, False, d, adj_in=leaf)).sum().backward()

    def rebuilt():
        leaf = pert.clone().requires_grad_()
        (up * egnn.graph_wavelet_features(leaf, k=K, s=SCALES, normalize=False)).sum().backward()

    row = dict(shape="n20k", n=n, nnz=g.nnz, input="dense leaf", flips=N_FLIPS)
    row["flips_fwd_bwd_ms"] = timed(flip_path, repeats)
    row["rebuilt_fwd_bwd_ms"] = timed(rebuilt, repeats)
    row["dense_to_graph_ms"] = timed(lambda: egnn.as_graph(pert), repeats)
    row["flip_terms_kernel_us"], row["flip_terms_launches"] = kernel_us(flip_path, "adj_grad_flip_terms", repeats)
    return row


def coo_workload(repeats):
    rp, ci, n = synth.synth_csr("reddit", self_loops=True, device="cuda")
    rows_of = torch.repeat_interleave(torch.arange(n, device="cuda"), (rp[1:] - rp[:-1]).long())
    key = (rows_of * n + ci.long())                 # sorted: the CSR is row-major with sorted rows
    rows_c, cols_c = rows_of.cpu(), ci.cpu()

    def is_stored(r, c):
        i = int(torch.searchsorted(key, torch.tensor([r * n + c], device="cuda")))
        return i < key.numel() and int(key[i]) == r * n + c

    rows, cols, vals = flips_on(rows_c, cols_c, is_stored, n, seed=2)
    g = egnn.CsrGraph(rp, ci, None, n)              # the resident graph
    # A' as a COO pattern: the removed entries dropped, the added ones appended
    drop = torch.tensor([r * n + c for r, c, v in zip(rows, cols, vals) if v < 0], device="cuda")
    keep = ~torch.isin(key, drop)
    add = [(r, c) for r, c, v in zip(rows, cols, vals) if v > 0]
    idx = torch.cat([torch.stack([rows_of[keep], ci.long()[keep]]), torch.tensor(add, device="cuda").T], dim=1)
    w = torch.ones(idx.shape[1], device="cuda")
    up = torch.randn(n, len(SCALES), device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))

    def flip_path():
        dv = torch.tensor(vals, device="cuda", requires_grad=True)
        (up * egnn.graph_wavelet_features(g, k=K, s=SCALES, normalize=False,
                                          deltas=(rows, cols, dv))).sum().backward()

    def rebuilt():
        a = torch.sparse_coo_tensor(idx, w.clone().requires_grad_(), (n, n))
        (up * egnn.graph_wavelet_features(a, k=K, s=SCALES, normalize=False)).sum().backward()

    row = dict(shape="reddit", n=n, nnz=g.nnz, input="COO values", flips=N_FLIPS)
    row["flips_fwd_bwd_ms"] = timed(flip_path, repeats)
    row["rebuilt_fwd_bwd_ms"] = timed(rebuilt, repeats)
    row["coo_to_graph_ms"] = timed(lambda: egnn.as_graph(torch.sparse_coo_tensor(idx, w, (n, n))), repeats)
    row["flip_terms_kernel_us"], row["flip_terms_launches"] = kernel_us(flip_path, "adj_grad_flip_terms", repeats)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    name, limit = card()
    print(f"card: {name}, power limit {limit}")
    rows = []
    for workload in (dense_workload, coo_workload):
        row = workload(args.repeats)
        row["rebuilt_over_flips"] = row["rebuilt_fwd_bwd_ms"] / row["flips_fwd_bwd_ms"]
        rows.append(row)
        print(json.dumps(row))
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_flip_structure_grad.json"), "w") as fh:
            json.dump(dict(card=name, power_limit=limit, rows=rows), fh, indent=1)


if __name__ == "__main__":
    main()
