#!/usr/bin/env python
"""Benchmark of the Chebyshev graph-wavelet feature path (BASELINE.json metric:
"Chebyshev-wavelet nnz*K*F/s & HBM GB/s at 1/2/4/8 B200 vs ref CPU").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload reddit|arxiv|physics|pubmed|cora] [--f F] [--order K] [--scales S]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic graph of the named
shape: K fused Chebyshev orders (SpMM over the implicit scaled Laplacian +
recurrence + scale accumulation + L1 normalisation).  Default workload: the
Reddit shape (232,965 nodes, 114.8 M stored entries) with the reference's
defaults K=3, S=1 (s=0.8), F=1 (X0 = log1p(degree)) - the largest named
configuration; it fits one B200 and is the only one whose index stream comes
from HBM every order.

Prints ONE JSON line (DESIGN.md section 7 explains the keys):

* ``value``: graph resident in HBM, whole step timed on the device;
* ``roofline``: the dominant kernel (the persistent step kernel of the narrow
  path = K orders in one launch) against the measured HBM copy bandwidth -
  ``achieved``/``frac`` on the bytes the kernel itself must stream (2-byte
  block-local indices + slice tables + per-order vectors), ``achieved_contract``
  on SURVEY 8d's int32-CSR model, ``b_gather`` on the north star's gathered-rows
  model, the phase split from the kernel's own timestamps, ``traffic`` from the
  ncu capture recorded in profiles/dram_traffic.json;
* ``roofline_wide``: the two wide shapes the >= 70 % target names (arxiv-shape
  F=128, Reddit-shape F=64), measured in the same run;
* ``ugca``: the per-perturbation recompute (5 symmetric flips around a target
  node on top of the resident graph), device-timed and end to end
  (host flip list in -> features on the host);
* ``e2e``: the same metric through the host-buffer entry (pinned host CSR ->
  H2D -> degree pass -> orders -> D2H of the features);
* ``cpu_baseline`` / ``--impl reference``: the REFERENCE's own
  ``graph_wavelet_features`` (calibration/WATS.py:39-74), byte-compiled into
  oracle/_ref by ``__graft_entry__.build()``, on the SAME full graph, scipy on
  one host core as the reference runs it, with the Laplacian / rescale /
  recurrence split of WATS.py:53,55,62.  Falls back to the oracle port
  (``kind: "port"``) when oracle/_ref is not staged.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "chebyshev_wavelet_nnz_k_f_per_s"
UNIT = "nnz*K*F/s"
DEFAULT_F = {"reddit": 1, "arxiv": 128, "physics": 1, "pubmed": 1, "cora": 1}
REFERENCE_MAX_TIMED_RUNS = 2     # stock-function runs of the reference arm (the full Reddit graph takes ~1 min each)
REFERENCE_FULL_GRAPH_LIMIT = 8   # K*F above which the CPU arm falls back to a scaled sample of the workload
DUMP_MAX_BYTES = 64_000_000      # --dump-outputs: bound on what one run writes


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="reddit", choices=sorted(DEFAULT_F))
    ap.add_argument("--f", type=int, default=None, help="feature columns of X0 (default: per workload)")
    ap.add_argument("--order", type=int, default=3, help="Chebyshev order K")
    ap.add_argument("--scales", type=int, default=1, help="number of wavelet scales S")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-wide", action="store_true", help="skip the roofline_wide sub-records")
    ap.add_argument("--no-ugca", action="store_true", help="skip the ugca sub-record")
    ap.add_argument("--no-graph", action="store_true", help="do not replay the step as a CUDA graph")
    ap.add_argument("--node-order", choices=["random", "degree"], default="random",
                    help="N > 1: 'degree' renumbers the synthetic graph by descending degree (skewed equal-rows shards)")
    ap.add_argument("--balance", action="store_true",
                    help="N > 1: renumber the nodes so that the equal-rows shards hold equal entries (sharded.BalancedOrder)")
    ap.add_argument("--entry", default="csr", choices=["csr", "dense"],
                    help="e2e entry: pinned host CSR (default) or the reference's own boundary, a dense [N,N] float32 "
                         "adjacency (calibration/WATS.py:99; small shapes only)")
    ap.add_argument("--replicas", action="store_true",
                    help="N>1: UGCA replica mode - every rank holds the whole graph and recomputes the features of its "
                         "own perturbation candidates (--flips, default 5); no exchange, weak scaling")
    ap.add_argument("--no-sell", action="store_true", help="F=1: use the generic CSR kernel instead of the SELL plan")
    ap.add_argument("--flips", type=int, default=0,
                    help="UGCA mode (N=1): every step recomputes the features of the graph with this many symmetric "
                         "edge flips around a random target node applied on top of the resident graph")
    ap.add_argument("--no-check", action="store_true",
                    help="N>1: skip the comparison of every rank's rows with the single-GPU path (outside the timed region)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU only: after the timed steps, write the features the last timed step returned as "
                         "DIR/features.npy (float32); above 64 MB a fixed, seeded sample of rows, with the sampled row "
                         "ids in DIR/features_rows.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
    return args


def scale_list(n_scales):
    base = [0.8, 0.4, 1.6, 3.2, 0.2, 6.4, 0.1, 12.8]
    return base[0] if n_scales == 1 else base[:n_scales]


def workload_config(workload, n, nnz, k, n_scales, f, flips=0):
    """The ``config`` object: what is computed, identical for both arms."""
    return {"workload": f"{workload}-shape", "n": int(n), "nnz": int(nnz), "k": int(k), "scales": int(n_scales),
            "f": int(f), "self_loops": True, "ugca_flips": int(flips),
            "l2_policy": ("inputs larger than L2 (index stream %.0f MB per order vs 126 MB L2), no flush" % (2 * nnz / 1e6)
                          if 2 * nnz > 126e6 else "inputs fit in L2: latency-bound configuration, no flush")}


# --------------------------------------------------------------------------- #
# bytes models                                                                  #
# --------------------------------------------------------------------------- #
def contract_bytes(n, nnz, f, k_max, n_scales):
    """Compulsory-traffic model B_k of SURVEY 8d (int32 indices, fp32 data,
    binary adjacency) for each order k = 1..K."""
    out = []
    for k in range(1, k_max + 1):
        t_terms = 1 + (1 if k >= 2 else 0) + (1 if k < k_max else 0)
        acc = 1 if k == 1 else 2
        out.append(4 * nnz + 4 * (n + 1) + 4 * n + 4 * n * f * t_terms + 4 * n_scales * n * f * acc)
    return out


def gather_bytes(n, nnz, f, k_max, n_scales):
    """SURVEY 8d's secondary, north-star-literal model B_gather: the T_{k-1} term
    is one gathered row per stored entry (4*nnz*F) instead of one read of T_{k-1}."""
    return [b - 4 * n * f + 4 * nnz * f for b in contract_bytes(n, nnz, f, k_max, n_scales)]


def sell_stream_bytes(plan, n, k_max, n_scales):
    """What the narrow-path step kernel itself must move per order (DESIGN.md 4.2):
    the 2-byte index stream of the padded entries, the slice tables (offset and
    partial-sum slot per virtual row), the partial sums (written, then read by the
    epilogue), the row pointers of the partial sums, and the per-row vectors
    (dinv, iso, T_{k-1}, T_{k-2}, T_k, operand written + staged once, S outputs)."""
    out = []
    for k in range(1, k_max + 1):
        stream = 2 * plan.n_entries + 4 * (plan.n_slices + 1) + 4 * plan.n_vrows
        partial = 2 * 4 * plan.n_rowv + 4 * (n + 1)
        t_terms = 1 + (1 if k >= 2 else 0) + (1 if k < k_max else 0)
        vectors = 4 * n + n + 4 * n * t_terms + (8 * n if k < k_max else 4 * n) + 4 * n_scales * n * (1 if k == 1 else 2)
        out.append(stream + partial + vectors)
    return out


class ClockSampler(threading.Thread):
    """Polls NVML for SM clock / throttle reasons while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def poll(self):
        nv = self.nv
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        names = {
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "hw_power_brake_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80),
        }
        for name, bit in names.items():
            if r & bit:
                self.reasons.add(name)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                self.poll()
            except Exception:
                break
            time.sleep(0.002)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def dram_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the
    committed `ncu --set full` capture of this configuration (profiles/dram_traffic.json; the
    capture's summary and command are named there) - None when this configuration has none."""
    path = os.path.join(ROOT, "profiles", "dram_traffic.json")
    if not os.path.isfile(path):
        return None, None
    try:
        rec = json.load(open(path)).get(key)
    except Exception:
        return None, None
    if rec is None:
        return None, None
    if isinstance(rec, dict):
        return rec.get("bytes_per_launch"), rec.get("source")
    return rec, "profiles/ (round 1 capture)"


# --------------------------------------------------------------------------- #
# CPU arm: the reference's own code (oracle/_ref), else the oracle port         #
# --------------------------------------------------------------------------- #
def host_graph(workload, scale=1.0):
    """The workload's synthetic graph as scipy CSR float32, generated on the host."""
    import scipy.sparse as sp
    from efficient_gnn_b200 import synth
    rp, ci, n = synth.synth_csr(workload, self_loops=True, device="cpu", scale=scale)
    return sp.csr_matrix((np.ones(ci.numel(), np.float32), ci.numpy(), rp.numpy()), shape=(n, n))


def load_reference_wats():
    """The reference's calibration/WATS.py module (unmodified), or None."""
    try:
        from oracle import ref_shim
        if ref_shim.reference_root() is None:
            return None
        return ref_shim.load_reference()[0]
    except Exception:
        return None


def cpu_path_once(wats, adj, k, scales, f, x0, split):
    """One pass of the CPU path.  With the reference module and the reference's
    own configuration (F = 1 default signal, one scale) this is literally
    ``graph_wavelet_features(adj, k, s)``; other configurations compose the
    reference's own functions the way that function does.  ``split``: run the
    three legs of WATS.py:53,55,62 separately and time each."""
    from scipy.sparse import identity
    stock = wats is not None and f == 1 and np.ndim(scales) == 0
    if stock and not split:
        t0 = time.perf_counter()
        wats.graph_wavelet_features(adj, k=k, s=scales)
        return {"total": time.perf_counter() - t0}
    if wats is None:
        from oracle import wats_oracle as orc
        t0 = time.perf_counter()
        lt = orc.rescaled_laplacian(adj)
        t1 = time.perf_counter()
        xx = orc.input_signal(adj) if x0 is None else x0
        orders = orc.chebyshev_orders(lt, k, xx)
        t2 = time.perf_counter()
        for a in orc.heat_coefficients(k, scales):
            comb = sum(a[i] * orders[i] for i in range(k + 1))
            comb / (np.abs(comb).sum(axis=1, keepdims=True) + 1e-8)
        t3 = time.perf_counter()
        return {"total": t3 - t0, "laplacian_and_rescale": t1 - t0, "recurrence": t2 - t1, "combine": t3 - t2}
    n = adj.shape[0]
    t0 = time.perf_counter()
    lap = wats.compute_normalized_laplacian(adj)                   # WATS.py:53
    t1 = time.perf_counter()
    l_rescaled = (2 / 2.0) * lap - identity(n)                     # WATS.py:55
    t2 = time.perf_counter()
    xx = np.log1p(np.array(adj.sum(axis=1)).flatten()).reshape(-1, 1) if x0 is None else x0   # WATS.py:58-59
    t_k = wats.chebyshev_polynomials(l_rescaled, k, xx)            # WATS.py:62
    t3 = time.perf_counter()
    for s in np.atleast_1d(scales):                                # WATS.py:65-72 per scale
        alpha = [np.exp(-s * i) for i in range(k + 1)]
        comb = sum(alpha[i] * t_k[i] for i in range(k + 1))
        comb / (np.linalg.norm(comb, ord=1, axis=1, keepdims=True) + 1e-8)
    t4 = time.perf_counter()
    return {"total": t4 - t0, "laplacian": t1 - t0, "rescale": t2 - t1, "recurrence": t3 - t2, "combine": t4 - t3}


def time_cpu_path(adj, k, scales, f, stock_runs, split_run=True):
    """Times the CPU arm on ``adj``.  Returns the ``cpu_baseline`` object (value =
    best stock run, or the split run's total when no stock run was asked for)."""
    wats = load_reference_wats()
    x0 = None
    if f > 1:
        x0 = np.random.default_rng(3).standard_normal((adj.shape[0], f)).astype(np.float32)
    runs = [cpu_path_once(wats, adj, k, scales, f, x0, split=False)["total"] for _ in range(stock_runs)]
    split = cpu_path_once(wats, adj, k, scales, f, x0, split=True) if split_run else None
    best = min(runs) if runs else split["total"]
    stock = wats is not None and f == 1 and np.ndim(scales) == 0
    kind = "reference" if wats is not None else "port"
    what = ("the reference's own graph_wavelet_features (calibration/WATS.py:39-74, unmodified, byte-compiled in "
            "oracle/_ref)" if stock else
            "the reference's own compute_normalized_laplacian / chebyshev_polynomials (calibration/WATS.py:24-37, "
            "oracle/_ref) composed as graph_wavelet_features does" if wats is not None else
            "oracle port of calibration/WATS.py:39-74 (oracle/_ref not staged)")
    return {"value": adj.nnz * k * f / best, "unit": UNIT, "cores": 1, "kind": kind, "host_cores": os.cpu_count(),
            "seconds": best, "runs_seconds": runs, "split_seconds": split,
            "sample": (f"full graph N={adj.shape[0]}, nnz={adj.nnz}, K={k}, S={np.size(scales)}, F={f}; {what}; scipy is "
                       f"single-threaded on this path; best of {max(1, len(runs))} run(s)"
                       + (", plus one run with the Laplacian / rescale / recurrence legs timed separately" if split else ""))}


def run_reference(args, rank, world):
    """`--impl reference`: the reference's CPU implementation of the path on the
    SAME configuration.  The full Reddit-shape graph costs about a minute per
    pass on one core, so the arm times min(--steps, 2) passes of the stock
    function plus one pass with the three legs split, whatever --steps/--warmup
    say (stated in the line: ``steps`` is what was run)."""
    if rank != 0:
        return
    from efficient_gnn_b200 import synth
    f = args.f or DEFAULT_F[args.workload]
    scales = scale_list(args.scales)
    sh = synth.SHAPES[args.workload]
    scale = 1.0
    if args.order * f > REFERENCE_FULL_GRAPH_LIMIT and sh.nnz > 5_000_000:
        scale = max(2e-3, min(1.0, 2.0e8 / (sh.nnz * args.order * f)))       # wide signals: bounded sample of the shape
    adj = host_graph(args.workload, scale)
    big = adj.nnz > 20_000_000
    stock_runs = max(1, min(args.steps, REFERENCE_MAX_TIMED_RUNS if big else 5))
    base = time_cpu_path(adj, args.order, scales, f, stock_runs, split_run=True)
    if scale != 1.0:
        base["sample"] = f"{args.workload}-shape generator at scale {scale:.4f}: " + base["sample"]
    cfg = workload_config(args.workload, adj.shape[0], adj.nnz, args.order, args.scales, f, args.flips)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": stock_runs, "steps_requested": args.steps, "warmup": 0, "warmup_requested": args.warmup,
        "ms_per_step": base["seconds"] * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# GPU arm                                                                       #
# --------------------------------------------------------------------------- #
def make_flips(n, budget, seed, graph_rowptr=None, graph_colidx=None):
    """calib_fga.py:897-904: `budget` symmetric flips incident to one target node (additions here;
    the kernels treat removals the same way: a -1 delta)."""
    gen = torch.Generator().manual_seed(seed)
    picks = torch.randint(0, n, (budget + 1,), generator=gen).tolist()
    target, others = picks[0], [j for j in picks[1:] if j != picks[0]]
    return ([target] * len(others) + others, others + [target] * len(others), [1.0] * (2 * len(others)))


def dump_features(out_dir, feats):
    """Writes the features a step returned ([N, S*F]) as ``out_dir/features.npy`` in float32, so that two builds
    can be compared output for output on the same seeded inputs.  Above DUMP_MAX_BYTES a fixed, seeded sample of
    whole rows is written instead, with the sampled row ids (ascending) in ``out_dir/features_rows.npy``."""
    os.makedirs(out_dir, exist_ok=True)
    h = feats.detach().float().cpu().numpy()
    n, width = h.shape
    if h.nbytes > DUMP_MAX_BYTES:
        budget = (DUMP_MAX_BYTES - 1024) // (4 * width + 8)        # float32 row + its float64 id, minus the headers
        rows = np.sort(np.random.default_rng(0).choice(n, budget, replace=False))
        h = h[rows]
        np.save(os.path.join(out_dir, "features_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "features.npy"), h)


def time_steps(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def wide_record(egnn, synth, workload, f, graph, dev, peak, k_max=3):
    """One wide-signal shape through cheb_wide_kernel: per-order CUDA events recorded by the library."""
    import ctypes as C
    sh = synth.SHAPES[workload]
    if graph is None:
        rp, ci, n = synth.synth_csr(workload, self_loops=True, device=dev)
        graph = egnn.CsrGraph(rp, ci, None, n)
    n, nnz = graph.n, graph.nnz
    x0 = torch.randn(n, f, device=dev, generator=torch.Generator(device=dev).manual_seed(sh.seed))
    steps = 12
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2 * k_max)] for _ in range(steps)]
    for row in ev:
        for e in row:
            e.record()
    torch.cuda.synchronize()
    arrays = [(C.c_void_p * (2 * k_max))(*[e.cuda_event for e in row]) for row in ev]
    for _ in range(3):
        egnn.graph_wavelet_features(graph, k=k_max, s=0.8, X0=x0)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        egnn.graph_wavelet_features(graph, k=k_max, s=0.8, X0=x0, _order_events=arrays[i])
    b.record()
    torch.cuda.synchronize()
    ms_step = a.elapsed_time(b) / steps
    order_ms = np.array([[row[2 * j].elapsed_time(row[2 * j + 1]) for j in range(k_max)] for row in ev]).mean(axis=0)
    b_k = contract_bytes(n, nnz, f, k_max, 1)
    g_k = gather_bytes(n, nnz, f, k_max, 1)
    avg = float(order_ms.mean())
    achieved = (sum(b_k) / k_max) / (avg * 1e-3) / 1e9
    traffic, src = dram_traffic(f"{workload}_f{f}_k{k_max}_s1")
    return {"workload": f"{workload}-shape", "n": n, "nnz": nnz, "f": f, "k": k_max, "kernel": "cheb_wide_kernel",
            "ms_per_step": ms_step, "per_order_ms": [float(v) for v in order_ms], "value": nnz * k_max * f / (ms_step * 1e-3),
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "algorithmic_bytes_per_launch": sum(b_k) / k_max,
            "b_gather_bytes_per_launch": sum(g_k) / k_max, "b_gather_achieved": (sum(g_k) / k_max) / (avg * 1e-3) / 1e9,
            "traffic": traffic, "traffic_source": src,
            "note": "contract-bytes model (every T row read once); the gathers are served by L2, see DESIGN.md 4.3"}


def run_ours(args, rank, local_rank, world):
    import efficient_gnn_b200 as egnn
    from efficient_gnn_b200 import synth
    from efficient_gnn_b200.graph import enable_phase_stamps, read_phase_stamps

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    f = args.f or DEFAULT_F[args.workload]
    k_max, n_scales = args.order, args.scales
    scales = scale_list(n_scales)
    sh = synth.SHAPES[args.workload]

    if world > 1 and args.replicas:
        return run_replicas(args, rank, local_rank, world)
    if world > 1:
        from efficient_gnn_b200 import sharded
        return sharded.bench_entry(args, rank, local_rank, world, METRIC, UNIT, contract_bytes, ClockSampler,
                                   physical_gpu_index, scale_list, workload_config, make_flips)

    # synthetic graph of the named shape, generated directly in HBM
    rp, ci, n = synth.synth_csr(args.workload, self_loops=True, device=dev)
    graph = egnn.CsrGraph(rp, ci, None, n)
    nnz = graph.nnz
    if f == 1:
        x0 = None                                  # reference default: log1p(degree), produced by the degree pass
    else:
        x0 = torch.randn(n, f, device=dev, generator=torch.Generator(device=dev).manual_seed(sh.seed))
    work = float(nnz) * k_max * f
    peak, peak_src = hbm_peak()

    use_sell = False if args.no_sell else None
    flips = make_flips(n, args.flips, 7) if args.flips > 0 else None

    def step(events=None):
        return egnn.graph_wavelet_features(graph, k=k_max, s=scales, X0=x0, deltas=flips, _order_events=events,
                                           _use_sell=use_sell)

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize()
    plan = graph.sell_plan() if (f == 1 and k_max >= 1 and not args.no_sell) else None
    narrow = plan is not None
    if narrow:
        enable_phase_stamps(plan)                  # CTA 0's globaltimer at every grid barrier (no effect on the timing)

    # per-launch CUDA events (recorded by the library on the launching stream) on every 8th step of the
    # timed region; the other steps replay the same pass as one CUDA graph (public API: WaveletSession)
    EV_STRIDE = 8
    ev_steps = list(range(0, args.steps, EV_STRIDE))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2 * k_max)] for _ in ev_steps]
    for row in ev:                                 # materialise the handles
        for e in row:
            e.record()
    torch.cuda.synchronize()
    import ctypes as C
    ev_arrays = [(C.c_void_p * (2 * k_max))(*[e.cuda_event for e in row]) for row in ev]
    session = None
    if flips is None and not args.no_graph and not args.no_sell:
        session = egnn.WaveletSession(graph, k=k_max, s=scales, f=f)
        if x0 is not None:
            session.x0.copy_(x0)
        for _ in range(3):
            session()
        torch.cuda.synchronize()

    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    # narrow path: the step is ONE kernel, so the events go around the graph replay itself (same
    # stream) and no step of the timed region pays an eager launch; other paths: the library records
    # the per-order events on eager steps
    replay_events = narrow and session is not None
    for i in range(args.steps):
        if i % EV_STRIDE == 0 and replay_events:
            row = ev[i // EV_STRIDE]
            row[0].record()
            out = session()
            row[1].record()
        elif i % EV_STRIDE == 0:
            out = step(ev_arrays[i // EV_STRIDE])
        elif session is not None:
            out = session()
        else:
            out = step()
    stop.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs:
        dump_features(args.dump_outputs, out)     # before anything else replays the session into the same buffer
    ms_per_step = start.elapsed_time(stop) / args.steps
    value = work / (ms_per_step * 1e-3)

    b_k = contract_bytes(n, nnz, f, k_max, n_scales)
    g_k = gather_bytes(n, nnz, f, k_max, n_scales)
    traffic, traffic_src = dram_traffic(f"{args.workload}_f{f}_k{k_max}_s{n_scales}")
    if narrow:
        # one launch = the whole step (K orders): events 0/1 bracket the kernel
        launch_ms = float(np.mean([row[0].elapsed_time(row[1]) for row in ev]))
        own = sell_stream_bytes(plan, n, k_max, n_scales)
        phases = read_phase_stamps(plan, k_max, first_operand_in_kernel=False)   # dinv * X0 is cached (and patched) per graph
        enable_phase_stamps(plan, False)
        achieved = sum(own) / (launch_ms * 1e-3) / 1e9
        spmv_us = float(np.mean(phases["spmv"]))
        roofline = {
            "bound": "hbm", "kernel": "sell_step_kernel", "launches_per_step": 1, "orders_per_launch": k_max,
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": float(sum(own)), "avg_launch_ms": launch_ms,
            "bytes_model": "own stream: 2 B x padded entries + slice tables + partial sums + per-row vectors, per order "
                           "(DESIGN.md 4.2); K orders per launch",
            "achieved_contract": sum(b_k) / (launch_ms * 1e-3) / 1e9, "frac_contract": sum(b_k) / (launch_ms * 1e-3) / 1e9 / peak,
            "contract_bytes_per_launch": float(sum(b_k)),
            "b_gather_bytes_per_launch": float(sum(g_k)), "b_gather_achieved": sum(g_k) / (launch_ms * 1e-3) / 1e9,
            "traffic": traffic, "traffic_source": traffic_src,
            "phase_us": phases,
            "spmv_phase": {"us_per_order": spmv_us, "bytes_per_order": float(own[0]),
                           "achieved": own[0] / (spmv_us * 1e-6) / 1e9, "frac": own[0] / (spmv_us * 1e-6) / 1e9 / peak,
                           "note": "operand staging + slices + closing grid barrier of one order, from the kernel's own "
                                   "globaltimer stamps (last launch of the timed region)"},
            "kernel_share_of_step": launch_ms / ms_per_step,
            # the events bracket a graph replay of the cooperative launch and include its launch latency
            # (share of step > 1); the kernel's own clock from its first to its last instruction:
            "kernel_clock_ms": phases["total"] * 1e-3,
            "frac_by_kernel_clock": sum(own) / (phases["total"] * 1e-6) / 1e9 / peak,
            "padded_entries": int(plan.n_entries), "virtual_rows": int(plan.n_rowv),
        }
        launches_per_step = (k_max + 15) // 16          # edge flips ride in the same launch (PATCH instantiation)
    else:
        order_ms = np.array([[row[2 * j].elapsed_time(row[2 * j + 1]) for j in range(k_max)] for row in ev])
        avg_launch_ms = float(order_ms.mean())
        achieved = (sum(b_k) / k_max) / (avg_launch_ms * 1e-3) / 1e9
        kernel_name = "cheb_wide_kernel" if f >= 8 else "cheb_order_kernel"
        roofline = {"bound": "hbm", "kernel": kernel_name, "launches_per_step": k_max, "achieved": achieved, "peak": peak,
                    "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": sum(b_k) / k_max, "avg_launch_ms": avg_launch_ms,
                    "bytes_model": "SURVEY 8d contract bytes B_k (int32 CSR, every T row read once), per order",
                    "b_gather_bytes_per_launch": sum(g_k) / k_max,
                    "b_gather_achieved": (sum(g_k) / k_max) / (avg_launch_ms * 1e-3) / 1e9,
                    "traffic": traffic, "traffic_source": traffic_src,
                    "per_order_ms": [float(v) for v in order_ms.mean(axis=0)],
                    "kernel_share_of_step": float(order_ms.sum(axis=1).mean() / ms_per_step)}
        if f >= 8:
            launches_per_step = 1 + k_max + (1 if (f + 3) // 4 * 4 > 128 else 0)
        else:
            launches_per_step = k_max + (1 if f <= 4 else 0)

    # the two wide shapes the >= 70 % target names, in the same run
    roofline_wide = None
    if not args.no_wide and args.workload == "reddit" and f == 1 and flips is None:
        roofline_wide = [wide_record(egnn, synth, "arxiv", 128, None, dev, peak),
                         wide_record(egnn, synth, "reddit", 64, graph, dev, peak)]

    # UGCA per-perturbation recompute on the resident graph: host flip list in -> features on the host
    ugca = None
    if not args.no_ugca and f == 1 and flips is None:
        budget = 5
        cands = [make_flips(n, budget, 100 + i) for i in range(64)]
        it = iter(cands * 8)
        dev_ms = time_steps(lambda: egnn.graph_wavelet_features(graph, k=k_max, s=scales, deltas=next(it)), 100, 5)
        out_h = torch.empty((n, n_scales), dtype=torch.float32).pin_memory()

        def ugca_e2e():
            feats = egnn.graph_wavelet_features(graph, k=k_max, s=scales, deltas=next(it))
            out_h.copy_(feats, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        for _ in range(5):
            ugca_e2e()
        t0 = time.perf_counter()
        for _ in range(100):
            ugca_e2e()
        e_ms = (time.perf_counter() - t0) / 100 * 1e3
        ugca = {"flips": budget, "recompute_ms": dev_ms, "value": work / (dev_ms * 1e-3),
                "e2e_ms": e_ms, "e2e_value": work / (e_ms * 1e-3), "h2d_bytes_per_step": 2 * budget * 12,
                "d2h_bytes_per_step": int(out_h.numel() * 4), "unperturbed_ms": ms_per_step,
                "entry": "graph_wavelet_features(resident graph, deltas=(rows, cols, vals)): degree patch + step kernel "
                         "with the flips as kernel arguments (calib_fga.py:868,908,952 recompute point); no CSR/plan rebuild"}

    # end to end through the host-buffer entry: pinned CSR -> device -> features -> host
    e2e = None
    if not args.no_e2e:
        rp_h = graph.rowptr.cpu().pin_memory()
        ci_h = graph.colidx.cpu().pin_memory()
        x0_h = None if x0 is None else x0.cpu().pin_memory()
        out_h = torch.empty((n, n_scales * f), dtype=torch.float32).pin_memory()
        h2d = rp_h.numel() * 4 + ci_h.numel() * 4 + (0 if x0_h is None else x0_h.numel() * 4)
        d2h = out_h.numel() * 4

        entry = "CsrGraph.from_host_csr + graph_wavelet_features (pinned host CSR in, host features out)"
        dense_h = None
        if args.entry == "dense":
            if 4 * n * n > 8e9:
                raise SystemExit("--entry dense needs the [N,N] float32 adjacency to fit comfortably; use cora/pubmed/physics")
            import scipy.sparse as sp
            adj = sp.csr_matrix((np.ones(nnz, np.float32), graph.colidx.cpu().numpy(), graph.rowptr.cpu().numpy()),
                                shape=(n, n))
            dense_h = torch.from_numpy(adj.toarray()).pin_memory()
            h2d = dense_h.numel() * 4 + (0 if x0_h is None else x0_h.numel() * 4)
            entry = ("graph_wavelet_features(dense [N,N] float32 adjacency): pinned host dense in -> device "
                     "dense->CSR kernels -> features -> host (the reference boundary, calibration/WATS.py:99-100)")

        def e2e_step():
            if dense_h is not None:
                g = egnn.CsrGraph.from_dense(dense_h.to(dev, non_blocking=True))
            else:
                g = egnn.CsrGraph.from_host_csr(rp_h, ci_h, None, n, device=dev)
            xx = None if x0_h is None else x0_h.to(dev, non_blocking=True)
            feats = egnn.graph_wavelet_features(g, k=k_max, s=scales, X0=xx, _use_sell=use_sell)
            out_h.copy_(feats, non_blocking=True)
            torch.cuda.current_stream().synchronize()

        e_steps = max(3, min(args.steps, 20))
        for _ in range(3):
            e2e_step()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(e_steps):
            e2e_step()
        torch.cuda.synchronize()
        e_dt = (time.perf_counter() - t0) / e_steps
        e2e = {"value": work / e_dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": e_dt * 1e3, "steps": e_steps, "entry": entry,
               "note": "one-shot use of a fresh graph: the plan-free blocked kernel for large column-sorted graphs, else the "
                       "generic CSR kernel (the SELL plan pays off from the second use of a graph on); the H2D copy of the "
                       "CSR is ~85 % of the step"}

    # the reference's own code on the SAME graph (host copy of the resident CSR), one core like the reference
    cpu_baseline = None
    if not args.no_cpu_baseline:
        import scipy.sparse as sp
        adj = sp.csr_matrix((np.ones(nnz, np.float32), graph.colidx.cpu().numpy(), graph.rowptr.cpu().numpy()), shape=(n, n))
        if k_max * f > REFERENCE_FULL_GRAPH_LIMIT and nnz > 5_000_000:
            cpu_baseline = {"skipped": "wide signal on a large graph: run `bench.py --impl reference` (bounded sample)"}
        else:
            cpu_baseline = time_cpu_path(adj, k_max, scales, f, stock_runs=1, split_run=False)

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, n, nnz, k_max, n_scales, f, args.flips),
        "run": {"parallelism": "1 GPU", "path": "sell-step" if narrow else ("wide" if f >= 8 else "csr-generic"),
                "cuda_graph": session is not None, "event_stride": EV_STRIDE,
                "events": "around the graph replay of the one-kernel step" if replay_events else "per order, recorded by the library on eager steps"},
        "roofline": roofline, "roofline_wide": roofline_wide, "ugca": ugca, "cpu_baseline": cpu_baseline, "e2e": e2e,
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": sampler.summary(),
    }
    print(json.dumps(line), flush=True)


def run_replicas(args, rank, local_rank, world):
    """UGCA replica mode (SURVEY 8e): candidates are independent, so each rank keeps the whole
    graph resident and recomputes the features of its own candidates (edge flips around a target
    node applied on top of the resident CSR / SELL plan).  No data-path collective."""
    import torch.distributed as dist
    import efficient_gnn_b200 as egnn
    from efficient_gnn_b200 import synth
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    f = args.f or DEFAULT_F[args.workload]
    k_max, n_scales = args.order, args.scales
    scales = scale_list(n_scales)
    rp, ci, n = synth.synth_csr(args.workload, self_loops=True, device=dev)
    graph = egnn.CsrGraph(rp, ci, None, n)
    nnz = graph.nnz
    x0 = None if f == 1 else torch.randn(n, f, device=dev, generator=torch.Generator(device=dev).manual_seed(3))
    budget = args.flips or 5
    cands = [make_flips(n, budget, 1000 * (rank + 1) + i) for i in range(args.steps + max(3, args.warmup))]
    it = iter(cands)
    for _ in range(max(3, args.warmup)):
        egnn.graph_wavelet_features(graph, k=k_max, s=scales, X0=x0, deltas=next(it))
    torch.cuda.synchronize()
    dist.barrier()
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        egnn.graph_wavelet_features(graph, k=k_max, s=scales, X0=x0, deltas=next(it))
    stop.record()
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join()
    ms = torch.tensor([start.elapsed_time(stop) / args.steps], device=dev, dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    dist.barrier()
    ms_per_step = float(ms.item())
    if rank == 0:
        work = float(nnz) * k_max * f * world            # every rank finishes one candidate per step
        line = {
            "metric": METRIC, "value": work / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, n, nnz, k_max, n_scales, f, budget),
            "run": {"parallelism": f"{world} replicas: whole graph per GPU, one perturbation candidate per rank "
                                   "per step, no exchange"},
            "roofline": None, "cpu_baseline": None, "e2e": None,
            "gpu_launches": int(5 * args.steps * world), "clocks": sampler.summary(),
        }
        print(json.dumps(line), flush=True)
    dist.barrier()
    sys.stdout.flush()
    os._exit(0)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs is implemented for the one-GPU run only; a multi-GPU run compares every "
                         "rank's rows with the single-GPU path instead (the 'check' record; off with --no-check)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
