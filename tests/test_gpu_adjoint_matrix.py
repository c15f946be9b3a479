"""Every adjoint instantiation against the float64 gradient, element-wise.

The backward of the wavelet pass launches one adjoint instantiation of the forward's order
kernel per application of the transposed operator (``egnn_cheb_adjoint``): the wide kernel
(``csrc/wide.cuh``, F >= 8) keyed by ``<NZ_LOG2, HAS_VALS, ALIGNED, PEER, DYN, ADJ>`` and the
generic kernel (``csrc/cheb.cuh``, F < 8) keyed by ``<VEC, U, HAS_VALS, PRESCALED, ADJ>``.

* ``TABLE``: one row per (graph, F) that reaches a given instantiation, each compared with
  ``tests/vjp_reference.wavelet_vjp`` (float64, explicit transposed operator) for the signal's
  and the scales' gradients: norm-wise <= 1e-5 (1e-4 above 16 orders) and element-wise ratio
  <= 1 at the 5e-2 floor; the ratio at the 1e-3 floor is printed beside them.
* Edges: K in {0, 1, 2, 20}, eight scales, the empty graph, a zero signal row under the
  normalisation, flips on a weighted directed graph with hub rows.
* ``test_every_reachable_adjoint_instantiation_runs``: the kernels the table launches, read
  from ``torch.profiler``, are exactly the 42 reachable ones.
* The helper routines through the C ABI: ``egnn_csr_transpose``, ``egnn_l1_normalize[_backward]``
  and ``egnn_cheb_coeff_grad`` against numpy, each run twice (bitwise equal).
* Caller buffers at an odd element offset give the same bits as aligned copies.
"""
import re
import zlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import _cabi
from helpers import elementwise_ratio, rel_max_err
from vjp_reference import wavelet_vjp

pytestmark = pytest.mark.gpu

SCALES = [0.8, 0.4, 1.3, 2.0, 0.2, 1.0, 0.6, 1.6]
ISOLATED = range(0, 5)          # nodes without any entry
LOOPS = range(10, 40)           # nodes with a stored self loop
OUT_HUB, IN_HUB, LAST_IN = 50, 60, 70
HUB_DEGREE = 2100               # >= 2048 (kHubDegree): summed by a whole CTA on the wide path
# the forward matrix's extra graphs ("dense_hubs_*", "sparse_long_*"): nodes whose only entry is a
# stored self loop, out-hub rows on a graph dense enough for the static wide schedule, and
# consecutive long rows that share one warp of the generic kernel
LOOP_ONLY = range(5, 8)
HUB_ROWS = (50, 51, 52)
LONG_ROWS = range(208, 216)


# ---- graphs ------------------------------------------------------------------------------------
def _pattern(rng, n, deg, directed):
    m = n * deg if directed else n * deg // 2
    r, c = rng.integers(0, n, m), rng.integers(0, n, m)
    keep = r != c
    r, c = r[keep], c[keep]
    if not directed:
        r, c = np.concatenate([r, c]), np.concatenate([c, r])
    a = sp.csr_matrix((np.ones(r.size, np.float32), (r, c)), shape=(n, n))
    a.sum_duplicates()
    return a.tocoo()


def build_graph(name):
    """Seeded scipy CSR (float32): binary symmetric or weighted (0.5-2) directed, with isolated
    nodes and stored self loops; the star variants add a row (out-star) or a column (in-star)
    of HUB_DEGREE entries to the weighted sparse graph.  "dense_hubs_*" (3000 nodes, ~72
    entries per row: >= 64 per row, the static wide schedule) adds the out-hub rows HUB_ROWS;
    "sparse_long_*" gives the rows LONG_ROWS 150-400 entries each.  Both have LOOP_ONLY nodes
    and a node LAST_IN with exactly one in-edge (from node 80), as "stars_w" has."""
    if name == "empty":
        return sp.csr_matrix((700, 700), dtype=np.float32)
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    dense = name.startswith("dense")
    weighted = not name.endswith("bin")
    extras = name.startswith(("dense_hubs", "sparse_long"))
    n, deg = (3000, 72) if name.startswith("dense_hubs") else (2000, 96) if dense else (3000, 8)
    a = _pattern(rng, n, deg, directed=weighted)
    r, c = a.row, a.col
    extra_r, extra_c = [np.asarray(LOOPS)], [np.asarray(LOOPS)]
    if name in ("out_star_w", "stars_w"):
        cols = rng.choice(np.arange(100, n), HUB_DEGREE, replace=False)
        extra_r.append(np.full(HUB_DEGREE, OUT_HUB)); extra_c.append(cols)
    if name in ("in_star_w", "stars_w"):
        rows = rng.choice(np.arange(100, n), HUB_DEGREE, replace=False)
        extra_r.append(rows); extra_c.append(np.full(HUB_DEGREE, IN_HUB))
    if name.startswith("dense_hubs"):
        for h in HUB_ROWS:
            extra_r.append(np.full(HUB_DEGREE, h)); extra_c.append(rng.choice(np.arange(100, n), HUB_DEGREE, replace=False))
    if name.startswith("sparse_long"):
        for i in LONG_ROWS:
            d = int(rng.integers(150, 400))
            extra_r.append(np.full(d, i)); extra_c.append(rng.choice(np.arange(100, n), d, replace=False))
    r, c = np.concatenate([r] + extra_r), np.concatenate([c] + extra_c)
    if name == "stars_w" or extras:        # LAST_IN keeps exactly one in-edge (from node 80)
        keep = c != LAST_IN
        r, c = np.concatenate([r[keep], [80]]), np.concatenate([c[keep], [LAST_IN]])
    cut = list(ISOLATED) + (list(LOOP_ONLY) if extras else [])
    iso = np.isin(r, cut) | np.isin(c, cut)
    r, c = r[~iso], c[~iso]
    if extras:
        r, c = np.concatenate([r, LOOP_ONLY]), np.concatenate([c, LOOP_ONLY])
    a = sp.csr_matrix((np.ones(r.size, np.float32), (r, c)), shape=(n, n))
    a.sum_duplicates()
    a.data[:] = 1.0
    if weighted:
        a.data = rng.uniform(0.5, 2.0, a.nnz).astype(np.float32)
    a.sort_indices()
    return a


_GRAPHS = {}


def graph(name):
    """(scipy adjacency, device graph); the device graph keeps its transpose and row order."""
    if name not in _GRAPHS:
        adj = build_graph(name)
        _GRAPHS[name] = (adj, egnn.as_graph(adj))
    return _GRAPHS[name]


# ---- one case ----------------------------------------------------------------------------------
def upstream(n, n_scales, f, k, seed, with_tbar):
    rng = np.random.default_rng(seed)
    f32 = lambda *shape: rng.standard_normal(shape).astype(np.float32).astype(np.float64)   # noqa: E731
    return f32(n, n_scales * f), f32(n, n_scales, f), (f32(k + 1, n, f) if with_tbar else None)


def run_gpu(g, n, f, k, n_scales, lam, normalize, seed, with_tbar=True, deltas=None, x_np=None):
    """Forward with return_parts and backward of <Hbar, features> + <Cbar, combined> (+ sum_k
    <Tbar_k, T_k>); returns (X0.grad, s.grad, the signal, the upstream gradients)."""
    rng = np.random.default_rng(seed + 1000)
    if x_np is None:
        x_np = rng.standard_normal((n, f)).astype(np.float32)
    hb, cb, tb = upstream(n, n_scales, f, k, seed, with_tbar)
    x = torch.tensor(x_np, device="cuda", requires_grad=True)
    s = torch.tensor(SCALES[:n_scales], dtype=torch.float64, requires_grad=True)
    res = egnn.graph_wavelet_features(g, k=k, s=s, X0=x, lambda_max=lam, normalize=normalize, return_parts=True,
                                      deltas=deltas)
    dev = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")      # noqa: E731
    loss = (dev(hb) * res.features).sum() + (dev(cb) * res.combined).sum()
    if tb is not None:
        loss = loss + sum((dev(tb[i]) * res.orders[i]).sum() for i in range(k + 1))
    loss.backward()
    return x.grad.cpu().numpy(), s.grad.numpy(), x_np, (hb, cb, tb)


def check(tag, got, ref, tol):
    err = rel_max_err(got, ref)
    r5 = elementwise_ratio(got, ref, tol)
    r3 = elementwise_ratio(got, ref, tol, floor=1e-3)
    print(f"\n[{tag}] rel {err:.2e}, elementwise_ratio x{r5:.2f} (floor 5e-2), x{r3:.2f} (floor 1e-3)")
    assert np.all(np.isfinite(got)), f"{tag}: non-finite gradient"
    assert err <= tol, f"{tag}: rel max err {err:.3e}"
    assert r5 <= 1.0, f"{tag}: elementwise ratio {r5:.2f} at the 5e-2 floor"


def tol_for(k):
    return 1e-4 if k > 16 else 1e-5


def compare(tag, adj, f, k, n_scales, lam, normalize, seed, with_tbar=True, deltas=None, ref_adj=None, g=None):
    n = adj.shape[0]
    xg, sg, x_np, (hb, cb, tb) = run_gpu(g, n, f, k, n_scales, lam, normalize, seed, with_tbar, deltas)
    xr, sr = wavelet_vjp(adj if ref_adj is None else ref_adj, k, SCALES[:n_scales], x_np.astype(np.float64), lam,
                         normalize, hb, cb, tb)
    check(f"{tag} Xbar", xg, xr, tol_for(k))
    check(f"{tag} sbar", sg, sr, tol_for(k))


# ---- the case table ----------------------------------------------------------------------------
# (graph, F, K, S, lambda_max, normalize, Tbar given, instantiation launched by every application).
# wide<NZ_LOG2, HAS_VALS, ALIGNED, PEER, DYN, ADJ>: NZ_LOG2 = 5 - ceil(log2(ceil4(F) / 4)) (0 from
# F = 100 up); DYN when one feature tile covers the row (F <= 128) and nnz < 64 n (the sparse
# graphs; the dense ones have ~96 entries per row).  order<VEC, U, HAS_VALS, PRESCALED, ADJ>:
# VEC = 4 for F = 4, PRESCALED for F <= 4.
TABLE = [
    ("sparse_bin", 8, 3, 1, 2.0, True, True, "wide<4,0,1,0,1,1>"),
    ("sparse_w", 8, 4, 2, 1.7, False, True, "wide<4,1,1,0,1,1>"),
    ("dense_bin", 8, 3, 3, 2.0, True, False, "wide<4,0,1,0,0,1>"),
    ("dense_w", 8, 2, 2, 1.7, True, True, "wide<4,1,1,0,0,1>"),
    ("sparse_bin", 12, 3, 2, 2.0, True, False, "wide<3,0,1,0,1,1>"),
    ("out_star_w", 12, 3, 1, 2.0, True, True, "wide<3,1,1,0,1,1>"),
    ("dense_bin", 12, 2, 1, 1.7, False, True, "wide<3,0,1,0,0,1>"),
    ("dense_w", 12, 3, 2, 2.0, True, True, "wide<3,1,1,0,0,1>"),
    ("sparse_bin", 10, 4, 1, 1.7, True, True, "wide<3,0,0,0,1,1>"),
    ("in_star_w", 10, 3, 2, 2.0, True, False, "wide<3,1,0,0,1,1>"),
    ("dense_bin", 10, 3, 2, 2.0, True, True, "wide<3,0,0,0,0,1>"),
    ("dense_w", 10, 2, 1, 1.7, False, True, "wide<3,1,0,0,0,1>"),
    ("sparse_bin", 24, 2, 3, 2.0, False, True, "wide<2,0,1,0,1,1>"),
    ("sparse_w", 24, 3, 2, 2.0, True, True, "wide<2,1,1,0,1,1>"),
    ("dense_bin", 24, 3, 1, 2.0, True, True, "wide<2,0,1,0,0,1>"),
    ("dense_w", 24, 3, 3, 1.7, True, False, "wide<2,1,1,0,0,1>"),
    ("sparse_bin", 19, 3, 1, 2.0, True, True, "wide<2,0,0,0,1,1>"),
    ("out_star_w", 19, 4, 2, 1.7, True, True, "wide<2,1,0,0,1,1>"),
    ("dense_bin", 19, 2, 2, 2.0, False, True, "wide<2,0,0,0,0,1>"),
    ("dense_w", 19, 3, 1, 2.0, True, True, "wide<2,1,0,0,0,1>"),
    ("sparse_bin", 48, 3, 2, 1.7, True, True, "wide<1,0,1,0,1,1>"),
    ("in_star_w", 48, 3, 1, 2.0, True, True, "wide<1,1,1,0,1,1>"),
    ("dense_bin", 48, 3, 1, 2.0, True, False, "wide<1,0,1,0,0,1>"),
    ("dense_w", 48, 2, 2, 2.0, False, True, "wide<1,1,1,0,0,1>"),
    ("sparse_bin", 37, 3, 1, 2.0, False, False, "wide<1,0,0,0,1,1>"),
    ("sparse_w", 37, 3, 2, 1.7, True, True, "wide<1,1,0,0,1,1>"),
    ("dense_bin", 37, 2, 1, 2.0, True, True, "wide<1,0,0,0,0,1>"),
    ("dense_w", 37, 3, 2, 2.0, True, True, "wide<1,1,0,0,0,1>"),
    ("sparse_bin", 128, 3, 1, 2.0, True, True, "wide<0,0,1,0,1,1>"),
    ("out_star_w", 128, 3, 2, 2.0, True, True, "wide<0,1,1,0,1,1>"),
    ("dense_bin", 128, 2, 2, 1.7, True, True, "wide<0,0,1,0,0,1>"),
    ("dense_w", 128, 3, 1, 2.0, False, True, "wide<0,1,1,0,0,1>"),
    ("sparse_bin", 99, 2, 2, 2.0, True, True, "wide<0,0,0,0,1,1>"),
    ("in_star_w", 99, 3, 1, 1.7, True, True, "wide<0,1,0,0,1,1>"),
    ("dense_bin", 99, 3, 1, 2.0, True, False, "wide<0,0,0,0,0,1>"),
    ("dense_w", 99, 2, 2, 2.0, True, True, "wide<0,1,0,0,0,1>"),
    ("sparse_bin", 130, 3, 2, 2.0, True, True, "wide<0,0,0,0,0,1>"),
    ("sparse_w", 130, 3, 1, 1.7, True, False, "wide<0,1,0,0,0,1>"),
    ("sparse_bin", 260, 2, 1, 2.0, True, True, "wide<0,0,1,0,0,1>"),
    ("in_star_w", 260, 3, 2, 2.0, True, True, "wide<0,1,1,0,0,1>"),
    ("sparse_bin", 1, 3, 2, 2.0, False, True, "order<1,1,0,1,1>"),
    ("out_star_w", 1, 4, 1, 1.7, False, True, "order<1,1,1,1,1>"),
    ("dense_bin", 2, 3, 1, 2.0, True, True, "order<1,1,0,1,1>"),
    ("in_star_w", 2, 3, 2, 2.0, True, False, "order<1,1,1,1,1>"),
    ("sparse_bin", 3, 3, 3, 1.7, True, True, "order<1,1,0,1,1>"),
    ("dense_w", 3, 2, 1, 2.0, True, True, "order<1,1,1,1,1>"),
    ("dense_bin", 4, 3, 2, 2.0, True, True, "order<4,1,0,1,1>"),
    ("sparse_w", 4, 3, 1, 1.7, True, True, "order<4,1,1,1,1>"),
    ("in_star_w", 4, 4, 2, 2.0, True, False, "order<4,1,1,1,1>"),
    ("sparse_bin", 5, 3, 2, 2.0, True, True, "order<1,1,0,0,1>"),
    ("out_star_w", 5, 3, 1, 2.0, True, True, "order<1,1,1,0,1>"),
    ("dense_bin", 6, 2, 1, 1.7, True, False, "order<1,1,0,0,1>"),
    ("dense_w", 6, 3, 2, 2.0, False, True, "order<1,1,1,0,1>"),
    ("sparse_bin", 7, 3, 1, 2.0, True, True, "order<1,1,0,0,1>"),
    ("sparse_w", 7, 4, 3, 2.0, True, True, "order<1,1,1,0,1>"),
]

# The 42 instantiations egnn_cheb_adjoint can launch on one GPU.  Compiled as well but unreachable
# (checked against `cuobjdump -symbols` of the library): wide<4,0,0,0,0,1>, wide<4,0,0,0,1,1>,
# wide<4,1,0,0,0,1>, wide<4,1,0,0,1,1> (NZ_LOG2 = 4 means F <= 8, and F = 5..7 run the generic
# kernel), order<4,1,*,0,1> (VEC = 4 only for F = 4, which is pre-scaled) and order<1,4,*,*,1>
# (U = 4 only for F > 32, which runs the wide kernel).
REACHABLE = {
    "wide<0,0,0,0,0,1>", "wide<0,0,0,0,1,1>", "wide<0,0,1,0,0,1>", "wide<0,0,1,0,1,1>",
    "wide<0,1,0,0,0,1>", "wide<0,1,0,0,1,1>", "wide<0,1,1,0,0,1>", "wide<0,1,1,0,1,1>",
    "wide<1,0,0,0,0,1>", "wide<1,0,0,0,1,1>", "wide<1,0,1,0,0,1>", "wide<1,0,1,0,1,1>",
    "wide<1,1,0,0,0,1>", "wide<1,1,0,0,1,1>", "wide<1,1,1,0,0,1>", "wide<1,1,1,0,1,1>",
    "wide<2,0,0,0,0,1>", "wide<2,0,0,0,1,1>", "wide<2,0,1,0,0,1>", "wide<2,0,1,0,1,1>",
    "wide<2,1,0,0,0,1>", "wide<2,1,0,0,1,1>", "wide<2,1,1,0,0,1>", "wide<2,1,1,0,1,1>",
    "wide<3,0,0,0,0,1>", "wide<3,0,0,0,1,1>", "wide<3,0,1,0,0,1>", "wide<3,0,1,0,1,1>",
    "wide<3,1,0,0,0,1>", "wide<3,1,0,0,1,1>", "wide<3,1,1,0,0,1>", "wide<3,1,1,0,1,1>",
    "wide<4,0,1,0,0,1>", "wide<4,0,1,0,1,1>", "wide<4,1,1,0,0,1>", "wide<4,1,1,0,1,1>",
    "order<4,1,0,1,1>", "order<4,1,1,1,1>", "order<1,1,0,1,1>", "order<1,1,1,1,1>",
    "order<1,1,0,0,1>", "order<1,1,1,0,1>",
}


def case_id(c):
    return f"{c[0]}-F{c[1]}-K{c[2]}-S{c[3]}"


@pytest.mark.parametrize("case", TABLE, ids=[case_id(c) for c in TABLE])
def test_adjoint_matrix_vs_float64(case):
    name, f, k, n_scales, lam, normalize, with_tbar, _kernel = case
    adj, g = graph(name)
    compare(f"{case_id(case)} lam={lam} norm={normalize} tbar={with_tbar}", adj, f, k, n_scales, lam, normalize,
            seed=f * 31 + k, with_tbar=with_tbar, g=g)


# ---- which kernels run -------------------------------------------------------------------------
_KERNEL = re.compile(r"(cheb_wide|cheb_order|sell_step|blocked_spmv)_kernel<([^>]*)>")
_SHORT = {"cheb_wide": "wide", "cheb_order": "order"}


def kernel_keys(names, adj):
    """Normalised ``wide<...>`` / ``order<...>`` keys of the order-kernel instantiations among
    kernel names whose last template argument (ADJ) equals ``adj``, whichever way the demangler
    spells the arguments.  With ``adj`` false the narrow forward kernels, which have no adjoint
    instantiation, are kept too: ``sell_step<PEER,PATCH>`` and ``blocked_spmv<HAS_VALS>``."""
    out = set()
    for name in names:
        m = _KERNEL.search(name)
        if not m:
            continue
        args = []
        for a in m.group(2).split(","):
            a = re.sub(r"^\((?:bool|int)\)", "", a.strip())
            args.append({"true": 1, "false": 0}[a] if a in ("true", "false") else int(a))
        family = m.group(1)
        if family in _SHORT and args[-1] != int(adj):
            continue
        if family not in _SHORT and adj:
            continue
        out.add(f"{_SHORT.get(family, family)}<{','.join(map(str, args))}>")
    return out


def adjoint_kernels(names):
    """Normalised keys of the adjoint (last template argument true) instantiations."""
    return kernel_keys(names, adj=True)


def _profiled_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


def test_every_reachable_adjoint_instantiation_runs():
    probe = _profiled_kernels(lambda: torch.ones(1 << 16, device="cuda").mul_(2.0))
    if not probe:
        pytest.skip("torch.profiler records no CUDA kernel here (CUPTI unavailable): coverage not measurable")
    assert adjoint_kernels(["void egnn::cheb_wide_kernel<(int)3, (bool)1, (bool)0, (bool)0, (bool)1, (bool)1>("
                            "egnn::WideParams)"]) == {"wide<3,1,0,0,1,1>"}
    assert adjoint_kernels(["void egnn::cheb_order_kernel<4, 1, true, true, true>(egnn::OrderParams)"]) == \
        {"order<4,1,1,1,1>"}
    launched = set()
    for case in TABLE:
        name, f, k, n_scales, lam, normalize, with_tbar, kernel = case
        adj, g = graph(name)
        got = adjoint_kernels(_profiled_kernels(
            lambda: run_gpu(g, adj.shape[0], f, k, n_scales, lam, normalize, seed=1, with_tbar=with_tbar)))
        assert got == {kernel}, f"{case_id(case)}: launched {sorted(got)}, the table says {kernel}"
        launched |= got
    assert len(REACHABLE) == 42
    print(f"\n[coverage] {len(launched & REACHABLE)} of {len(REACHABLE)} reachable adjoint instantiations launched")
    assert launched == REACHABLE, f"missing {sorted(REACHABLE - launched)}, unexpected {sorted(launched - REACHABLE)}"


# ---- edges -------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [0, 1, 2, 20])
@pytest.mark.parametrize("f", [1, 4, 8, 130])
def test_order_count_edges(f, k):
    """K = 0 (the prologue alone writes Xbar), K = 1 (one application, no b_{k+2}), K > 16."""
    adj, g = graph("sparse_w")
    compare(f"sparse_w F={f} K={k}", adj, f, k, 2, 1.7, f > 1, seed=7 * f + k, g=g)


@pytest.mark.parametrize("name,f", [("sparse_bin", 1), ("sparse_w", 1), ("sparse_w", 130), ("dense_bin", 130)])
def test_eight_scales(name, f):
    adj, g = graph(name)
    compare(f"{name} F={f} S=8", adj, f, 3, 8, 2.0, f > 1, seed=f + 8, g=g)


@pytest.mark.parametrize("f", [1, 4, 8, 130])
def test_empty_graph_closed_form(f):
    """No edges, lambda_max = 2: M = -I, so Xbar = sum_k (-1)^k v_k."""
    adj, g = graph("empty")
    n, k, n_scales = adj.shape[0], 3, 2
    xg, sg, x_np, (hb, cb, tb) = run_gpu(g, n, f, k, n_scales, 2.0, False, seed=f)
    alpha = egnn.heat_coefficients(k, SCALES[:n_scales])
    cbar = cb + hb.reshape(n, n_scales, f)
    want = sum((-1) ** i * (np.einsum("s,nsf->nf", alpha[:, i], cbar) + tb[i]) for i in range(k + 1))
    check(f"empty F={f} Xbar", xg, want, 1e-5)
    # T_k = (-1)^k X0: sbar_j = -sum_k k alpha[j,k] (-1)^k <Cbar_j, X0>
    dots = np.einsum("nsf,nf->s", cbar, x_np.astype(np.float64))
    swant = np.array([-sum(i * alpha[j, i] * (-1) ** i for i in range(k + 1)) * dots[j] for j in range(n_scales)])
    check(f"empty F={f} sbar", sg, swant, 1e-5)


@pytest.mark.parametrize("f", [3, 8, 130])
def test_zero_signal_row_under_normalisation(f):
    """An isolated node with a zero signal row: its combination is exactly zero, so the
    normalisation's backward divides by 1e-8 alone.  The gradient there is finite and equals the
    reference's Hbar / 1e-8 carried through M^T = -1 on that row; every other row is compared as usual."""
    adj, g = graph("sparse_bin")
    n, k, n_scales = adj.shape[0], 3, 2
    x_np = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)
    x_np[0] = 0.0                                             # node 0 is isolated
    xg, sg, _, (hb, cb, tb) = run_gpu(g, n, f, k, n_scales, 2.0, True, seed=f, x_np=x_np)
    xr, sr = wavelet_vjp(adj, k, SCALES[:n_scales], x_np.astype(np.float64), 2.0, True, hb, cb, tb)
    assert np.all(np.isfinite(xg))
    alpha = egnn.heat_coefficients(k, SCALES[:n_scales])
    v = [np.einsum("s,sf->f", alpha[:, i], cb[0] + hb[0].reshape(n_scales, f) / 1e-8) + tb[i][0] for i in range(k + 1)]
    closed = sum((-1) ** i * v[i] for i in range(k + 1))
    np.testing.assert_allclose(xr[0], closed, rtol=1e-12)
    assert np.abs(xr[0]).max() > 1e6
    check(f"zero row F={f} Xbar[0]", xg[0], xr[0], 1e-5)
    check(f"zero row F={f} Xbar[1:]", xg[1:], xr[1:], 1e-5)
    check(f"zero row F={f} sbar", sg, sr, 1e-5)


def star_flips(adj):
    """Flips on the weighted directed star graph: remove LAST_IN's only in-edge, remove one entry of
    the out-hub's row, add an edge into the in-hub (a new entry of the transpose's hub row), and a
    few random additions and removals."""
    a = adj.tocsr()
    rows, cols, vals = [80], [LAST_IN], [-float(a[80, LAST_IN])]
    c = int(a.indices[a.indptr[OUT_HUB] + 7])
    rows.append(OUT_HUB); cols.append(c); vals.append(-float(a[OUT_HUB, c]))
    r = next(i for i in range(100, adj.shape[0]) if a[i, IN_HUB] == 0)
    rows.append(r); cols.append(IN_HUB); vals.append(1.25)
    rng = np.random.default_rng(3)
    for _ in range(4):
        i, j = (int(v) for v in rng.choice(np.arange(100, adj.shape[0]), 2, replace=False))
        v = float(a[i, j])
        rows.append(i); cols.append(j); vals.append(-v if v != 0 else 0.75)
    pert = (a + sp.csr_matrix((np.array(vals, np.float32), (rows, cols)), shape=a.shape)).tocsr()
    pert.eliminate_zeros()
    assert pert[:, LAST_IN].nnz == 0
    return (rows, cols, vals), pert


@pytest.mark.parametrize("f", [5, 6, 7, 19, 128])
def test_flips_on_weighted_directed_graph(f):
    """The forward's flips, applied transposed by the adjoint, against wavelet_vjp of the
    perturbed matrix (not against the GPU's own result on the rebuilt graph)."""
    adj, g = graph("stars_w")
    deltas, pert = star_flips(adj)
    compare(f"stars_w flips F={f}", adj, f, 3, 2, 1.7, True, seed=f, deltas=deltas, ref_adj=pert, g=g)


# ---- caller buffers at an odd element offset ---------------------------------------------------
@pytest.mark.parametrize("f", [4, 8, 128])
def test_misaligned_caller_buffers(f):
    """A contiguous view 4 bytes past an allocation as X0, and an upstream gradient that is a slice
    of a torch.cat of flattened tensors, give the same bits as aligned copies."""
    adj, g = graph("sparse_w")
    n, k, sc = adj.shape[0], 3, [0.8, 1.6]
    gen = torch.Generator(device="cuda").manual_seed(f)
    x_al = torch.randn(n, f, device="cuda", generator=gen)
    g_al = torch.randn(n, 2 * f, device="cuda", generator=gen)
    for normalize in (False, True):
        buf = torch.cat([torch.zeros(1, device="cuda"), x_al.flatten()]).requires_grad_()
        x_mis = buf[1:].view(n, f)
        assert x_mis.is_contiguous() and x_mis.data_ptr() % 16 == 4
        g_mis = torch.cat([torch.zeros(3, device="cuda"), g_al.flatten()])[3:].view(n, 2 * f)
        assert g_mis.data_ptr() % 16 == 12
        with torch.no_grad():
            assert torch.equal(egnn.graph_wavelet_features(g, k=k, s=sc, X0=x_mis, normalize=normalize),
                               egnn.graph_wavelet_features(g, k=k, s=sc, X0=x_al, normalize=normalize))
        x_ref = x_al.clone().requires_grad_()
        out_ref = egnn.graph_wavelet_features(g, k=k, s=sc, X0=x_ref, normalize=normalize)
        out_ref.backward(g_al)
        out = egnn.graph_wavelet_features(g, k=k, s=sc, X0=x_mis, normalize=normalize)
        assert torch.equal(out.detach(), out_ref.detach())
        out.backward(g_mis)                  # normalize=False: the view reaches the adjoint as cbar
        assert torch.equal(buf.grad[1:].view(n, f), x_ref.grad)


# ---- helper routines through the C ABI ---------------------------------------------------------
def _dev(a, dtype):
    return torch.from_numpy(np.ascontiguousarray(a)).to(device="cuda", dtype=dtype)


def gpu_transpose(rowptr, colidx, vals, n):
    lib = _cabi.load()
    nnz = int(colidx.size)
    rp, ci = _dev(rowptr, torch.int32), _dev(colidx, torch.int32)
    vv = None if vals is None else _dev(vals, torch.float32)
    results = []
    for _ in range(2):
        rpt = torch.full((n + 1,), -7, dtype=torch.int32, device="cuda")
        cit = torch.full((max(nnz, 1),), -7, dtype=torch.int32, device="cuda")
        vvt = None if vals is None else torch.full((max(nnz, 1),), -7.0, device="cuda")
        ws_bytes = int(lib.egnn_csr_transpose_ws_bytes(n, nnz))
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _cabi.check(lib.egnn_csr_transpose(_cabi.ptr(rp), _cabi.ptr(ci) if nnz else None, _cabi.ptr(vv), n, nnz,
                                           _cabi.ptr(rpt), _cabi.ptr(cit) if nnz else None, _cabi.ptr(vvt),
                                           _cabi.ptr(ws), ws_bytes, _cabi.current_stream()), "egnn_csr_transpose")
        torch.cuda.synchronize()
        results.append((rpt.cpu().numpy(), cit[:nnz].cpu().numpy(),
                        None if vvt is None else vvt[:nnz].cpu().numpy()))
    return results


def transpose_cases():
    rng = np.random.default_rng(11)

    def rand_csr(n, nnz, dup=False, shuffle=False, weighted=False, empty_rows=(), empty_cols=()):
        r, c = rng.integers(0, n, nnz), rng.integers(0, n, nnz)
        keep = ~np.isin(r, empty_rows) & ~np.isin(c, empty_cols)
        r, c = np.append(r[keep], 1), np.append(c[keep], n - 1)      # the last column is used
        if dup:
            r, c = np.concatenate([r, r[:50]]), np.concatenate([c, c[:50]])
        else:
            key = np.unique(r.astype(np.int64) * n + c)
            r, c = key // n, key % n
        order = np.lexsort((c, r))
        r, c = r[order], c[order]
        if shuffle:                                  # columns unsorted inside every row
            perm = np.lexsort((rng.random(r.size), r))
            r, c = r[perm], c[perm]
        rowptr = np.zeros(n + 1, np.int64)
        np.add.at(rowptr, r + 1, 1)
        rowptr = np.cumsum(rowptr)
        vals = rng.uniform(-2, 2, c.size).astype(np.float32) if weighted else None
        return rowptr.astype(np.int32), c.astype(np.int32), vals, n

    yield "nnz0", (np.zeros(6, np.int32), np.zeros(0, np.int32), None, 5)
    yield "n1", (np.array([0, 1], np.int32), np.array([0], np.int32), np.array([2.5], np.float32), 1)
    yield "n1_empty", (np.array([0, 0], np.int32), np.zeros(0, np.int32), None, 1)
    yield "n65536", rand_csr(65536, 300_000, weighted=True)
    yield "n65537", rand_csr(65537, 300_000)
    yield "empty_rows_cols", rand_csr(4000, 30_000, weighted=True, empty_rows=np.arange(0, 4000, 7),
                                      empty_cols=np.arange(3, 4000, 5))
    yield "duplicates", rand_csr(3000, 20_000, dup=True, weighted=True)
    yield "unsorted", rand_csr(3000, 20_000, shuffle=True, weighted=True)
    # one column with 70 001 entries (one per row of a 100 000-node graph), plus a few others
    n = 100_000
    r = np.concatenate([np.arange(70_001), rng.integers(0, n, 5000)])
    c = np.concatenate([np.full(70_001, 4), rng.integers(0, n, 5000)])
    key = np.unique(r.astype(np.int64) * n + c)
    r, c = key // n, key % n
    rowptr = np.cumsum(np.concatenate([[0], np.bincount(r, minlength=n)]))
    yield "long_column", (rowptr.astype(np.int32), c.astype(np.int32), rng.uniform(0.5, 2, c.size).astype(np.float32), n)


def transpose_reference(rowptr, colidx, vals, n):
    """Stable counting transpose in numpy: entries of a column keep their CSR order."""
    rows = np.repeat(np.arange(n), np.diff(rowptr))
    order = np.argsort(colidx, kind="stable")
    rp = np.concatenate([[0], np.cumsum(np.bincount(colidx, minlength=n))]).astype(np.int32)
    return rp, rows[order].astype(np.int32), None if vals is None else vals[order]


@pytest.mark.parametrize("tag,case", list(transpose_cases()), ids=[t for t, _ in transpose_cases()])
def test_csr_transpose(tag, case):
    rowptr, colidx, vals, n = case
    (rp1, ci1, vv1), (rp2, ci2, vv2) = gpu_transpose(rowptr, colidx, vals, n)
    assert np.array_equal(rp1, rp2) and np.array_equal(ci1, ci2)
    assert vals is None or np.array_equal(vv1.view(np.int32), vv2.view(np.int32))
    rp, ci, vv = transpose_reference(rowptr, colidx, vals, n)
    assert np.array_equal(rp1, rp) and np.array_equal(ci1, ci)
    if vals is not None:
        assert np.array_equal(vv1.view(np.int32), vv.view(np.int32))
    rows = np.repeat(np.arange(n), np.diff(rp1))
    assert np.all((np.diff(ci1) >= 0) | (np.diff(rows) > 0)), "a transposed row is not sorted"
    if tag not in ("duplicates",):                  # scipy agrees where the input is canonical or merely unsorted
        m = sp.csr_matrix((np.ones(colidx.size, np.float32) if vals is None else vals, colidx, rowptr), shape=(n, n))
        t = m.T.tocsr()
        t.sort_indices()
        assert np.array_equal(t.indptr, rp1) and np.array_equal(t.indices, ci1)
        if vals is not None:
            assert np.array_equal(t.data.view(np.int32), vv1.view(np.int32))


def _l1_data(n_vec, f, seed):
    rng = np.random.default_rng(seed)
    c = rng.standard_normal((n_vec, f)).astype(np.float32)
    c[::7] = 0.0                                  # zero rows
    c[rng.random(c.shape) < 0.1] = 0.0            # exact zeros inside rows: sign(0) = 0
    c[3::11] *= 1e-6
    return c, rng.standard_normal((n_vec, f)).astype(np.float32), rng.standard_normal((n_vec, f)).astype(np.float32)


@pytest.mark.parametrize("f", [1, 31, 32, 33, 130])
def test_l1_normalize_and_backward(f):
    lib = _cabi.load()
    n_vec = 1500
    c, hbar, base = _l1_data(n_vec, f, f)
    c64, g64, b64 = c.astype(np.float64), hbar.astype(np.float64), base.astype(np.float64)
    r = np.abs(c64).sum(axis=1, keepdims=True) + 1e-8
    h_ref = c64 / r
    dot = (g64 * h_ref).sum(axis=1, keepdims=True)
    grad_ref = (g64 - np.sign(c64) * dot) / r
    scale = (np.abs(g64) + np.abs(dot)) / r
    st = _cabi.current_stream()
    cd, gd = _dev(c, torch.float32), _dev(hbar, torch.float32)
    hs = []
    for _ in range(2):
        h = torch.full_like(cd, np.nan)
        _cabi.check(lib.egnn_l1_normalize(_cabi.ptr(cd), _cabi.ptr(h), n_vec, f, st), "egnn_l1_normalize")
        hs.append(h.cpu().numpy())
    assert np.array_equal(hs[0].view(np.int32), hs[1].view(np.int32))
    assert np.all(np.abs(hs[0] - h_ref) <= 1e-5 * np.abs(h_ref))
    assert np.all(hs[0][::7] == 0)
    for mode in ("null", "separate", "aliased"):
        outs = []
        for _ in range(2):
            bd = _dev(base, torch.float32)
            out = bd if mode == "aliased" else torch.full_like(cd, np.nan)
            cin = None if mode == "null" else bd
            _cabi.check(lib.egnn_l1_normalize_backward(_cabi.ptr(cd), _cabi.ptr(gd), _cabi.ptr(cin), _cabi.ptr(out),
                                                       n_vec, f, st), "egnn_l1_normalize_backward")
            outs.append(out.cpu().numpy())
        assert np.array_equal(outs[0].view(np.int32), outs[1].view(np.int32)), mode
        want = grad_ref + (0.0 if mode == "null" else b64)
        bound = 1e-5 * (scale + (0.0 if mode == "null" else np.abs(b64)))
        bad = np.abs(outs[0] - want) > bound
        assert not bad.any(), f"F={f} {mode}: {int(bad.sum())} elements off, worst at {np.argwhere(bad)[0]}"
        np.testing.assert_allclose(outs[0][::7], want[::7], rtol=1e-6)       # zero rows: Hbar / 1e-8


@pytest.mark.parametrize("f", [1, 7, 130])
@pytest.mark.parametrize("k", [0, 3, 20])
@pytest.mark.parametrize("n_scales", [1, 8])
@pytest.mark.parametrize("n", [1, 295, 296, 297, 10007])
def test_cheb_coeff_grad(n, n_scales, k, f):
    """G[s, k] = <Cbar[:, s, :], T_k> in float64; n around the 296 CTAs of the reduction."""
    lib = _cabi.load()
    rng = np.random.default_rng(n + 7 * f + k)
    cbar = rng.standard_normal((n, n_scales, f)).astype(np.float32)
    t_all = rng.standard_normal((k + 1, n, f)).astype(np.float32)
    terms = np.einsum("nsf,knf->skn", cbar.astype(np.float64), t_all.astype(np.float64))
    want = terms.sum(axis=2)
    size = np.einsum("nsf,knf->sk", np.abs(cbar).astype(np.float64), np.abs(t_all).astype(np.float64))
    cd, td = _dev(cbar, torch.float32), _dev(t_all, torch.float32)
    ws_bytes = int(lib.egnn_cheb_coeff_grad_ws_bytes(k, n_scales))
    got = []
    for _ in range(2):
        g = torch.full((n_scales, k + 1), np.nan, dtype=torch.float64, device="cuda")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        _cabi.check(lib.egnn_cheb_coeff_grad(_cabi.ptr(cd), _cabi.ptr(td), n, f, k, n_scales, _cabi.ptr(g),
                                             _cabi.ptr(ws), ws_bytes, _cabi.current_stream()), "egnn_cheb_coeff_grad")
        got.append(g.cpu().numpy())
    assert np.array_equal(got[0].view(np.int64), got[1].view(np.int64))
    assert np.all(np.abs(got[0] - want) <= 1e-13 * size + 1e-300)
