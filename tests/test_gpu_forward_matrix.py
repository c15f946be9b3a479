"""Every forward instantiation of the order kernels against the float64 oracle, element-wise.

One call of ``egnn_cheb_wavelet`` on one GPU launches one of four kernel families for its orders:
the wide kernel (``csrc/wide.cuh``, F >= 8) keyed by ``<NZ_LOG2, HAS_VALS, ALIGNED, PEER, DYN,
ADJ>``, the generic kernel (``csrc/cheb.cuh``, F < 8) keyed by ``<VEC, U, HAS_VALS, PRESCALED,
ADJ>``, and at F = 1 the SELL step kernel (``csrc/sell_step.cuh``, ``<PEER, PATCH>``) or the
plan-free blocked kernel (``csrc/blocked.cuh``, ``<HAS_VALS>``).

* ``TABLE``: one row per (graph, F) that reaches a given instantiation.  Every case
  (``run_case``) makes four checks:
  - parts (``return_parts=True``): every T_k and every S_j against ``oracle.wats_oracle``,
    norm-wise <= 1e-5 (1e-4 above 16 orders) and element-wise ratio <= 1 at the 5e-2 floor
    (the ratio at the 1e-3 floor is printed beside it);
  - production (``return_parts=False, normalize=True``: the L1 normalisation fused into the
    last order): H against ``S / (sum |S| + 1e-8)`` in float64 of the parts pass's S, per
    element ``|dH| <= (F + 4) 2^-24 |H64|`` with equal signs - a float32 sum of F non-negative
    terms, one addition, one division and one product;
  - ``normalize=False`` gives the parts pass's S bit for bit (same path: ``_use_sell`` pinned);
  - a second production pass gives the same bits.
* ``test_every_reachable_forward_instantiation_runs``: each row launches exactly the
  instantiation it names (``torch.profiler``), and the table launches all 46 reachable ones.
* Edges on every family where they apply: ``lambda_max`` 1.7 and 3.3 on a graph with isolated
  and self-loop-only nodes, K in {0, 1, 2, 17, 20}, eight scales, 64 edge flips (and 65
  refused), flips on the diagonal, hub rows on the static wide schedule, long rows sharing a
  warp of the generic kernel, column-block tails of the narrow paths, the empty graph.
"""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import _cabi
from oracle import wats_oracle as orc
from test_gpu_adjoint_matrix import (HUB_ROWS, LAST_IN, LONG_ROWS, LOOP_ONLY, LOOPS, SCALES, _pattern,
                                     _profiled_kernels, graph, kernel_keys)
from test_gpu_parity import check_parts

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
H_WORST = {}                  # tag -> worst |dH| / ((F + 4) 2^-24 |H64|) of the production pass


def tol_for(k):
    return 1e-4 if k > 16 else 1e-5


def signal(n, f, seed):
    return np.random.default_rng(seed).standard_normal((n, f)).astype(np.float32)


def run_case(tag, adj, g, f, k, n_scales, lam, use_sell, x_np, deltas=None, ref_adj=None):
    """The four checks of one case; ``x_np`` None: the graph's default signal (F = 1)."""
    n = adj.shape[0]
    sc = SCALES[:n_scales]
    kw = dict(k=k, s=sc, X0=None if x_np is None else torch.from_numpy(x_np), lambda_max=lam, deltas=deltas,
              _use_sell=use_sell)
    res = egnn.graph_wavelet_features(g, return_parts=True, **kw)
    p = orc.wavelet_parts(adj if ref_adj is None else ref_adj, k=k, s=sc, x0=x_np, lambda_max=lam)
    check_parts(res, p["T"], p["S"], p["H"], tag, tol=tol_for(k))

    # production: the fused normalisation against float64 of the same S
    h = egnn.graph_wavelet_features(g, **kw)
    comb = res.combined.cpu().numpy().astype(np.float64)
    h64 = comb / (np.abs(comb).sum(axis=2, keepdims=True) + 1e-8)
    hg = h.cpu().numpy().astype(np.float64).reshape(n, n_scales, f)
    bound = (f + 4) * EPS32 * np.abs(h64)
    diff = np.abs(hg - h64)
    bad = diff > bound
    H_WORST[tag] = float((diff / np.where(bound > 0, bound, 1.0)).max()) if n else 0.0
    print(f"[{tag}] fused H: worst |dH| / ((F+4) 2^-24 |H64|) = {H_WORST[tag]:.3f}")
    assert not bad.any(), f"{tag}: fused H off at {np.argwhere(bad)[0]}: {hg[bad][0]!r} vs {h64[bad][0]!r}"
    assert np.array_equal(np.sign(hg), np.sign(h64)), f"{tag}: fused H has a wrong sign"

    # the un-normalised production pass is the parts pass's S, bit for bit
    plain = egnn.graph_wavelet_features(g, normalize=False, **kw)
    assert torch.equal(plain, res.combined.reshape(n, -1)), f"{tag}: S differs from the parts pass"
    assert torch.equal(egnn.graph_wavelet_features(g, **kw), h), f"{tag}: production pass not repeatable"
    return res


# ---- the case table ----------------------------------------------------------------------------
# (graph, F, K, S, lambda_max, _use_sell, flips, instantiation launched by every order).
# wide<NZ_LOG2, HAS_VALS, ALIGNED, PEER, DYN, ADJ>: ldy = ceil4(F), NZ_LOG2 = 5 - ceil(log2(ldy / 4))
# (0 from F = 65 up, ring_config); ALIGNED = F % 4 == 0; DYN when one feature tile covers the row
# (F <= 128) and nnz < 64 n: the sparse graphs (~8 entries per row).  The dense graphs ("dense_*":
# ~96 per row, "dense_hubs_*": ~72 per row plus three 2100-entry hub rows) and every F > 128 take
# the static schedule.  order<VEC, U, HAS_VALS, PRESCALED, ADJ> (choose_config): VEC = 4 for F = 4,
# PRESCALED for F <= 4.  At F = 1, _use_sell True forces the SELL plan (binary adjacency only;
# PATCH when edge flips come with it), "blocked" the plan-free blocked kernel, False the generic one.
TABLE = [
    ("sparse_bin", 8, 3, 1, 2.0, None, False, "wide<4,0,1,0,1,0>"),
    ("sparse_w", 8, 4, 2, 1.7, None, False, "wide<4,1,1,0,1,0>"),
    ("dense_bin", 8, 3, 3, 2.0, None, False, "wide<4,0,1,0,0,0>"),
    ("dense_hubs_w", 8, 3, 2, 1.7, None, False, "wide<4,1,1,0,0,0>"),
    ("sparse_long_bin", 12, 3, 2, 2.0, None, False, "wide<3,0,1,0,1,0>"),
    ("out_star_w", 12, 3, 1, 2.0, None, False, "wide<3,1,1,0,1,0>"),
    ("dense_hubs_bin", 12, 2, 1, 1.7, None, False, "wide<3,0,1,0,0,0>"),
    ("dense_hubs_w", 12, 3, 2, 2.0, None, False, "wide<3,1,1,0,0,0>"),
    ("sparse_bin", 10, 4, 1, 1.7, None, False, "wide<3,0,0,0,1,0>"),
    ("stars_w", 10, 3, 2, 2.0, None, False, "wide<3,1,0,0,1,0>"),
    ("dense_bin", 10, 3, 2, 2.0, None, False, "wide<3,0,0,0,0,0>"),
    ("dense_w", 10, 2, 1, 1.7, None, False, "wide<3,1,0,0,0,0>"),
    ("sparse_bin", 24, 2, 3, 2.0, None, False, "wide<2,0,1,0,1,0>"),
    ("sparse_long_w", 24, 3, 2, 2.0, None, False, "wide<2,1,1,0,1,0>"),
    ("dense_bin", 24, 3, 1, 2.0, None, False, "wide<2,0,1,0,0,0>"),
    ("dense_hubs_w", 24, 3, 3, 1.7, None, False, "wide<2,1,1,0,0,0>"),
    ("sparse_long_bin", 19, 3, 1, 2.0, None, False, "wide<2,0,0,0,1,0>"),
    ("out_star_w", 19, 4, 2, 1.7, None, False, "wide<2,1,0,0,1,0>"),
    ("dense_hubs_bin", 19, 2, 2, 2.0, None, False, "wide<2,0,0,0,0,0>"),
    ("dense_w", 19, 3, 1, 2.0, None, False, "wide<2,1,0,0,0,0>"),
    ("sparse_bin", 48, 3, 2, 1.7, None, False, "wide<1,0,1,0,1,0>"),
    ("in_star_w", 48, 3, 1, 2.0, None, False, "wide<1,1,1,0,1,0>"),
    ("dense_hubs_bin", 48, 3, 1, 2.0, None, False, "wide<1,0,1,0,0,0>"),
    ("dense_hubs_w", 48, 2, 2, 2.0, None, False, "wide<1,1,1,0,0,0>"),
    ("sparse_bin", 37, 3, 1, 2.0, None, False, "wide<1,0,0,0,1,0>"),
    ("sparse_w", 37, 3, 2, 1.7, None, False, "wide<1,1,0,0,1,0>"),
    ("dense_bin", 37, 2, 1, 2.0, None, False, "wide<1,0,0,0,0,0>"),
    ("dense_hubs_w", 37, 3, 2, 2.0, None, False, "wide<1,1,0,0,0,0>"),
    ("sparse_bin", 128, 3, 1, 2.0, None, False, "wide<0,0,1,0,1,0>"),
    ("out_star_w", 128, 3, 2, 2.0, None, False, "wide<0,1,1,0,1,0>"),
    ("dense_bin", 128, 2, 2, 1.7, None, False, "wide<0,0,1,0,0,0>"),
    ("sparse_w", 260, 3, 1, 2.0, None, False, "wide<0,1,1,0,0,0>"),
    ("sparse_long_bin", 99, 2, 2, 2.0, None, False, "wide<0,0,0,0,1,0>"),
    ("in_star_w", 99, 3, 1, 1.7, None, False, "wide<0,1,0,0,1,0>"),
    ("sparse_bin", 130, 3, 2, 2.0, None, False, "wide<0,0,0,0,0,0>"),
    ("dense_hubs_w", 99, 2, 2, 2.0, None, False, "wide<0,1,0,0,0,0>"),
    ("sparse_long_bin", 1, 3, 2, 2.0, False, False, "order<1,1,0,1,0>"),
    ("sparse_bin", 2, 4, 1, 1.7, False, False, "order<1,1,0,1,0>"),
    ("sparse_long_w", 3, 3, 2, 2.0, False, False, "order<1,1,1,1,0>"),
    ("dense_w", 1, 3, 1, 1.7, False, False, "order<1,1,1,1,0>"),
    ("dense_bin", 4, 3, 2, 2.0, False, False, "order<4,1,0,1,0>"),
    ("sparse_long_w", 4, 4, 1, 1.7, False, False, "order<4,1,1,1,0>"),
    ("sparse_long_bin", 6, 3, 2, 2.0, False, False, "order<1,1,0,0,0>"),
    ("dense_hubs_w", 5, 3, 1, 2.0, False, False, "order<1,1,1,0,0>"),
    ("in_star_w", 7, 2, 2, 1.7, False, False, "order<1,1,1,0,0>"),
    ("sparse_long_bin", 1, 3, 2, 2.0, True, False, "sell_step<0,0>"),
    ("dense_hubs_bin", 1, 4, 1, 1.7, True, True, "sell_step<0,1>"),
    ("sparse_long_bin", 1, 3, 2, 1.7, "blocked", False, "blocked_spmv<0>"),
    ("dense_hubs_w", 1, 4, 3, 2.0, "blocked", True, "blocked_spmv<1>"),
]

# The 46 instantiations egnn_cheb_wavelet can launch on one GPU.  Compiled as well but unreachable
# there (checked against `cuobjdump -symbols` of the library): wide<4,*,0,0,*,0> (NZ_LOG2 = 4 means
# F = 8, a multiple of 4), the PEER instantiations wide<*,*,*,1,0,0> and sell_step<1,*> (world > 1,
# tests/test_gpu_peer.py), order<4,1,*,0,0> (VEC = 4 only for F % 4 == 0, which is F = 4, pre-scaled,
# or F >= 8, wide) and order<1,4,*,*,0> (U = 4 only for F > 32, which runs the wide kernel).
REACHABLE = {f"wide<{nz},{hv},{al},0,{dyn},0>" for nz in range(5) for hv in (0, 1) for al in (0, 1)
             for dyn in (0, 1) if nz < 4 or al} | {
    "order<1,1,0,1,0>", "order<1,1,1,1,0>", "order<4,1,0,1,0>", "order<4,1,1,1,0>",
    "order<1,1,0,0,0>", "order<1,1,1,0,0>",
    "sell_step<0,0>", "sell_step<0,1>", "blocked_spmv<0>", "blocked_spmv<1>",
}


def case_id(c):
    return f"{c[0]}-F{c[1]}-K{c[2]}-S{c[3]}-{c[7]}"


def flips64(adj):
    """64 directed flips touching 128 distinct nodes: LAST_IN's only in-edge removed (it becomes
    isolated), one stored entry of the first hub row removed and entries added to the other hub
    rows (graphs with HUB_ROWS), the rest random additions (values 1.0 / 0.75 / 1.5) and removals
    between distinct nodes.  Returns (deltas, perturbed adjacency)."""
    a = adj.tocsr()
    n = a.shape[0]
    rows, cols, vals = [], [], []
    used = {80, LAST_IN}
    rng = np.random.default_rng(17)

    def add(i, j, v):
        rows.append(int(i)); cols.append(int(j)); vals.append(float(v)); used.update((int(i), int(j)))

    assert a[80, LAST_IN] != 0 and a[:, LAST_IN].nnz == 1
    add(80, LAST_IN, -a[80, LAST_IN])
    hubs = [h for h in HUB_ROWS if a.indptr[h + 1] - a.indptr[h] >= 2048]
    for t, h in enumerate(hubs):
        stored = set(a.indices[a.indptr[h]:a.indptr[h + 1]].tolist())
        if t == 0:
            c = next(int(j) for j in rng.permutation(sorted(stored)) if j not in used and j != h)
            add(h, c, -a[h, c])
        else:
            c = next(int(j) for j in rng.permutation(np.arange(100, n)) if j not in stored and j not in used)
            add(h, c, 0.75 if t == 1 else 1.0)
    pool = [int(i) for i in rng.permutation(np.arange(100, n)) if int(i) not in used]
    while len(rows) < 64:
        i, j = pool.pop(), pool.pop()
        v = float(a[i, j])
        add(i, j, -v if v != 0 else (1.0, 0.75, 1.5)[len(rows) % 3])
    assert len(set(rows) | set(cols)) == 128
    d = sp.csr_matrix((np.array(vals, np.float32), (rows, cols)), shape=a.shape)
    pert = (a + d).tocsr()
    pert.eliminate_zeros()
    assert pert[:, LAST_IN].nnz == 0
    assert any(v < 0 for v in vals) and any(v > 0 for v in vals) and 0.75 in vals
    return (rows, cols, vals), pert


@pytest.mark.parametrize("case", TABLE, ids=[case_id(c) for c in TABLE])
def test_forward_matrix_vs_float64(case):
    name, f, k, n_scales, lam, use_sell, flips, _kernel = case
    adj, g = graph(name)
    deltas, pert = flips64(adj) if flips else (None, None)
    x = None if (f == 1 and use_sell in (True, "blocked")) else signal(adj.shape[0], f, f * 31 + k)
    run_case(f"{case_id(case)} lam={lam}", adj, g, f, k, n_scales, lam, use_sell, x, deltas, pert)


# ---- which kernels run -------------------------------------------------------------------------
def test_every_reachable_forward_instantiation_runs():
    probe = _profiled_kernels(lambda: torch.ones(1 << 16, device="cuda").mul_(2.0))
    if not probe:
        pytest.skip("torch.profiler records no CUDA kernel here (CUPTI unavailable): coverage not measurable")
    assert kernel_keys(["void egnn::cheb_wide_kernel<(int)3, (bool)1, (bool)0, (bool)0, (bool)1, (bool)0>("
                        "egnn::WideParams)", "void egnn::sell_step_kernel<false, true>(egnn::SellStepParams)",
                        "void egnn::cheb_order_kernel<4, 1, true, true, true>(egnn::OrderParams)"], adj=False) == \
        {"wide<3,1,0,0,1,0>", "sell_step<0,1>"}
    launched = set()
    for case in TABLE:
        name, f, k, n_scales, lam, use_sell, flips, kernel = case
        adj, g = graph(name)
        deltas = flips64(adj)[0] if flips else None
        x = None if (f == 1 and use_sell in (True, "blocked")) else torch.from_numpy(signal(adj.shape[0], f, 1))
        kw = dict(k=k, s=SCALES[:n_scales], X0=x, lambda_max=lam, deltas=deltas, _use_sell=use_sell)

        def passes():
            egnn.graph_wavelet_features(g, return_parts=True, **kw)
            egnn.graph_wavelet_features(g, **kw)
            egnn.graph_wavelet_features(g, normalize=False, **kw)
        got = kernel_keys(_profiled_kernels(passes), adj=False)
        assert got == {kernel}, f"{case_id(case)}: launched {sorted(got)}, the table says {kernel}"
        launched |= got
    assert len(REACHABLE) == 46
    print(f"\n[coverage] {len(launched & REACHABLE)} of {len(REACHABLE)} reachable forward instantiations launched")
    assert launched == REACHABLE, f"missing {sorted(REACHABLE - launched)}, unexpected {sorted(launched - REACHABLE)}"


# ---- edges -------------------------------------------------------------------------------------
# one representative per family: (graph, F, _use_sell)
FAMILIES = {
    "generic F=1": ("sparse_long_w", 1, False),
    "generic F=4": ("sparse_long_bin", 4, None),
    "wide DYN": ("sparse_long_w", 8, None),
    "wide static": ("dense_hubs_w", 48, None),
    "SELL": ("sparse_long_bin", 1, True),
    "blocked": ("sparse_long_w", 1, "blocked"),
}

LAM_FAMILIES = [("sparse_long_bin", 1, False), ("sparse_long_w", 3, None), ("sparse_long_w", 6, None),
                ("sparse_long_bin", 12, None), ("dense_hubs_w", 24, None), ("dense_hubs_bin", 130, None),
                ("sparse_long_bin", 1, True), ("sparse_long_bin", 1, "blocked"), ("sparse_long_w", 1, "blocked")]


@pytest.mark.parametrize("lam", [1.7, 3.3])
@pytest.mark.parametrize("name,f,use_sell", LAM_FAMILIES, ids=[f"{a}-F{b}-{c}" for a, b, c in LAM_FAMILIES])
def test_lambda_max_every_family(name, f, use_sell, lam):
    """lambda_max != 2: theta = 2 / lambda_max - 1 != 0 on every row, with isolated nodes
    (theta = -1) and self-loop-only nodes (isolated too, but log1p(1) in the default signal)."""
    adj, g = graph(name)
    iso = np.asarray((adj - sp.diags(adj.diagonal())).sum(axis=0)).ravel() == 0
    assert iso[list(LOOP_ONLY)].all() and all(adj[i, i] != 0 for i in LOOP_ONLY)
    run_case(f"{name} F={f} sell={use_sell} lam={lam}", adj, g, f, 3, 2, lam, use_sell,
             signal(adj.shape[0], f, int(lam * 10) + f))


@pytest.mark.parametrize("k", [0, 1, 2, 17, 20])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_order_count_edges(family, k):
    """K = 0 (order 0 alone), K = 1 (the first order is the last one), K = 17 (the step kernel's
    second 16-order launch holds one order), K = 20."""
    name, f, use_sell = FAMILIES[family]
    adj, g = graph(name)
    run_case(f"{family} K={k}", adj, g, f, k, 2, 2.0, use_sell, signal(adj.shape[0], f, 5 * f + k))


@pytest.mark.parametrize("family", list(FAMILIES))
def test_eight_scales(family):
    name, f, use_sell = FAMILIES[family]
    adj, g = graph(name)
    run_case(f"{family} S=8", adj, g, f, 3, 8, 2.0, use_sell, signal(adj.shape[0], f, f + 8))


FLIP_CASES = [("sparse_long_bin", 1, False, True), ("sparse_long_w", 1, False, False),
              ("sparse_long_w", 6, None, False), ("sparse_long_bin", 3, None, False),
              ("sparse_long_w", 12, None, False), ("dense_hubs_w", 24, None, False),
              ("dense_hubs_bin", 8, None, False), ("dense_hubs_bin", 1, True, True),
              ("sparse_long_bin", 1, True, False), ("sparse_long_bin", 1, "blocked", True),
              ("dense_hubs_w", 1, "blocked", False)]


@pytest.mark.parametrize("name,f,use_sell,default", FLIP_CASES,
                         ids=[f"{a}-F{b}-{c}-{'default' if d else 'caller'}" for a, b, c, d in FLIP_CASES])
def test_64_flips(name, f, use_sell, default):
    """EGNN_MAX_DELTA flips, 128 distinct touched nodes (patch_nodes_kernel and the step kernel's
    PATCH prologue use every thread), against the oracle on the perturbed matrix."""
    adj, g = graph(name)
    deltas, pert = flips64(adj)
    x = None if default else signal(adj.shape[0], f, f + 64)
    run_case(f"{name} F={f} sell={use_sell} 64 flips", adj, g, f, 3, 2, 1.7 if f % 2 else 2.0, use_sell, x,
             deltas, pert)


@pytest.mark.parametrize("use_sell", [False, True, "blocked"])
def test_65_flips_refused(use_sell):
    adj, g = graph("sparse_long_bin")
    rows, cols, vals = (list(v) for v in flips64(adj)[0])
    rows.append(90); cols.append(91); vals.append(1.0)
    x8 = torch.ones(adj.shape[0], 8)
    before = (egnn.graph_wavelet_features(g, _use_sell=use_sell), egnn.graph_wavelet_features(g, X0=x8))
    with pytest.raises(egnn.EgnnError):
        egnn.graph_wavelet_features(g, deltas=(rows, cols, vals), _use_sell=use_sell)
    with pytest.raises(egnn.EgnnError):
        egnn.graph_wavelet_features(g, X0=x8, deltas=(rows, cols, vals))
    # nothing of the refused flips stays behind on the graph
    assert torch.equal(egnn.graph_wavelet_features(g, _use_sell=use_sell), before[0])
    assert torch.equal(egnn.graph_wavelet_features(g, X0=x8), before[1])


DIAG_CASES = [("sparse_long_bin", 1, False, True), ("sparse_long_w", 4, None, False),
              ("sparse_long_bin", 12, None, False), ("dense_hubs_w", 24, None, False),
              ("sparse_long_bin", 1, True, True), ("sparse_long_w", 1, "blocked", True)]


@pytest.mark.parametrize("name,f,use_sell,default", DIAG_CASES,
                         ids=[f"{a}-F{b}-{c}" for a, b, c, _ in DIAG_CASES])
def test_flips_on_the_diagonal(name, f, use_sell, default):
    """row == col: a self loop added to a node without one, a stored one removed (LOOPS), and one
    added to a self-loop-only node.  Self loops are not part of L, but they count in the row sum
    of the default signal."""
    adj, g = graph(name)
    a = adj.tocsr()
    fresh = next(i for i in range(100, a.shape[0]) if a[i, i] == 0)
    rows = [fresh, LOOPS[0], LOOP_ONLY[0], 300]
    cols = [fresh, LOOPS[0], LOOP_ONLY[0], 301 if a[300, 301] == 0 else 302]
    vals = [1.0, -float(a[LOOPS[0], LOOPS[0]]), 0.5, 1.0]
    pert = (a + sp.csr_matrix((np.array(vals, np.float32), (rows, cols)), shape=a.shape)).tocsr()
    pert.eliminate_zeros()
    x = None if default else signal(a.shape[0], f, 77 + f)
    run_case(f"{name} F={f} sell={use_sell} diagonal flips", adj, g, f, 3, 2, 2.0, use_sell, x,
             (rows, cols, vals), pert)


@pytest.mark.parametrize("f", [8, 12, 24, 48])
def test_hub_rows_on_the_static_wide_schedule(f):
    """Phase A (one CTA per row of >= 2048 entries) with NZ_LOG2 > 0, static schedule."""
    adj, g = graph("dense_hubs_bin")
    n = adj.shape[0]
    assert adj.nnz >= 64 * n
    assert int(g.row_order()[n].item()) == len(HUB_ROWS)
    run_case(f"dense_hubs_bin F={f} hubs", adj, g, f, 3, 2, 2.0, None, signal(n, f, 900 + f))


@pytest.mark.parametrize("name", ["sparse_long_bin", "sparse_long_w"])
@pytest.mark.parametrize("f", [1, 2, 3, 4])
def test_long_rows_in_one_warp(name, f):
    """Eight consecutive rows in one warp of the generic kernel, each longer than NZ * 4 * 8
    entries (NZ = 4 here: ~9 entries per row on average, choose_config), so every lane group of
    the warp defers its row to the whole warp, one after another."""
    adj, g = graph(name)
    deg = np.diff(adj.indptr)
    assert LONG_ROWS[0] % 8 == 0 and (deg[list(LONG_ROWS)] > 4 * 4 * 8).all()
    run_case(f"{name} F={f} long rows", adj, g, f, 3, 2, 2.0, False, signal(adj.shape[0], f, 40 + f))


# ---- column-block tails of the narrow paths ----------------------------------------------------
def sell_geometry(n):
    """(n_blocks, col_block) of the SELL plan; the blocked kernel uses the same geometry
    (narrow_geometry in egnn_cabi.cu)."""
    nb, cb, lmax = C.c_int32(), C.c_int32(), C.c_int32()
    _cabi.check(_cabi.load().egnn_sell_geometry(n, 0, C.byref(nb), C.byref(cb), C.byref(lmax)), "egnn_sell_geometry")
    return nb.value, cb.value


def tail_sizes():
    """n whose last column block holds 1, 2 or 3 columns past a multiple of 4 (two blocks, and
    three blocks with 1), and n = 1: the last block then holds a single column.  For n >= 2 the
    block width rounded up to 32 leaves no last block of one column below ~7.5e7 nodes."""
    out = [1]
    for blocks, rem in ((2, 1), (2, 2), (2, 3), (3, 1)):
        n = 49153 if blocks == 2 else 98305
        while True:
            nb, cb = sell_geometry(n)
            if nb == blocks and (n - (nb - 1) * cb) % 4 == rem:
                break
            n += 1
        out.append(n)
    return out


_TAILS = {}


def tail_graph(n, weighted):
    key = (n, weighted)
    if key not in _TAILS:
        if n == 1:
            adj = sp.csr_matrix(np.ones((1, 1), np.float32) * (1.5 if weighted else 1.0))
        else:
            rng = np.random.default_rng(n + weighted)
            a = _pattern(rng, n, 8, directed=weighted).tocsr()
            a.data[:] = 1.0
            if weighted:
                a.data = rng.uniform(0.5, 2.0, a.nnz).astype(np.float32)
            a.sort_indices()
            adj = a
        _TAILS[key] = (adj, egnn.as_graph(adj))
    return _TAILS[key]


@pytest.mark.parametrize("path,weighted", [(True, False), ("blocked", False), ("blocked", True)],
                         ids=["sell-bin", "blocked-bin", "blocked-w"])
def test_column_block_tails(path, weighted):
    sizes = tail_sizes()
    for n in sizes:
        nb, cb = sell_geometry(n)
        adj, g = tail_graph(n, weighted)
        tag = f"{'sell' if path is True else path} {'w' if weighted else 'bin'} n={n} ({nb} blocks of {cb}, " \
              f"last holds {n - (nb - 1) * cb})"
        run_case(tag, adj, g, 1, 3, 2, 2.0, path, signal(n, 1, n))
        run_case(tag + " default signal", adj, g, 1, 4, 1, 1.7, path, None)


@pytest.mark.parametrize("f", [1, 4, 8, 130])
def test_empty_graph_closed_form(f):
    """No edges, lambda_max = 2: M = -I, so T_k = (-1)^k X0 exactly."""
    adj, g = graph("empty")
    x = signal(adj.shape[0], f, f)
    res = run_case(f"empty F={f}", adj, g, f, 3, 2, 2.0, False, x)
    for i, t in enumerate(res.orders):
        assert np.array_equal(t.cpu().numpy(), (-1) ** i * x), f"T_{i}"
