"""Gradient of the wavelet pass w.r.t. the adjacency and ``lambda_max`` on the GPU
(egnn_cheb_adjoint_all + egnn_adj_grad_degree / _pairs / _dense, DESIGN.md section 11).

* Golden graphs: the dense gradient of a dense ``[N, N]`` leaf and ``dLoss/dlambda_max`` against
  the float64 ``tests/adjacency_reference.adjacency_vjp``, K = 0, 1, 3, 4, 6, F = 1 (SELL and
  generic kernels), 3, 8, 37 and 130, S = 1 and 3: norm-wise error <= 1e-5 and element-wise ratio
  <= 1 at the 5e-2 floor (DESIGN sections 2 and 10), the ratio at the 1e-3 floor printed beside them.
  F = 1 runs without the normalisation (see the top of test_gpu_backward.py).
* A sparse COO adjacency: the gradient on its value leaf, with a duplicate edge and an explicit zero.
* A CPU float64 leaf, a 0-d ``lambda_max``, unchanged signal / scale gradients and features, and
  bitwise-repeatable backward passes.
* Full size against float64 sums over the explicit operator built with scipy: arxiv directed
  weighted F = 16 on every stored entry, Reddit F = 1 default signal on sampled rows (hub rows
  included), and a 20,000-node graph F = 1 dense on sampled rows and columns.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import synth
from oracle import wats_oracle as orc
from adjacency_reference import adjacency_vjp
from helpers import elementwise_ratio, load_case, rel_max_err

pytestmark = pytest.mark.gpu

TOL = 1e-5


def report(tag, got, ref):
    err = rel_max_err(got, ref)
    ratio = elementwise_ratio(got, ref, TOL)
    ratio3 = elementwise_ratio(got, ref, TOL, floor=1e-3)
    print(f"\n[{tag}] rel {err:.2e}, elementwise_ratio x{ratio:.2f} (floor 5e-2), x{ratio3:.2f} (floor 1e-3)")
    assert err <= TOL, f"{tag}: rel max err {err:.3e}"
    assert ratio <= 1.0, f"{tag}: elementwise ratio {ratio:.2f} at the 5e-2 floor"


def report_lambda_max(tag, got, ref, size):
    """``dLoss/dlambda_max`` sums terms that cancel to ``m_k <lambda_k, L T_{k-1}>``; with a smooth
    signal (the default ``log1p(degree)``) ``L T`` is small against ``T``, so the float32 rounding of
    the orders is amplified in the plain relative error.  The bar is the error over the size of the
    sum before cancellation (DESIGN.md section 11); the plain relative error is printed beside it."""
    if size == 0.0:                          # K = 0: lambda_max does not enter the pass
        assert got == 0.0 and ref == 0.0, (tag, got, ref)
        return
    rel = abs(got - ref) / max(abs(ref), 1e-300)
    cond = abs(got - ref) / size
    print(f"\n[{tag}] rel {rel:.2e}, error / size of the sum {cond:.2e}")
    assert cond <= TOL, f"{tag}: error / size {cond:.3e}"


def dev(a):
    return torch.tensor(np.asarray(a), dtype=torch.float32, device="cuda")


def upstream(n, n_scales, f, k, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, n_scales * f)), rng.standard_normal((n, n_scales, f)),
            rng.standard_normal((k + 1, n, f)))


def pass_loss(res, hb, cb, tb, k):
    loss = (dev(hb) * res.features).sum() + (dev(cb) * res.combined).sum()
    return loss + sum((dev(tb[i]) * res.orders[i]).sum() for i in range(k + 1))


# name, F (None: the default signal, F = 1), scales, normalize, use_sell
GOLDEN = [
    ("cora_k0", None, 1, False, False),
    ("cora_k1", None, 3, False, False),
    ("cora_noloop", None, 1, False, True),           # F = 1 on the SELL step kernel
    ("cora_noloop", None, 3, False, False),          # F = 1 on the generic CSR kernel
    ("cora_k6_s04", None, 1, False, False),
    ("kat_path_loops", None, 1, False, False),
    ("directed_weighted", None, 3, False, False),
    ("directed_weighted", 1, 1, False, False),
    ("directed_weighted", 3, 3, True, False),
    ("cora_loops", 8, 1, True, False),
    ("directed_weighted", 37, 3, True, False),
    ("small_wide130", 130, 1, True, False),
]


def scales_for(case, n_scales):
    return [case["s"]] if n_scales == 1 else [case["s"], 0.4, 1.3]


@pytest.mark.parametrize("name,f,n_scales,normalize,use_sell", GOLDEN)
def test_dense_gradient_matches_reference(name, f, n_scales, normalize, use_sell):
    case = load_case(name)
    adj, k, n = case["adj"], case["k"], case["n"]
    fw = 1 if f is None else f
    scales = scales_for(case, n_scales)
    lam_v = 2.0 if n_scales == 1 else 1.7
    rng = np.random.default_rng(fw + n_scales)
    x_np = None if f is None else rng.standard_normal((n, f)).astype(np.float32)
    hb, cb, tb = upstream(n, n_scales, fw, k, seed=3 * fw + n_scales)
    a = torch.tensor(adj.toarray(), dtype=torch.float32, device="cuda", requires_grad=True)
    lam = torch.tensor(lam_v, dtype=torch.float64, requires_grad=True)
    x = None if x_np is None else dev(x_np)
    res = egnn.graph_wavelet_features(a, k=k, s=scales, X0=x, lambda_max=lam, normalize=normalize,
                                      return_parts=True, _use_sell=use_sell)
    pass_loss(res, hb, cb, tb, k).backward()
    dA, dlam, size = adjacency_vjp(adj, k, scales, None if x_np is None else x_np.astype(np.float64), lam_v,
                                   normalize, hb, cb, tb, with_scale=True)
    tag = f"{name} F={f} S={n_scales} sell={use_sell}"
    assert a.grad.shape == (n, n) and a.grad.dtype == torch.float32
    report(f"{tag} dA", a.grad.cpu().numpy(), dA)
    assert lam.grad.shape == () and lam.grad.dtype == torch.float64
    report_lambda_max(f"{tag} dlambda_max", float(lam.grad), dlam, size)


def coo_with_duplicate_and_zero(adj):
    """COO pattern of ``adj`` plus a duplicate of one stored entry (split weight) and an explicit zero."""
    coo = adj.tocoo()
    r, c, v = list(coo.row), list(coo.col), list(coo.data.astype(np.float64))
    r.append(r[5]); c.append(c[5]); v[5] *= 0.25; v.append(v[5] * 3.0)          # the two parts sum to the entry
    dense = adj.toarray()
    zi, zj = [(i, j) for i in range(adj.shape[0]) for j in range(adj.shape[0]) if i != j and dense[i, j] == 0][7]
    r.append(zi); c.append(zj); v.append(0.0)
    return np.array([r, c]), np.array(v)


@pytest.mark.parametrize("name,f", [("directed_weighted", 1), ("directed_weighted", 8), ("cora_loops", None)])
def test_sparse_coo_gradient_is_the_dense_gradient_at_the_pattern(name, f):
    case = load_case(name)
    adj, k, n = case["adj"], case["k"], case["n"]
    ei, vals = coo_with_duplicate_and_zero(adj)
    rng = np.random.default_rng(2)
    fw = 1 if f is None else f
    x_np = None if f is None else rng.standard_normal((n, f)).astype(np.float32)
    hb, cb, tb = upstream(n, 1, fw, k, seed=8)
    normalize = fw > 1
    w = torch.tensor(vals, dtype=torch.float32, device="cuda", requires_grad=True)
    A = torch.sparse_coo_tensor(torch.tensor(ei, device="cuda"), w, (n, n))
    res = egnn.graph_wavelet_features(A, k=k, s=0.8, X0=None if x_np is None else dev(x_np), normalize=normalize,
                                      return_parts=True)
    pass_loss(res, hb, cb, tb, k).backward()
    summed = sp.csr_matrix((vals, (ei[0], ei[1])), shape=(n, n))
    dA, _ = adjacency_vjp(summed, k, 0.8, None if x_np is None else x_np.astype(np.float64), 2.0, normalize, hb, cb, tb)
    assert w.grad.shape == w.shape
    report(f"{name} F={f} COO pattern", w.grad.cpu().numpy(), dA[ei[0], ei[1]])
    # duplicates share their entry's gradient; the explicit zero gets the gradient at its position
    g = w.grad.cpu().numpy()
    assert g[5] == g[-2]
    assert g[-1] != 0.0


def test_cpu_float64_leaf_and_0d_lambda_max():
    case = load_case("directed_weighted")
    adj, k, n = case["adj"], case["k"], case["n"]
    a = torch.tensor(adj.toarray(), dtype=torch.float64, requires_grad=True)
    lam = torch.tensor(1.7, dtype=torch.float32, requires_grad=True)
    hb, _, _ = upstream(n, 2, 1, k, seed=4)
    feats = egnn.graph_wavelet_features(a, k=k, s=[0.8, 1.4], lambda_max=lam, normalize=False)
    (dev(hb) * feats).sum().backward()
    assert a.grad.device.type == "cpu" and a.grad.dtype == torch.float64 and a.grad.shape == a.shape
    assert lam.grad.shape == () and lam.grad.dtype == torch.float32 and lam.grad.device.type == "cpu"
    dA, dlam, size = adjacency_vjp(adj, k, [0.8, 1.4], None, 1.7, False, hb, with_scale=True)
    report("cpu float64 leaf dA", a.grad.numpy(), dA)
    report_lambda_max("0-d float32 lambda_max", float(lam.grad), dlam, size)
    # lambda_max alone (nothing else needs a gradient)
    lam2 = torch.tensor(1.7, dtype=torch.float64, requires_grad=True)
    (dev(hb) * egnn.graph_wavelet_features(adj, k=k, s=[0.8, 1.4], lambda_max=lam2, normalize=False)).sum().backward()
    report_lambda_max("lambda_max alone", float(lam2.grad), dlam, size)


@pytest.mark.parametrize("f", [3, 8])
def test_signal_and_scale_gradients_unchanged(f):
    case = load_case("directed_weighted")
    adj, k, n = case["adj"], case["k"], case["n"]
    rng = np.random.default_rng(6)
    x_np = rng.standard_normal((n, f)).astype(np.float32)
    hb = dev(rng.standard_normal((n, 2 * f)))
    grads = []
    for with_adj in (False, True):
        x = dev(x_np).requires_grad_()
        s = torch.tensor([0.8, 1.6], dtype=torch.float64, requires_grad=True)
        a = torch.tensor(adj.toarray(), dtype=torch.float32, device="cuda", requires_grad=with_adj)
        lam = torch.tensor(1.7, dtype=torch.float64, requires_grad=with_adj)
        (hb * egnn.graph_wavelet_features(a, k=k, s=s, X0=x, lambda_max=lam)).sum().backward()
        assert (a.grad is not None) == with_adj and (lam.grad is not None) == with_adj
        grads.append((x.grad, s.grad))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


def ulps(a, b):
    a, b = a.double(), b.double()
    spacing = torch.from_numpy(np.spacing(np.abs(b.cpu().numpy()).astype(np.float32))).double().to(b.device)
    return ((a - b).abs() / spacing).max().item()


@pytest.mark.parametrize("name,f", [("cora_noloop", None), ("cora_wide8", 8)])
def test_features_unchanged(name, f):
    case = load_case(name)
    d = torch.tensor(case["adj"].toarray(), dtype=torch.float32, device="cuda")
    x = None if f is None else torch.tensor(case["X0"], device="cuda")
    with torch.no_grad():
        ref = egnn.graph_wavelet_features(d, k=case["k"], s=[0.8, 1.6], X0=x)
    feats = egnn.graph_wavelet_features(d.clone().requires_grad_(), k=case["k"], s=[0.8, 1.6], X0=x)
    assert feats.grad_fn is not None
    print(f"\n[{name}] features with an adjacency gradient vs no grad: {ulps(feats.detach(), ref):.1f} ulp")
    assert ulps(feats.detach(), ref) <= 4


@pytest.mark.parametrize("layout", ["dense", "coo"])
def test_backward_is_deterministic(layout):
    case = load_case("cora_wide8")
    adj, n = case["adj"], case["n"]
    hb = torch.randn(n, 16, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    coo = adj.tocoo()
    grads = []
    for _ in range(2):
        if layout == "dense":
            leaf = torch.tensor(adj.toarray(), dtype=torch.float32, device="cuda", requires_grad=True)
            a = leaf
        else:
            leaf = torch.tensor(coo.data, dtype=torch.float32, device="cuda", requires_grad=True)
            a = torch.sparse_coo_tensor(torch.tensor(np.array([coo.row, coo.col]), device="cuda"), leaf, (n, n))
        lam = torch.tensor(1.8, dtype=torch.float64, requires_grad=True)
        x = torch.tensor(case["X0"], device="cuda", requires_grad=True)
        (hb * egnn.graph_wavelet_features(a, k=case["k"], s=[0.8, 1.6], X0=x, lambda_max=lam)).sum().backward()
        grads.append((leaf.grad, lam.grad, x.grad))
    for u, v in zip(*grads):
        assert torch.equal(u, v)


# ---- full size -----------------------------------------------------------------------------------
def sparse_reference(adj, k, scales, x0, cb, lambda_max=2.0):
    """Float64 pieces of the adjacency gradient over the explicit operator (scipy): the orders, the
    Clenshaw vectors, ``d``, ``gw`` and ``grho``, for the upstream ``cb`` ``[N, S, F]`` on the
    un-normalised combination.  ``x0 = None``: the default signal."""
    A = orc.as_csr32(adj).astype(np.float64)
    n = A.shape[0]
    off = (A - sp.diags(A.diagonal())).tocsr()
    off.eliminate_zeros()
    w = np.asarray(off.sum(axis=0)).ravel()
    iso = w == 0
    d = np.where(iso, 1.0, 1.0 / np.sqrt(np.where(iso, 1.0, w)))
    M = orc.rescaled_laplacian(adj, lambda_max)
    MT = M.T.tocsr()
    x = (orc.input_signal(adj) if x0 is None else x0).astype(np.float64)
    T = orc.chebyshev_orders(M, k, x)
    alpha = orc.heat_coefficients(k, scales)
    v = [np.einsum("s,nsf->nf", alpha[:, i], cb) for i in range(k + 1)]
    lam = [np.zeros_like(x) for _ in range(k + 3)]
    for i in range(k, 0, -1):
        lam[i] = v[i] + 2 * (MT @ lam[i + 1]) - lam[i + 2]
    xbar = v[0] + (MT @ lam[1] - lam[2] if k > 0 else 0.0)
    a = 2.0 / lambda_max
    offT = off.T.tocsr()
    R, Q = np.zeros(n), np.zeros(n)
    for i in range(1, k + 1):
        m = 1.0 if i == 1 else 2.0
        R += m * (lam[i] * (off @ (d[:, None] * T[i - 1]))).sum(axis=1)
        Q += m * (T[i - 1] * (offT @ (d[:, None] * lam[i]))).sum(axis=1)
    gw = np.where(iso, 0.0, 0.5 * a * d ** 3 * (R + Q))
    grho = xbar[:, 0] / (1.0 + np.asarray(A.sum(axis=1)).ravel()) if x0 is None else np.zeros(n)
    return dict(T=T, lam=lam, d=d, gw=gw, grho=grho, a=a, k=k)


def pair_reference(ref, rows, cols):
    g = np.zeros(rows.shape[0])
    for i in range(1, ref["k"] + 1):
        g += (1.0 if i == 1 else 2.0) * (ref["lam"][i][rows] * ref["T"][i - 1][cols]).sum(axis=1)
    g *= ref["d"][rows] * ref["d"][cols]
    return np.where(rows != cols, -ref["a"] * g + ref["gw"][cols], 0.0) + ref["grho"][rows]


def coo_leaf(rp, ci, vals, n):
    """A sparse COO adjacency over a device CSR (row-major order: the coalesced order) with a value leaf."""
    rows = torch.repeat_interleave(torch.arange(n, device="cuda"), (rp[1:] - rp[:-1]).long())
    w = (torch.ones(ci.numel(), device="cuda") if vals is None else vals.clone()).requires_grad_()
    return torch.sparse_coo_tensor(torch.stack([rows, ci.long()]), w, (n, n)), w


def test_full_size_arxiv_directed_weighted_pattern():
    from test_gpu_backward import full_graph
    g = full_graph("arxiv", "weighted")
    n, f, k, scales = g.n, 16, 3, [0.8, 1.6]
    A, w = coo_leaf(g.rowptr, g.colidx, g.vals, n)
    gen = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(n, f, device="cuda", generator=gen)
    G = torch.randn(n, len(scales) * f, device="cuda", generator=gen)
    (G * egnn.graph_wavelet_features(A, k=k, s=scales, X0=x, normalize=False)).sum().backward()
    adj = g.to_scipy()
    ref = sparse_reference(adj, k, scales, x.double().cpu().numpy(), G.reshape(n, 2, f).double().cpu().numpy())
    rows = np.repeat(np.arange(n), np.diff(adj.indptr))
    report("arxiv directed weighted F=16 every entry", w.grad.cpu().numpy(), pair_reference(ref, rows, adj.indices))


def test_full_size_reddit_default_signal_sampled_rows():
    rp, ci, n = synth.synth_csr("reddit", self_loops=True, device="cuda")
    A, w = coo_leaf(rp, ci, None, n)
    G = torch.randn(n, 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    (G * egnn.graph_wavelet_features(A, k=3, s=0.8, normalize=False)).sum().backward()
    rp_h, ci_h = rp.cpu().numpy(), ci.cpu().numpy()
    adj = sp.csr_matrix((np.ones(ci_h.size, np.float32), ci_h, rp_h), shape=(n, n))
    del A
    ref = sparse_reference(adj, 3, 0.8, None, G.reshape(n, 1, 1).double().cpu().numpy())
    deg = np.diff(rp_h)
    rng = np.random.default_rng(11)
    sample = np.unique(np.concatenate([np.argsort(deg)[-4:], rng.choice(n, size=60, replace=False)]))
    ent = np.concatenate([np.arange(rp_h[r], rp_h[r + 1]) for r in sample])
    rows = np.repeat(sample, deg[sample])
    got = w.grad[torch.from_numpy(ent).cuda()].cpu().numpy()
    report(f"reddit F=1 default signal, {sample.size} rows ({ent.size} entries)", got,
           pair_reference(ref, rows, ci_h[ent]))


def test_full_size_20k_dense_sampled():
    n = 20_000
    e = synth.synth_edges(n, 10 * n, seed=6, device="cuda")
    keep = torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(8), device="cuda") < 0.6
    e = e[:, keep]
    vals = 0.5 + torch.rand(e.shape[1], generator=torch.Generator(device="cuda").manual_seed(9), device="cuda")
    a = torch.zeros((n, n), device="cuda")
    a[e[0], e[1]] = vals
    a[torch.arange(0, n, 97, device="cuda"), torch.arange(0, n, 97, device="cuda")] = 1.0     # a few self loops
    a.requires_grad_()
    G = torch.randn(n, 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(10))
    (G * egnn.graph_wavelet_features(a, k=3, s=0.8, normalize=False)).sum().backward()
    adj = sp.csr_matrix(sp.coo_matrix((vals.cpu().numpy(), (e[0].cpu().numpy(), e[1].cpu().numpy())), shape=(n, n)))
    adj = (adj + sp.diags(np.where(np.arange(n) % 97 == 0, 1.0, 0.0))).tocsr().astype(np.float32)
    ref = sparse_reference(adj, 3, 0.8, None, G.reshape(n, 1, 1).double().cpu().numpy())
    deg = np.diff(adj.indptr)
    rng = np.random.default_rng(12)
    rs = np.unique(np.concatenate([np.argsort(deg)[-2:], rng.choice(n, size=40, replace=False), [0, 97]]))
    cs = np.unique(np.concatenate([rs[:10], rng.choice(n, size=40, replace=False)]))
    rr, cc = np.meshgrid(rs, cs, indexing="ij")
    got = a.grad[torch.from_numpy(rs).cuda()][:, torch.from_numpy(cs).cuda()].cpu().numpy()
    report(f"20k dense F=1 default signal, {rs.size} x {cs.size}", got,
           pair_reference(ref, rr.ravel(), cc.ravel()).reshape(rr.shape))


@pytest.mark.parametrize("n_flips", [10, 100])
def test_wats_recompute_passes_no_wavelet_gradient_to_the_adjacency(n_flips):
    """``WATS`` stays forward-only in the adjacency: with ``recompute_on_forward`` a dense leaf that
    requires grad (the attack's ``modified_adj``) gets no gradient through the wavelet features,
    whether its flips take the no-rebuild path (<= 64) or the rebuilt graph (> 64)."""
    from models_for_tests import FixedLogits
    sh = synth.SHAPES["cora"]
    rp, ci, n = synth.synth_csr("cora", self_loops=True)
    adj = torch.tensor(sp.csr_matrix((np.ones(ci.numel(), np.float32), ci.numpy(), rp.numpy()), shape=(n, n)).toarray())
    y, logits, val, _ = synth.synth_labels(sh.n, sh.n_classes, seed=42)
    torch.manual_seed(3)
    cal = egnn.WATS(FixedLogits(logits), torch.zeros(n, 4), y, adj, val, verbose=False, train=False,
                    recompute_on_forward=True)
    rng = np.random.default_rng(n_flips)
    pert = cal.adj.clone()
    for i, j in rng.choice(n, size=(n_flips, 2)):
        if i != j:
            pert[i, j] = 1.0 - pert[i, j]
    leaf = pert.clone().requires_grad_()
    assert cal.features_for(leaf).grad_fn is None
    cal(cal.x, leaf).sum().backward()                  # the base model ignores adj: only the features could reach it
    assert leaf.grad is None
