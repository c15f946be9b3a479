"""Backward of the wavelet pass on the GPU (adjoint Chebyshev kernels).

* Parity of the signal's gradient with ``tests/vjp_reference.wavelet_vjp`` (float64,
  explicit transposed operator) on the golden graphs, with random upstream
  gradients on the features, the combination and the orders: norm-wise
  ``||Xbar_gpu - Xbar_ref||_inf / ||Xbar_ref||_inf <= 1e-5`` and element-wise ratio
  <= 1 at the 5e-2 floor (the forward's bars), the ratio at the 1e-3 floor printed beside them.  The scales' gradient against the
  oracle at the same bar; ``chebyshev_polynomials``, ``L @ x`` and the explicit
  scipy operator.
* Flips: the gradient on ``deltas=`` equals the gradient on the rebuilt graph.
* Full size: the signal's gradient element-wise on chosen columns against the float64
  transposed operator, and the scales' gradient against float64 sums of the pass's own orders.
  Every adjoint instantiation at small size: test_gpu_adjoint_matrix.py.
* Determinism and no change of the forward when nothing needs a gradient.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import synth
from oracle import wats_oracle as orc
from helpers import elementwise_ratio, load_case, rel_max_err
from vjp_reference import wavelet_vjp

pytestmark = pytest.mark.gpu

TOL = 1e-5

# F = 1 golden signals are checked without the normalisation: there H = sign(C) and its derivative,
# 1e-8 / r^2, is below the float32 rounding of 1 - |C| / r (it vanishes almost everywhere).
PARITY = [(name, n_scales, normalize)
          for name in ["cora_noloop", "cora_loops", "directed_weighted", "cora_k0", "cora_k1", "cora_k6_s04", "cora_wide8",
                       "small_wide130"]
          for n_scales in (1, 3) for normalize in (False, True)
          if normalize is False or name in ("cora_wide8", "small_wide130")]


def scales_for(case, n_scales):
    return [case["s"]] if n_scales == 1 else [case["s"], 0.4, 1.3]


def report(tag, got, ref):
    err = rel_max_err(got, ref)
    ratio = elementwise_ratio(got, ref, TOL)
    ratio3 = elementwise_ratio(got, ref, TOL, floor=1e-3)
    print(f"\n[{tag}] rel {err:.2e}, elementwise_ratio x{ratio:.2f} (floor 5e-2), x{ratio3:.2f} (floor 1e-3)")
    assert err <= TOL, f"{tag}: rel max err {err:.3e}"
    assert ratio <= 1.0, f"{tag}: elementwise ratio {ratio:.2f} at the 5e-2 floor"
    return err


def upstream(n, n_scales, f, k, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, n_scales * f)), rng.standard_normal((n, n_scales, f)),
            rng.standard_normal((k + 1, n, f)))


@pytest.mark.parametrize("name,n_scales,normalize", PARITY)
def test_vjp_parity_with_oracle(name, n_scales, normalize):
    case = load_case(name)
    adj, k, n = case["adj"], case["k"], case["n"]
    x_np = case["X0"].astype(np.float32)
    f = x_np.shape[1]
    scales = scales_for(case, n_scales)
    lam = 2.0 if n_scales == 1 else 1.7
    hb, cb, tb = upstream(n, n_scales, f, k, seed=n_scales + 2 * normalize)
    x = torch.tensor(x_np, device="cuda", requires_grad=True)
    s = torch.tensor(scales, dtype=torch.float64, requires_grad=True)
    res = egnn.graph_wavelet_features(adj, k=k, s=s, X0=x, lambda_max=lam, normalize=normalize, return_parts=True)
    dev = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")
    loss = (dev(hb) * res.features).sum() + (dev(cb) * res.combined).sum()
    loss = loss + sum((dev(tb[i]) * res.orders[i]).sum() for i in range(k + 1))
    loss.backward()
    xbar_ref, sbar_ref = wavelet_vjp(adj, k, scales, x_np.astype(np.float64), lam, normalize, hb, cb, tb)
    report(f"{name} S={n_scales} normalize={normalize} Xbar", x.grad.cpu().numpy(), xbar_ref)
    assert s.grad.shape == s.shape and s.grad.dtype == torch.float64
    report(f"{name} S={n_scales} normalize={normalize} sbar", s.grad.numpy(), sbar_ref)


def test_scalar_scale_gradient_and_x0_on_the_host():
    """A 0-d ``s`` and a float64 CPU leaf: the gradients come back in their shape, dtype and device."""
    case = load_case("cora_wide8")
    adj, k, n = case["adj"], case["k"], case["n"]
    x = torch.tensor(case["X0"], dtype=torch.float64, requires_grad=True)
    s = torch.tensor(0.8, dtype=torch.float32, requires_grad=True)
    hb, _, _ = upstream(n, 1, 8, k, seed=11)
    feats = egnn.graph_wavelet_features(adj, k=k, s=s, X0=x)
    (torch.tensor(hb, dtype=torch.float32, device="cuda") * feats).sum().backward()
    assert x.grad.device.type == "cpu" and x.grad.dtype == torch.float64 and x.grad.shape == x.shape
    assert s.grad.shape == () and s.grad.dtype == torch.float32
    xbar_ref, sbar_ref = wavelet_vjp(adj, k, 0.8, case["X0"].astype(np.float32).astype(np.float64), 2.0, True, hb)
    report("cora_wide8 cpu leaf Xbar", x.grad.numpy(), xbar_ref)
    report("cora_wide8 0-d sbar", s.grad.reshape(1).numpy(), sbar_ref)


@pytest.mark.parametrize("name", ["cora_loops", "directed_weighted"])
def test_chebyshev_polynomials_and_operator_gradients(name):
    case = load_case(name)
    adj, k, n = case["adj"], case["k"], case["n"]
    lam = 1.7
    rng = np.random.default_rng(5)
    x_np = rng.standard_normal((n, 3)).astype(np.float32)
    tb = rng.standard_normal((k + 1, n, 3))
    dev = lambda a: torch.tensor(a, dtype=torch.float32, device="cuda")
    want, _ = wavelet_vjp(adj, k, 0.8, x_np.astype(np.float64), lam, False, None, np.zeros((n, 1, 3)), tb)
    # implicit operator (fused orders) and the reference's explicit scipy matrix (one application per order)
    for tag, L in (("implicit", egnn.compute_normalized_laplacian(adj).rescaled(lam)),
                   ("explicit scipy", orc.rescaled_laplacian(adj, lam))):
        x = dev(x_np).requires_grad_()
        orders = egnn.chebyshev_polynomials(L, k, x)
        sum((dev(tb[i]) * orders[i]).sum() for i in range(k + 1)).backward()
        report(f"{name} chebyshev_polynomials {tag}", x.grad.cpu().numpy(), want)
    # one application: L @ x, and the explicit operator's @
    gb = rng.standard_normal((n, 3))
    one = np.stack([np.zeros((n, 3)), gb])
    want1, _ = wavelet_vjp(adj, 1, 0.8, x_np.astype(np.float64), lam, False, None, np.zeros((n, 1, 3)), one)
    x = dev(x_np).requires_grad_()
    (dev(gb) * (egnn.compute_normalized_laplacian(adj).rescaled(lam) @ x)).sum().backward()
    report(f"{name} L @ x", x.grad.cpu().numpy(), want1)
    from efficient_gnn_b200.wats import ExplicitOperator
    x = dev(x_np).requires_grad_()
    (dev(gb) * (ExplicitOperator(orc.rescaled_laplacian(adj, lam)) @ x)).sum().backward()
    report(f"{name} explicit @", x.grad.cpu().numpy(), want1)


def test_csr_adjoint_is_the_transpose_with_the_forward_degree_vectors():
    case = load_case("directed_weighted")
    g = egnn.as_graph(case["adj"])
    gt = g.adjoint()
    assert gt is not g and gt is g.adjoint()
    assert gt.dinv is g.dinv and gt.iso is g.iso
    want = case["adj"].T.tocsr()
    want.sort_indices()
    assert np.array_equal(gt.rowptr.cpu().numpy(), want.indptr)
    assert np.array_equal(gt.colidx.cpu().numpy(), want.indices)
    assert np.array_equal(gt.vals.cpu().numpy(), want.data.astype(np.float32))
    sym = egnn.as_graph(load_case("cora_noloop")["adj"])
    assert sym.adjoint() is sym


@pytest.mark.parametrize("name,f", [("cora_noloop", 1), ("directed_weighted", 4), ("cora_loops", 16)])
def test_flip_gradient_equals_rebuilt_graph(name, f):
    case = load_case(name)
    adj, n = case["adj"].tocsr(), case["n"]
    rng = np.random.default_rng(9)
    x_np = rng.standard_normal((n, f)).astype(np.float32)
    rows, cols, vals = [], [], []
    dense_rows = adj.toarray()
    for _ in range(6):                                   # directed flips: the adjoint takes them transposed
        i, j = (int(v) for v in rng.choice(n, size=2, replace=False))
        v = -float(dense_rows[i, j]) if dense_rows[i, j] != 0 else 1.0
        rows.append(i); cols.append(j); vals.append(v)
        dense_rows[i, j] += v
    rebuilt = sp.csr_matrix(dense_rows)
    s = [0.8, 1.6]
    g = torch.tensor(rng.standard_normal((n, 2 * f)), dtype=torch.float32, device="cuda")
    grads = []
    for a, d in ((egnn.as_graph(adj), (rows, cols, vals)), (egnn.as_graph(rebuilt), None)):
        x = torch.tensor(x_np, device="cuda", requires_grad=True)
        st = torch.tensor(s, dtype=torch.float64, requires_grad=True)
        feats = egnn.graph_wavelet_features(a, k=3, s=st, X0=x, deltas=d, normalize=f > 1)
        (g * feats).sum().backward()
        grads.append((x.grad.double(), st.grad))
    (xa, sa), (xb, sb) = grads
    assert ((xa - xb).abs().max() / xb.abs().max()).item() <= 2e-6
    assert ((sa - sb).abs().max() / sb.abs().max()).item() <= 2e-6


# ---- full size -----------------------------------------------------------------------------------
def directed_half(rp, ci, n, seed):
    keep = torch.rand(ci.numel(), generator=torch.Generator(device="cuda").manual_seed(seed), device="cuda") < 0.5
    row = torch.repeat_interleave(torch.arange(n, device="cuda"), (rp[1:] - rp[:-1]).long())
    counts = torch.bincount(row[keep], minlength=n)
    rp2 = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rp2[1:] = torch.cumsum(counts, 0)
    return rp2.to(torch.int32), ci[keep].contiguous()


def full_graph(shape, directed):
    """Device graph of a full-size shape: binary symmetric with self loops; directed=True keeps a
    seeded half of the entries, "weighted" also gives them seeded weights in [0.5, 2)."""
    rp, ci, n = synth.synth_csr(shape, self_loops=True, device="cuda")
    vals = None
    if directed:
        rp, ci = directed_half(rp, ci, n, seed=2)
    if directed == "weighted":
        gen = torch.Generator(device="cuda").manual_seed(4)
        vals = 0.5 + 1.5 * torch.rand(ci.numel(), generator=gen, device="cuda")
    return egnn.CsrGraph(rp, ci, vals, n)


_MT = {}


@pytest.fixture(scope="module")
def transposed_operator():
    """``rescaled_laplacian(adj).T`` (float64 CSR) of a full-size graph, built once per graph."""
    def get(shape, directed, g):
        key = (shape, directed)
        if key not in _MT:
            data = np.ones(g.nnz, np.float32) if g.vals is None else g.vals.cpu().numpy()
            adj = sp.csr_matrix((data, g.colidx.cpu().numpy(), g.rowptr.cpu().numpy()), shape=(g.n, g.n))
            _MT[key] = orc.rescaled_laplacian(adj).T.tocsr()
        return _MT[key]
    yield get
    _MT.clear()


def check_columns(f):
    """Columns on both sides of the 4-column groups and of the 128-column feature tiles."""
    return sorted(c for c in {0, 1, 3, 4, 31, 32, 63, 64, 127, f - 5, f - 4, f - 1} if 0 <= c < f)


FULL = [("arxiv", 128, [0.3, 0.8, 1.6, 2.4], False), ("reddit", 64, [0.8], False),
        ("reddit", 1, [0.8, 1.6], False), ("arxiv", 16, [0.8, 1.6], True), ("arxiv", 37, [0.8, 1.3], "weighted")]


@pytest.mark.parametrize("shape,f,scales,directed", FULL)
def test_adjoint_identity_full_size(shape, f, scales, directed, transposed_operator):
    """Full size, element-wise on chosen columns: with normalize=False the columns are independent,
    so ``Xbar[:, cols]`` is compared with ``sum_i T_i(M^T) v_i`` on those columns (scipy, float64);
    F = 1 on the Reddit shape checks every row, hub rows included.  The scales' gradient is compared
    with ``-sum_k k alpha_jk <Cbar_j, T_k>`` summed in float64 from the pass's own orders (checked
    against the oracle by test_gpu_full_size.py): that isolates the coefficient-gradient reduction."""
    g = full_graph(shape, directed)
    n = g.n
    if directed:
        assert g.adjoint() is not g
    gen = torch.Generator(device="cuda").manual_seed(7)
    x = torch.randn(n, f, device="cuda", generator=gen).requires_grad_()
    s = torch.tensor(scales, dtype=torch.float64, requires_grad=True)
    G = torch.randn(n, len(scales) * f, device="cuda", generator=gen)
    res = egnn.graph_wavelet_features(g, k=3, s=s, X0=x, normalize=False, return_parts=True)
    (G * res.features).sum().backward()
    k, n_scales = 3, len(scales)
    alpha = egnn.heat_coefficients(k, scales)
    cbar = G.reshape(n, n_scales, f)
    # scale gradient: float64 sums of the pass's own float32 orders
    terms = torch.stack([torch.stack([(cbar[:, j].double() * res.orders[i].detach().double()).sum()
                                      for i in range(k + 1)]) for j in range(n_scales)]).cpu().numpy()
    size = torch.stack([torch.stack([(cbar[:, j].double().abs() * res.orders[i].detach().double().abs()).sum()
                                     for i in range(k + 1)]) for j in range(n_scales)]).cpu().numpy()
    kk = np.arange(k + 1)
    s_ref = -(kk * alpha * terms).sum(axis=1)
    s_size = (kk * alpha * size).sum(axis=1)
    s_rel = float((np.abs(s.grad.numpy() - s_ref) / s_size).max())
    tag = f"{shape} F={f} S={n_scales} directed={directed}"
    print(f"\n[{tag} sbar] rel to sum|terms| {s_rel:.2e}")
    assert s_rel <= 1e-10
    # signal gradient on chosen columns
    mt = transposed_operator(shape, directed, g)
    cols = check_columns(f)
    cb = cbar[:, :, cols].double().cpu().numpy()
    want = np.zeros((n, len(cols)))
    for i in range(k + 1):
        v = np.einsum("s,nsc->nc", alpha[:, i], cb)
        want += orc.chebyshev_orders(mt, i, v)[i]
    report(f"{tag} Xbar[:, {cols}]", x.grad[:, cols].cpu().numpy(), want)


# ---- determinism and the forward ----------------------------------------------------------------
@pytest.mark.parametrize("name", ["directed_weighted", "cora_wide8"])
def test_backward_is_deterministic(name):
    case = load_case(name)
    g = egnn.as_graph(case["adj"])
    hb = torch.randn(case["n"], 2 * case["X0"].shape[1], device="cuda",
                     generator=torch.Generator(device="cuda").manual_seed(1))
    grads = []
    for _ in range(2):
        x = torch.tensor(case["X0"], device="cuda", requires_grad=True)
        s = torch.tensor([0.8, 1.6], dtype=torch.float64, requires_grad=True)
        (hb * egnn.graph_wavelet_features(g, k=case["k"], s=s, X0=x)).sum().backward()
        grads.append((x.grad, s.grad))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


def ulps(a, b):
    a, b = a.double(), b.double()
    spacing = torch.from_numpy(np.spacing(np.abs(b.cpu().numpy()).astype(np.float32))).double().to(b.device)
    return ((a - b).abs() / spacing).max().item()


@pytest.mark.parametrize("name", ["cora_noloop", "cora_wide8", "small_wide130"])
def test_forward_unchanged(name):
    case = load_case(name)
    g = egnn.as_graph(case["adj"])
    k, x_np = case["k"], case["X0"]
    x = torch.tensor(x_np, device="cuda")
    with torch.no_grad():
        ref = egnn.graph_wavelet_features(g, k=k, s=[0.8, 1.6], X0=x)
        ref_parts = egnn.graph_wavelet_features(g, k=k, s=[0.8, 1.6], X0=x, return_parts=True)
    plain = egnn.graph_wavelet_features(g, k=k, s=[0.8, 1.6], X0=x)        # grad mode, nothing needs grad
    assert plain.grad_fn is None and torch.equal(plain, ref)
    xg = x.clone().requires_grad_()
    parts = egnn.graph_wavelet_features(g, k=k, s=[0.8, 1.6], X0=xg, return_parts=True)
    assert parts.features.grad_fn is not None and parts.combined.grad_fn is not None
    assert torch.equal(parts.combined, ref_parts.combined)
    for a, b in zip(parts.orders, ref_parts.orders):
        assert torch.equal(a, b)
    feats = egnn.graph_wavelet_features(g, k=k, s=[0.8, 1.6], X0=xg)
    assert torch.equal(feats.detach(), parts.features.detach())
    print(f"\n[{name}] grad-mode features vs the fused forward: {ulps(feats.detach(), ref):.1f} ulp")
    assert ulps(feats.detach(), ref) <= 4
