"""Gradients through edge flips on one GPU (egnn_adj_grad_degree_flips, DESIGN.md section 14).

The reference is the float64 ``adjacency_vjp`` of the dense flipped graph ``A' = A + delta``.  Bars of
sections 2 and 10: norm-wise <= 1e-5 (1e-4 above 16 orders), element-wise ratio <= 1 at the 5e-2
floor, the 1e-3-floor ratio printed; ``lambda_max`` against section 11's size-relative bar.

* Routes: the SELL plan (F = 1 default signal), the generic kernel at F = 1 and 3, the wide kernel at
  F = 8 and 37; a binary symmetric graph and a weighted directed one with a hub; K = 0, 1, 3, 17;
  S = 1, 3; a dense leaf or COO values as the base, with the flip values and ``lambda_max`` as
  inputs too; 1, 10 and 64 flips (added, removed, weighted, diagonal, isolating, repeated).
* Determinism, features against the no-grad call, unchanged signal / scale gradients, and the
  launched kernels.
* ``WATS(..., recompute_on_forward=True, adjacency_grad=True)`` on a Cora-shape graph with 10 and 100
  flips (the resident graph with flips, and a rebuilt graph).
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import efficient_gnn_b200 as egnn
from efficient_gnn_b200 import wats
from efficient_gnn_b200.graph import deltas_from_dense
from adjacency_reference import adjacency_vjp
from helpers import elementwise_ratio, load_case, rel_max_err

pytestmark = pytest.mark.gpu


def report(tag, got, ref, tol, whole=None):
    """``whole``: ``|dLoss/dA'|`` when ``got`` / ``ref`` are some of its entries (the flip values): its
    size scales both bars, as for every other entry of that gradient."""
    if whole is not None:
        got, ref = np.append(got, whole.max()), np.append(ref, whole.max())   # one exact entry of the size
    err = rel_max_err(got, ref)
    ratio = elementwise_ratio(got, ref, tol)
    ratio3 = elementwise_ratio(got, ref, tol, floor=1e-3)
    print(f"\n[{tag}] rel {err:.2e}, elementwise_ratio x{ratio:.2f} (floor 5e-2), x{ratio3:.2f} (floor 1e-3)")
    assert err <= tol, f"{tag}: rel max err {err:.3e}"
    assert ratio <= 1.0, f"{tag}: elementwise ratio {ratio:.2f} at the 5e-2 floor"


def report_lambda_max(tag, got, ref, size, tol):
    if size == 0.0:                          # K = 0: lambda_max does not enter the pass
        assert got == 0.0 and ref == 0.0, (tag, got, ref)
        return
    cond = abs(got - ref) / size
    print(f"\n[{tag}] rel {abs(got - ref) / max(abs(ref), 1e-300):.2e}, error / size of the sum {cond:.2e}")
    assert cond <= tol, f"{tag}: error / size {cond:.3e}"


def dev(a):
    return torch.tensor(np.asarray(a), dtype=torch.float32, device="cuda")


def ulps(a, b):
    a, b = a.double(), b.double()
    spacing = torch.from_numpy(np.spacing(np.abs(b.cpu().numpy()).astype(np.float32))).double().to(b.device)
    return ((a - b).abs() / spacing).max().item()


def base_graph(name):
    """``binary``: the symmetric Cora golden graph; ``hub``: the weighted directed golden graph with
    node 0 made a hub (weighted edges to and from a third of the nodes)."""
    if name == "binary":
        return load_case("cora_noloop")["adj"].toarray().astype(np.float64)
    A = load_case("directed_weighted")["adj"].toarray().astype(np.float64)
    rng = np.random.default_rng(4)
    n = A.shape[0]
    for j in rng.choice(np.arange(1, n), size=n // 3, replace=False):
        A[0, j] = np.float32(0.5 + rng.random())
        A[j, 0] = np.float32(0.5 + rng.random())
    return A


def make_flips(A, m, seed):
    """``m`` flips on ``A``: an added entry, a removed stored entry, a weighted flip on a stored entry, a
    diagonal flip, one that removes the only in-edge of a column (isolating it) and a repeat of an
    earlier entry, cycled; with one flip, an added entry."""
    rng = np.random.default_rng(seed)
    n = A.shape[0]
    off = A - np.diag(np.diag(A))
    one_in = [c for c in range(n) if (off[:, c] != 0).sum() == 1]
    iso_col = one_in[0] if one_in else None
    rows, cols, vals = [], [], []
    used = set()

    def pick(stored):
        while True:
            r, c = map(int, rng.integers(0, n, size=2))
            if r != c and (A[r, c] != 0) == stored and c != iso_col and (r, c) not in used:
                used.add((r, c))
                return r, c

    kinds = ["added", "removed", "weighted", "diagonal", "isolate", "repeat"]
    for p in range(m):
        kind = kinds[p % len(kinds)] if m > 1 else "added"
        if kind == "isolate" and (iso_col is None or (p // len(kinds)) > 0):
            kind = "added"
        if kind == "added":
            (r, c), v = pick(False), float(np.float32(0.5 + rng.random()))
        elif kind == "removed":
            r, c = pick(True)
            v = -float(A[r, c])
        elif kind == "weighted":
            (r, c), v = pick(True), float(np.float32(rng.random() - 0.3))
        elif kind == "diagonal":
            r = c = int(rng.integers(0, n))
            v = float(np.float32(0.25 + rng.random()))
        elif kind == "isolate":
            r, c = int(np.nonzero(off[:, iso_col])[0][0]), iso_col
            v = -float(A[r, c])
        else:
            q = int(rng.integers(0, len(rows)))
            r, c, v = rows[q], cols[q], float(np.float32(0.3 + rng.random()))
        rows.append(r)
        cols.append(c)
        vals.append(v)
    return rows, cols, vals


def flipped(A, flips):
    Ap = A.copy()
    for r, c, v in zip(*flips):
        Ap[r, c] += v
    return Ap


# graph, F (None: default signal), K, S, flips, base input, use_sell
CASES = [
    ("binary", None, 3, 1, 10, "dense", True),
    ("binary", None, 17, 3, 64, "coo", True),
    ("binary", None, 1, 3, 1, "dense", False),
    ("hub", None, 3, 3, 64, "coo", None),
    ("hub", 3, 3, 3, 10, "dense", None),
    ("hub", 3, 0, 1, 10, "dense", None),
    ("hub", 8, 3, 1, 64, "coo", None),
    ("binary", 8, 17, 1, 64, "dense", None),
    ("hub", 37, 3, 3, 10, "dense", None),
    ("binary", 37, 1, 1, 1, "coo", None),
]


def run_case(graph, f, k, n_scales, n_flips, base, use_sell, seed=0):
    A = base_graph(graph)
    n = A.shape[0]
    flips = make_flips(A, n_flips, seed=n_flips + k)
    scales = [0.8] if n_scales == 1 else [0.8, 0.4, 1.3]
    normalize = f is not None
    fw = 1 if f is None else f
    rng = np.random.default_rng(fw + n_scales + k)
    x_np = None if f is None else rng.standard_normal((n, f)).astype(np.float32)
    hb = rng.standard_normal((n, n_scales * fw))
    if base == "dense":
        leaf = torch.tensor(A, dtype=torch.float32, device="cuda", requires_grad=True)
        adj = leaf
    else:
        r, c = np.nonzero(A)
        leaf = torch.tensor(A[r, c], dtype=torch.float32, device="cuda", requires_grad=True)
        adj = torch.sparse_coo_tensor(torch.tensor(np.array([r, c]), device="cuda"), leaf, (n, n))
    dv = torch.tensor(flips[2], dtype=torch.float32, device="cuda", requires_grad=True)
    lam = torch.tensor(1.7, dtype=torch.float64, requires_grad=True)
    feats = egnn.graph_wavelet_features(adj, k=k, s=scales, X0=None if x_np is None else dev(x_np), lambda_max=lam,
                                        normalize=normalize, deltas=(flips[0], flips[1], dv), _use_sell=use_sell)
    (dev(hb) * feats).sum().backward()
    return dict(A=A, flips=flips, scales=scales, normalize=normalize, x=x_np, hb=hb, leaf=leaf, dv=dv, lam=lam,
                base=base, k=k, feats=feats)


@pytest.mark.parametrize("graph,f,k,n_scales,n_flips,base,use_sell", CASES)
def test_flip_gradients_match_reference(graph, f, k, n_scales, n_flips, base, use_sell):
    c = run_case(graph, f, k, n_scales, n_flips, base, use_sell)
    Ap = flipped(c["A"], c["flips"])
    dA, dlam, size = adjacency_vjp(Ap, k, c["scales"], None if c["x"] is None else c["x"].astype(np.float64), 1.7,
                                   c["normalize"], c["hb"], with_scale=True)
    tol = 1e-4 if k > 16 else 1e-5
    tag = f"{graph} F={f} K={k} S={n_scales} flips={n_flips} {c['base']} sell={use_sell}"
    if c["base"] == "dense":
        report(f"{tag} dA'", c["leaf"].grad.cpu().numpy(), dA, tol)
    else:
        r, cc = np.nonzero(c["A"])
        report(f"{tag} COO values", c["leaf"].grad.cpu().numpy(), dA[r, cc], tol)
    rows, cols, _ = c["flips"]
    report(f"{tag} flip values", c["dv"].grad.cpu().numpy(), dA[rows, cols], tol, whole=np.abs(dA))
    report_lambda_max(f"{tag} dlambda_max", float(c["lam"].grad), dlam, size, tol)


def test_repeated_flips_share_the_entry_gradient():
    c = run_case("hub", 3, 3, 1, 10, "dense", None)
    rows, cols, _ = c["flips"]
    g = c["dv"].grad.cpu().numpy()
    seen = {}
    repeats = 0
    for p, key in enumerate(zip(rows, cols)):
        if key in seen:
            assert g[p] == g[seen[key]]
            repeats += 1
        seen.setdefault(key, p)
    assert repeats >= 1


@pytest.mark.parametrize("graph,f,base,use_sell", [("binary", None, "dense", True), ("hub", 8, "coo", None)])
def test_backward_is_deterministic(graph, f, base, use_sell):
    runs = [run_case(graph, f, 3, 3, 64, base, use_sell) for _ in range(2)]
    for name in ("leaf", "dv", "lam"):
        assert torch.equal(runs[0][name].grad, runs[1][name].grad), name


@pytest.mark.parametrize("graph,f,use_sell", [("binary", None, True), ("binary", 8, None), ("hub", 3, None)])
def test_features_match_the_no_grad_call(graph, f, use_sell):
    A = base_graph(graph)
    n = A.shape[0]
    flips = make_flips(A, 10, seed=5)
    x = None if f is None else dev(np.random.default_rng(1).standard_normal((n, f)))
    d = torch.tensor(A, dtype=torch.float32, device="cuda")
    with torch.no_grad():
        ref = egnn.graph_wavelet_features(d, k=3, s=[0.8, 1.6], X0=x, deltas=flips, _use_sell=use_sell)
    dv = torch.tensor(flips[2], device="cuda", requires_grad=True)
    feats = egnn.graph_wavelet_features(d.clone().requires_grad_(), k=3, s=[0.8, 1.6], X0=x,
                                        deltas=(flips[0], flips[1], dv), _use_sell=use_sell)
    assert feats.grad_fn is not None
    print(f"\n[{graph} F={f}] flipped features with gradients vs no grad: {ulps(feats.detach(), ref):.1f} ulp")
    # the no-grad pass normalises inside its last order's kernel, the differentiable one out of place
    assert ulps(feats.detach(), ref) <= 8


@pytest.mark.parametrize("f", [3, 8])
def test_signal_and_scale_gradients_unchanged_with_flips(f):
    A = base_graph("hub")
    n = A.shape[0]
    flips = make_flips(A, 10, seed=2)
    rng = np.random.default_rng(6)
    x_np = rng.standard_normal((n, f)).astype(np.float32)
    hb = dev(rng.standard_normal((n, 2 * f)))
    grads = []
    for with_adj in (False, True):
        x = dev(x_np).requires_grad_()
        s = torch.tensor([0.8, 1.6], dtype=torch.float64, requires_grad=True)
        a = torch.tensor(A, dtype=torch.float32, device="cuda", requires_grad=with_adj)
        dv = torch.tensor(flips[2], device="cuda", requires_grad=with_adj)
        lam = torch.tensor(1.7, dtype=torch.float64, requires_grad=with_adj)
        (hb * egnn.graph_wavelet_features(a, k=3, s=s, X0=x, lambda_max=lam,
                                          deltas=(flips[0], flips[1], dv))).sum().backward()
        assert (a.grad is not None) == with_adj and (dv.grad is not None) == with_adj
        assert (lam.grad is not None) == with_adj
        grads.append((x.grad, s.grad))
    assert torch.equal(grads[0][0], grads[1][0]) and torch.equal(grads[0][1], grads[1][1])


def kernels_of(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == "CUDA"]


def test_flip_kernel_launches_only_with_flips():
    A = base_graph("hub")
    flips = make_flips(A, 10, seed=3)
    hb = torch.randn(A.shape[0], 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))

    def backward(with_flips, grad):
        a = torch.tensor(A, dtype=torch.float32, device="cuda", requires_grad=grad)
        feats = egnn.graph_wavelet_features(a, k=3, s=0.8, normalize=False, deltas=flips if with_flips else None)
        if grad:
            (hb * feats).sum().backward()

    for with_flips in (False, True):
        backward(with_flips, True)                   # warm up: the transposed graph and the modules
        names = kernels_of(lambda: backward(with_flips, True))
        n_flip = sum("adj_grad_flip_terms_kernel" in m for m in names)
        assert n_flip == (1 if with_flips else 0), (with_flips, names)
        assert sum("adj_grad_degree_kernel" in m for m in names) == 2
        assert sum("adj_grad_finish_kernel" in m for m in names) == 1
        assert sum("adj_grad_dense_kernel" in m for m in names) == 1
        plain = kernels_of(lambda: backward(with_flips, False))
        assert not any("adj_grad" in m for m in plain), plain


# ---- WATS, attack-shaped --------------------------------------------------------------------------
@pytest.mark.parametrize("model_name", ["fixed", "gcn"])
@pytest.mark.parametrize("n_flips", [10, 100])
def test_wats_adjacency_grad(n_flips, model_name):
    """The leaf's gradient is the base model's term plus ``adjacency_vjp(A', upstream)``, ``upstream``
    being the gradient of the head (torch autograd) and of the normalisation w.r.t. the un-normalised
    combination ``S``.  With one feature per scale the normalised feature is ``S/(|S| + 1e-8)``, whose
    float32 backward ``(hbar - sign(S) <hbar, h>)/r`` is a difference of two nearly equal numbers: it is
    rounding-level, and any change in the last bit of ``S`` changes it.  So the upstream is taken at the
    library's own ``S`` (the same pass, rerun without gradients) through the library's normalisation,
    and the reference checks everything after it in float64.  ``fixed``: a base model that ignores the
    adjacency, so the leaf's gradient is the wavelet term alone (about 1e-7 here, far below the base
    term of ``gcn``, a dense GCN)."""
    from efficient_gnn_b200 import synth
    from models_for_tests import DenseGCN, FixedLogits
    sh = synth.SHAPES["cora"]
    rp, ci, n = synth.synth_csr("cora", self_loops=True)
    A = sp.csr_matrix((np.ones(ci.numel(), np.float32), ci.numpy(), rp.numpy()), shape=(n, n)).toarray()
    y, logits, val, _ = synth.synth_labels(sh.n, sh.n_classes, seed=42)
    torch.manual_seed(3)
    x = torch.randn(n, 8)
    model = FixedLogits(logits) if model_name == "fixed" else DenseGCN(8, sh.n_classes, nhid=16, dropout=0.0)
    scales = [0.8, 0.4, 1.3]
    cal = egnn.WATS(model, x, y, torch.tensor(A), val, s=scales, verbose=False, train=False,
                    recompute_on_forward=True, adjacency_grad=True)
    cal.eval()
    rng = np.random.default_rng(n_flips)
    pert = A.copy()
    for i, j in rng.choice(n, size=(n_flips, 2)):
        if i != j:
            pert[i, j] = 1.0 - pert[i, j]
    G = torch.randn(n, sh.n_classes, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    leaf = torch.tensor(pert, device="cuda", requires_grad=True)
    (G * cal(cal.x, leaf)).sum().backward()
    # the reference: the base model's term by torch, the upstream at the features by torch
    leaf2 = torch.tensor(pert, device="cuda", requires_grad=True)
    flips = deltas_from_dense(cal.adj, torch.tensor(pert, device="cuda"))
    assert (flips is not None) == (n_flips <= 64)
    with torch.no_grad():
        if flips is not None:          # the resident graph with the flips, as the calibrator ran it
            parts = wats._graph_features(cal.graph, 3, scales, None, 2.0, False, True, flips)
        else:                          # a graph rebuilt from the tensor
            parts = egnn.graph_wavelet_features(torch.tensor(pert, device="cuda"), k=3, s=scales, normalize=False,
                                                return_parts=True)
    comb = parts.combined.clone().requires_grad_()
    feats = wats._L1Normalize.apply(comb).flatten(1)
    logits = cal.base_model(cal.x, leaf2)
    t = torch.log(torch.exp(cal.net(feats).squeeze()) + 1.1)
    (G * torch.log_softmax(logits / t.unsqueeze(1), dim=1)).sum().backward()
    dA, _ = adjacency_vjp(pert, 3, scales, None, 2.0, False, None, Cbar=comb.grad.double().cpu().numpy())
    base_term = 0.0 if leaf2.grad is None else leaf2.grad.double().cpu().numpy()
    assert (leaf2.grad is None) == (model_name == "fixed")
    print(f"\n[WATS {n_flips} flips {model_name}] |wavelet term| {np.abs(dA).max():.2e}, "
          f"|base term| {np.abs(base_term).max():.2e}")
    report(f"WATS {n_flips} flips {model_name} leaf gradient", leaf.grad.cpu().numpy(), base_term + dA, 1e-5)
    # with the option off the leaf gets the base model's term only
    cal.adjacency_grad = False
    leaf3 = torch.tensor(pert, device="cuda", requires_grad=True)
    assert cal.features_for(leaf3).grad_fn is None
    (G * cal(cal.x, leaf3)).sum().backward()
    if model_name == "fixed":
        assert leaf3.grad is None
    else:
        assert torch.equal(leaf3.grad, leaf2.grad)
