"""The float64 surrogate reference (``tests/surrogate_reference.GcnReference``) against float64 dense
torch autograd of the row-normalised GCN, the way the attack computes the structure gradient
(``gcn(x, adj_leaf)[[t]]``, ``autograd.grad(loss, adj_leaf)``, row and column ``t``).  No GPU needed.

The dense model is ``tests/models_for_tests.DenseGCN`` and, when ``ref_shim.reference_root()``
finds the reference, its own ``CompatibleGCN``; both in float64 in eval mode.  Covered: a clamped
target and a clamped neighbour, a directed graph (``A[i,t]`` unstored while ``A[t,i]`` is stored), a
stored self loop and a flip on ``(t, t)``, weights that cancel to a zero row sum (dyadic values, so
every summation order gives exactly 0), flips that add, remove and re-weight an entry, and a flip
that empties the target's row.  Agreement is at float64 rounding.
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from models_for_tests import DenseGCN
from oracle import ref_shim
from surrogate_reference import GcnReference

N, NFEAT, NHID, NCLASS = 14, 6, 8, 3
EMPTY, ZERO_SUM, LOOP, HUB = 3, 4, 5, 6          # node roles in the base graph


def base_graph():
    """Weighted directed graph: node EMPTY has no out-edge (clamped, but has in-edges); node
    ZERO_SUM has entries 0.5 (self loop), 0.25, -0.75 (row sum exactly 0: clamped with a non-empty
    row); node LOOP has a stored self loop; node HUB reaches both clamped nodes."""
    rng = np.random.default_rng(7)
    a = np.where(rng.random((N, N)) < 0.3, rng.uniform(0.5, 2.0, (N, N)), 0.0)
    np.fill_diagonal(a, 0.0)
    a[EMPTY, :] = 0.0
    a[ZERO_SUM, :] = 0.0
    a[ZERO_SUM, [ZERO_SUM, 1, 9]] = [0.5, 0.25, -0.75]
    a[LOOP, LOOP] = 1.25
    a[HUB, [EMPTY, ZERO_SUM, LOOP, 1, 2]] = [1.0, 0.75, 1.5, 0.5, 2.0]
    a[2, HUB] = 0.0                                    # HUB -> 2 stored, 2 -> HUB not: directed
    a[EMPTY, HUB] = 0.0
    return a


def flips(a, entries):
    """Delta list setting A[i, j] to the given values (adds, removes, re-weights)."""
    r, c, v = [], [], []
    for (i, j), val in entries:
        r.append(i); c.append(j); v.append(val - a[i, j])
    return r, c, v


def dense_models():
    out = [("DenseGCN", lambda: DenseGCN(NFEAT, NCLASS, nhid=NHID))]
    if ref_shim.reference_root() is not None:
        cls = ref_shim.load_reference()[1].CompatibleGCN
        out.append(("CompatibleGCN", lambda: cls(NFEAT, nhid=NHID, nclass=NCLASS)))
    return out


def apply_deltas(a, deltas):
    a = a.copy()
    if deltas is not None:
        for i, j, v in zip(*deltas):
            a[i, j] += v
    return a


CASES = {
    # name: (deltas as a function of the base graph, targets)
    "clamped_target_and_neighbour": (None, [EMPTY, HUB]),
    "directed": (None, [2, HUB]),
    "self_loop": (None, [LOOP]),
    "flip_on_diagonal": (lambda a: flips(a, [((HUB, HUB), 0.5), ((LOOP, LOOP), 0.0)]), [HUB, LOOP]),
    "zero_row_sum": (None, [ZERO_SUM, 1]),
    "add_remove_reweight": (lambda a: flips(a, [((HUB, 8), 1.0), ((HUB, LOOP), 0.0), ((HUB, 1), 1.75),
                                                 ((8, HUB), 1.0), ((1, 11), 0.5)]), [HUB, 8, 1]),
    "same_entry_twice": (lambda a: ([HUB, HUB], [2, 2], [-a[HUB, 2], 0.5]), [HUB, 2]),
    "empty_target_row": (lambda a: flips(a, [((HUB, j), 0.0) for j in np.nonzero(a[HUB])[0]]), [HUB]),
}


def kl_to_uniform(out):
    logp = F.log_softmax(out, dim=1)
    return F.kl_div(logp, torch.full_like(logp, 1.0 / logp.shape[1]), reduction="batchmean")


@pytest.mark.parametrize("model", [m[0] for m in dense_models()])
@pytest.mark.parametrize("case", sorted(CASES))
def test_reference_matches_float64_dense_autograd(case, model):
    make = dict(dense_models())[model]
    a0 = base_graph()
    mk, targets = CASES[case]
    deltas = None if mk is None else mk(a0)
    a = apply_deltas(a0, deltas)
    if case == "empty_target_row":
        assert not a[HUB].any()
    torch.manual_seed(3)
    gcn = make().double().eval()
    x = torch.randn(N, NFEAT, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    w1, b1 = gcn.gc1.weight.detach(), gcn.gc1.bias.detach()
    w2, b2 = gcn.gc2.weight.detach(), gcn.gc2.bias.detach()
    xw = (x @ w1.T).numpy()
    ref = GcnReference(a0, xw, b1.numpy(), w2.numpy(), b2.numpy(), deltas)
    assert ref.ties == 0
    leaf_all = torch.tensor(a)
    with torch.no_grad():
        full = gcn(x, leaf_all).numpy()
    assert np.abs(ref.all_logits() - full).max() <= 1e-12 * np.abs(full).max()
    u = np.random.default_rng(5).standard_normal(NCLASS)
    for t in targets:
        for loss_name in ("linear", "kl"):
            leaf = torch.tensor(a, requires_grad=True)
            out = gcn(x, leaf)[[t]]
            assert np.abs(ref.logits(t) - out.detach().numpy()[0]).max() <= 1e-12 * np.abs(full).max()
            if loss_name == "linear":
                loss, u_t = (out * torch.tensor(u)).sum(), u
            else:
                o = out.detach().requires_grad_(True)
                u_t = torch.autograd.grad(kl_to_uniform(o), o)[0].numpy()[0]
                loss = kl_to_uniform(out)
            g = torch.autograd.grad(loss, leaf)[0].numpy()
            row, col = ref.structure_grad(t, u_t)
            scale = max(np.abs(g[t]).max(), np.abs(g[:, t]).max())
            assert scale > 0
            assert np.abs(row - g[t]).max() <= 1e-12 * scale, (case, t, loss_name, "row")
            assert np.abs(col - g[:, t]).max() <= 1e-12 * scale, (case, t, loss_name, "column")
            score = ref.flip_scores(row, col, t)
            assert np.abs(score - (g[t] + g[:, t]) * (1 - 2 * a[t])).max() <= 3e-12 * scale


def test_case_table_exercises_what_it_names():
    a = base_graph()
    ref = GcnReference(a, np.ones((N, 4)), np.zeros(4), np.ones((2, 4)), np.zeros(2))
    assert ref.clamped[EMPTY] and ref.clamped[ZERO_SUM] and a[ZERO_SUM].any()
    assert a[HUB, EMPTY] and a[HUB, ZERO_SUM] and a[HUB, 2] and not a[2, HUB]
    assert a[LOOP, LOOP] and a[ZERO_SUM, ZERO_SUM]
