"""The reference adjacency gradient (``tests/adjacency_reference.adjacency_vjp``) against central
finite differences of a float64 forward, and that forward against the oracle.  No GPU needed.

The oracle rounds the Laplacian entries to float32 (``normalized_laplacian_parts``), so finite
differences through it are quantised; ``forward64`` restates the pass in float64 and is checked to
agree with the oracle to float32 rounding.  Covered: stored, unstored and diagonal entries; the
default signal (which depends on the adjacency through ``log1p`` of the row sums) and a custom one;
with and without the L1 normalisation; several scales; ``lambda_max != 2``; a weighted directed
graph, a graph with self loops and a graph with an isolated node and an empty row.

Isolated-node convention: ``w^-1/2`` has no derivative at ``w = 0``, so the gradient holds an
isolated node's ``d`` at 1.  The unstored off-diagonal entries of an isolated node's column are the
only entries that convention affects; they are the only entries left out of the finite differences.
"""
import numpy as np
import pytest
import scipy.sparse as sp

from oracle import wats_oracle as orc
from adjacency_reference import adjacency_vjp, forward64
from helpers import load_case


def isolated_graph():
    """7 weighted directed nodes plus node 7 with no in-edge (isolated: its column is empty) that
    still has out-edges, and node 3 with an empty row; one self loop."""
    rng = np.random.default_rng(21)
    n = 8
    A = np.zeros((n, n))
    for i, j in [(0, 1), (1, 0), (1, 2), (2, 4), (4, 1), (5, 6), (6, 5), (2, 3), (4, 5), (6, 0), (0, 6),
                 (7, 2), (7, 5), (5, 5)]:
        A[i, j] = 0.5 + rng.random()
    return sp.csr_matrix(A)


def graph(name):
    if name == "isolated":
        return isolated_graph(), 3
    case = load_case(name)
    return case["adj"], case["k"]


def loss(A, k, s, x0, lam, normalize, hb, cb, tb):
    p = forward64(A, k, s, x0, lam)
    n, f = p["X0"].shape
    feats = np.stack(p["H"] if normalize else p["S"], axis=1).reshape(n, -1)
    val = float((hb * feats).sum()) + float((cb * np.stack(p["S"], axis=1)).sum())
    return val + sum(float((tb[i] * p["T"][i]).sum()) for i in range(k + 1))


@pytest.mark.parametrize("name", ["kat_path_loops", "directed_weighted", "isolated"])
def test_float64_forward_matches_the_oracle(name):
    adj, k = graph(name)
    rng = np.random.default_rng(1)
    for x0 in (None, rng.standard_normal((adj.shape[0], 2))):
        p = forward64(adj, k, [0.8, 1.5], x0, 1.7)
        q = orc.wavelet_parts(adj, k, [0.8, 1.5], x0, 1.7)
        for a, b in zip(p["T"], q["T"]):
            assert np.abs(a - b).max() <= 1e-6 * max(1.0, np.abs(b).max())


CASES = [
    # name, F (None: default signal), scales, lambda_max, normalize
    ("kat_path_loops", None, [0.8], 2.0, False),
    ("kat_path_loops", 2, [0.8, 1.6], 1.7, True),
    ("directed_weighted", None, [0.8], 1.7, False),
    ("directed_weighted", 3, [0.4, 1.1, 2.0], 1.7, True),
    ("directed_weighted", 1, [0.8], 2.0, False),
    ("isolated", None, [0.8, 1.3], 1.7, False),
    ("isolated", 2, [0.8], 2.5, True),
]


@pytest.mark.parametrize("name,f,scales,lam,normalize", CASES)
def test_adjacency_vjp_matches_finite_differences(name, f, scales, lam, normalize):
    adj, k = graph(name)
    A = adj.toarray().astype(np.float64)
    n = A.shape[0]
    rng = np.random.default_rng(5)
    x0 = None if f is None else rng.standard_normal((n, f))
    fw = 1 if f is None else f
    S = len(scales)
    hb = rng.standard_normal((n, S * fw))
    cb = rng.standard_normal((n, S, fw))
    tb = rng.standard_normal((k + 1, n, fw))
    dA, dlam = adjacency_vjp(adj, k, scales, x0, lam, normalize, hb, cb, tb)
    assert dA.shape == (n, n)
    p = forward64(A, k, scales, x0, lam)
    skip = p["iso"][None, :] & (A == 0) & ~np.eye(n, dtype=bool)      # the isolated-node convention
    stored = list(zip(*np.nonzero((A != 0) & ~np.eye(n, dtype=bool))))
    unstored = list(zip(*np.nonzero((A == 0) & ~np.eye(n, dtype=bool) & ~skip)))
    diag = [(i, i) for i in range(n)]
    if n > 16:            # a seeded spread of each kind on the larger graphs
        pick = lambda lst, m: [lst[i] for i in rng.choice(len(lst), size=min(m, len(lst)), replace=False)]  # noqa: E731
        stored, unstored, diag = pick(stored, 24), pick(unstored, 24), pick(diag, 8)
    assert stored and unstored and diag
    eps = 1e-6
    scale = max(1.0, np.abs(dA).max())
    for kind, entries in (("stored", stored), ("unstored", unstored), ("diagonal", diag)):
        for i, j in entries:
            ap, am = A.copy(), A.copy()
            ap[i, j] += eps
            am[i, j] -= eps
            fd = (loss(ap, k, scales, x0, lam, normalize, hb, cb, tb) -
                  loss(am, k, scales, x0, lam, normalize, hb, cb, tb)) / (2 * eps)
            assert abs(fd - dA[i, j]) <= 2e-6 * scale, (kind, i, j, fd, dA[i, j])
    fd = (loss(A, k, scales, x0, lam + eps, normalize, hb, cb, tb) -
          loss(A, k, scales, x0, lam - eps, normalize, hb, cb, tb)) / (2 * eps)
    assert abs(fd - dlam) <= 1e-6 * max(1.0, abs(fd)), (fd, dlam)


def test_isolated_convention_entries_exist():
    """The isolated graph does exercise the convention: node 7's column is empty but its row is not."""
    adj, _ = graph("isolated")
    p = forward64(adj, 3, 0.8, None, 2.0)
    assert p["iso"][7] and adj[7].nnz > 0 and adj[3].nnz == 0
