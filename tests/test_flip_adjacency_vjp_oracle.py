"""Gradient w.r.t. edge flips (DESIGN.md section 14), no GPU needed.

* The float64 reference ``adjacency_vjp`` of the dense flipped graph ``A' = A + delta`` against central
  differences w.r.t. the flip values: ``dLoss/dv_p = dLoss/dA'`` at ``(r_p, c_p)``.  Cases: an added
  entry, a removed stored entry, a weighted flip, a diagonal flip, a flip that isolates a node and
  two flips on one entry.
* The degree terms split as the library computes them: ``R`` and ``Q`` over the stored entries of ``A``
  plus the off-diagonal flips folded in list order equal ``R`` and ``Q`` of ``A'``.
* ``egnn_adj_grad_degree_flips`` refuses a bad flip list (more than 64, an index out of range, missing
  arrays) and a short workspace before anything is launched.  The device pointers are fakes that are
  never dereferenced: with a device present a passing check could reach a launch, so that test skips.
"""
import numpy as np
import pytest
import torch

from adjacency_reference import adjacency_vjp, forward64
from helpers import load_case


def base_graph():
    """12 weighted directed nodes; node 9 has exactly one in-edge (from 4), node 2 a self loop."""
    rng = np.random.default_rng(31)
    n = 12
    A = np.zeros((n, n))
    edges = [(0, 1), (1, 0), (1, 2), (2, 3), (3, 1), (4, 5), (5, 4), (5, 6), (6, 7), (7, 8), (8, 6), (4, 9),
             (9, 10), (10, 11), (11, 10), (3, 0), (6, 5), (2, 2)]
    for i, j in edges:
        A[i, j] = 0.5 + rng.random()
    return A


A0 = base_graph()

# name -> flips (rows, cols, vals) on A0
FLIPS = {
    "added": ([0, 7], [5, 2], [1.0, 1.0]),
    "removed_stored": ([3], [1], [-A0[3, 1]]),
    "weighted": ([3, 8], [8, 3], [0.37, -0.2]),
    "diagonal": ([5, 0], [5, 11], [0.8, 1.0]),
    "isolates_node": ([4, 9], [9, 1], [-A0[4, 9], 0.6]),          # column 9 loses its only in-edge
    "two_on_one_entry": ([6, 6, 2], [0, 0, 9], [0.4, 0.7, 1.0]),
}


def flipped(A, flips):
    Ap = A.copy()
    for r, c, v in zip(*flips):
        Ap[r, c] += v
    return Ap


def loss(A, k, s, x0, lam, normalize, hb, tb):
    p = forward64(A, k, s, x0, lam)
    n = p["X0"].shape[0]
    feats = np.stack(p["H"] if normalize else p["S"], axis=1).reshape(n, -1)
    return float((hb * feats).sum()) + sum(float((tb[i] * p["T"][i]).sum()) for i in range(k + 1))


@pytest.mark.parametrize("name", list(FLIPS))
@pytest.mark.parametrize("f,scales,normalize", [(None, [0.8, 1.6], False), (2, [0.8], True)])
def test_flip_gradient_matches_finite_differences(name, f, scales, normalize):
    flips = FLIPS[name]
    k, lam = 3, 1.8
    n = A0.shape[0]
    rng = np.random.default_rng(7)
    x0 = None if f is None else rng.standard_normal((n, f))
    fw = 1 if f is None else f
    hb = rng.standard_normal((n, len(scales) * fw))
    tb = rng.standard_normal((k + 1, n, fw))
    Ap = flipped(A0, flips)
    dA, _ = adjacency_vjp(Ap, k, scales, x0, lam, normalize, hb, None, tb)
    iso = forward64(Ap, k, scales, x0, lam)["iso"]
    eps = 1e-6
    checked = 0
    for p, (r, c, v) in enumerate(zip(*flips)):
        if iso[c] and r != c and Ap[r, c] == 0:
            # the isolated-node convention: w^-1/2 has no derivative at w = 0, d_c is held at 1
            assert name == "isolates_node"
            continue
        vp, vm = list(flips[2]), list(flips[2])
        vp[p] += eps
        vm[p] -= eps
        fd = (loss(flipped(A0, (flips[0], flips[1], vp)), k, scales, x0, lam, normalize, hb, tb) -
              loss(flipped(A0, (flips[0], flips[1], vm)), k, scales, x0, lam, normalize, hb, tb)) / (2 * eps)
        assert abs(fd - dA[r, c]) <= 2e-6 * max(1.0, np.abs(dA).max()), (name, p, fd, dA[r, c])
        checked += 1
    assert checked >= 1
    if name == "isolates_node":
        assert iso[9] and not forward64(A0, k, scales, x0, lam)["iso"][9]
    if name == "two_on_one_entry":           # duplicates each get the entry's value
        assert flips[0][0] == flips[0][1] and flips[1][0] == flips[1][1]


@pytest.mark.parametrize("name", list(FLIPS))
def test_degree_terms_split_into_stored_entries_and_flips(name):
    """``R_i = sum_{j != i} A'_ij g_ij`` is the stored sum over ``A`` plus ``v_p g_{r_p c_p}`` for every
    off-diagonal flip in list order, and the same for ``Q``; the degree vectors are those of ``A'``."""
    flips = FLIPS[name]
    Ap = flipped(A0, flips)
    n = A0.shape[0]
    G = np.random.default_rng(3).standard_normal((n, n))
    off = lambda M: M - np.diag(np.diag(M))           # noqa: E731
    R, Q = (off(A0) * G).sum(axis=1), (off(A0) * G).sum(axis=0)
    for r, c, v in zip(*flips):
        if r != c:
            R[r] += v * G[r, c]
            Q[c] += v * G[r, c]
    np.testing.assert_allclose(R, (off(Ap) * G).sum(axis=1), rtol=0, atol=1e-12)
    np.testing.assert_allclose(Q, (off(Ap) * G).sum(axis=0), rtol=0, atol=1e-12)


def test_golden_graph_flip_matches_the_dense_perturbed_reference():
    """On a golden graph the flip route and a fresh dense ``A'`` are one and the same function: the
    reference of ``A'`` at a removed entry is the finite difference w.r.t. that flip's value."""
    case = load_case("cora_noloop")
    A = case["adj"].toarray().astype(np.float64)
    i, j = map(int, np.argwhere(A > 0)[3])
    flips = ([i, 0], [j, 5], [-1.0, 1.0])
    k = case["k"]
    rng = np.random.default_rng(9)
    n = A.shape[0]
    hb, tb = rng.standard_normal((n, 3)), rng.standard_normal((k + 1, n, 1))
    dA, _ = adjacency_vjp(flipped(A, flips), k, [0.8, 0.4, 1.3], None, 2.0, False, hb, None, tb)
    eps = 1e-6
    up = loss(flipped(A, (flips[0], flips[1], [-1.0 + eps, 1.0])), k, [0.8, 0.4, 1.3], None, 2.0, False, hb, tb)
    dn = loss(flipped(A, (flips[0], flips[1], [-1.0 - eps, 1.0])), k, [0.8, 0.4, 1.3], None, 2.0, False, hb, tb)
    assert abs((up - dn) / (2 * eps) - dA[i, j]) <= 2e-6 * max(1.0, np.abs(dA).max())


# ---- the C ABI's refusals ------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.is_available(), reason="fake device pointers: must not reach a launch on a GPU")
def test_degree_flips_refusals_launch_nothing():
    from efficient_gnn_b200 import _cabi

    N = 8

    def ok(i):
        return (1 << 20) + 4096 * i          # 16-byte aligned fakes

    def flips(row=0, col=1, n=1):
        rows, cols = np.zeros(n, dtype=np.int32), np.ones(n, dtype=np.int32)
        rows[0], cols[0] = row, col
        vals = np.ones(n, dtype=np.float32)
        flips.keep = (rows, cols, vals)
        return rows.ctypes.data, cols.ctypes.data, vals.ctypes.data, n

    def too_many():
        return None, None, None, 65

    lib = _cabi.load()
    ws = int(lib.egnn_adj_grad_degree_ws_bytes(N))

    def call(d, ws_bytes=ws):
        return lib.egnn_adj_grad_degree_flips(ok(1), ok(2), None, ok(3), ok(4), None, ok(5), ok(6), N, 16, 4, 3, 1.0,
                                              ok(7), ok(8), None, None, *d, ok(9), ok(10), ok(11), ws_bytes, None)

    def error():
        return lib.egnn_last_error()

    assert call(too_many()) == -1 and b"n_delta" in error(), error()
    assert call((None, None, None, 1)) == -1 and b"delta arrays missing" in error(), error()
    for row, col in ((N, 0), (0, N), (-1, 0), (0, -1)):
        assert call(flips(row, col)) == -1 and b"delta index out of range" in error(), (row, col, error())
    assert call(flips(0, 1, n=64), ws - 1) == -4 and b"workspace too small" in error(), error()
    # a bad flip list is refused even when the workspace is short as well
    assert call(too_many(), ws - 1) == -1 and b"n_delta" in error(), error()
    # the flip-free entry point is the same call without flips
    assert lib.egnn_adj_grad_degree(ok(1), ok(2), None, ok(3), ok(4), None, ok(5), ok(6), N, 16, 4, 3, 1.0, ok(7),
                                    ok(8), None, None, ok(9), ok(10), ok(11), ws - 1, None) == -4
