"""The reference gradient of the wavelet pass (``tests/vjp_reference.wavelet_vjp``)
against central finite differences of the oracle's own forward, in float64:
w.r.t. the signal and the heat scales, with and without the row L1
normalisation, with upstream gradients on the features, the combination and
the orders.  No GPU needed."""
import numpy as np
import pytest

from oracle import wats_oracle as orc
from helpers import load_case
from vjp_reference import wavelet_vjp

CASES = [
    ("kat_path", [0.8], 1, 2.0),
    ("directed_weighted", [0.8], 1, 2.0),          # asymmetric, weighted: M^T != M
    ("directed_weighted", [0.4, 1.1, 2.0], 3, 1.7),  # several scales, F > 1, lambda_max != 2
]


def loss(adj, k, s, x0, lam, normalize, hb, cb, tb):
    p = orc.wavelet_parts(adj, k, s, x0, lam)
    n, f = p["X0"].shape
    feats = np.stack(p["H"] if normalize else p["S"], axis=1).reshape(n, -1)
    val = float((hb * feats).sum()) + float((cb * np.stack(p["S"], axis=1)).sum())
    return val + sum(float((tb[i] * p["T"][i]).sum()) for i in range(k + 1))


@pytest.mark.parametrize("normalize", [True, False])
@pytest.mark.parametrize("name,scales,f,lam", CASES)
def test_vjp_matches_finite_differences(name, scales, f, lam, normalize):
    case = load_case(name)
    adj, k, n = case["adj"], case["k"], case["n"]
    rng = np.random.default_rng(7)
    x0 = rng.standard_normal((n, f))
    S = len(scales)
    hb = rng.standard_normal((n, S * f))
    cb = rng.standard_normal((n, S, f))
    tb = rng.standard_normal((k + 1, n, f))
    xbar, sbar = wavelet_vjp(adj, k, scales, x0, lam, normalize, hb, cb, tb)
    assert xbar.shape == (n, f) and sbar.shape == (S,)
    eps = 1e-6
    # a spread of signal entries (every entry on the small graphs would be slow for no gain)
    idx = [(i, j) for i in rng.choice(n, size=min(n, 12), replace=False) for j in range(f)][:24]
    for i, j in idx:
        xp, xm = x0.copy(), x0.copy()
        xp[i, j] += eps
        xm[i, j] -= eps
        fd = (loss(adj, k, scales, xp, lam, normalize, hb, cb, tb) - loss(adj, k, scales, xm, lam, normalize, hb, cb, tb)) / (2 * eps)
        assert abs(fd - xbar[i, j]) <= 1e-6 * max(1.0, abs(fd)), (i, j, fd, xbar[i, j])
    for j in range(S):
        sp_, sm_ = list(scales), list(scales)
        sp_[j] += eps
        sm_[j] -= eps
        fd = (loss(adj, k, sp_, x0, lam, normalize, hb, cb, tb) - loss(adj, k, sm_, x0, lam, normalize, hb, cb, tb)) / (2 * eps)
        assert abs(fd - sbar[j]) <= 1e-6 * max(1.0, abs(fd)), (j, fd, sbar[j])


def test_vjp_only_cbar_is_the_adjoint_of_the_combination():
    """<Cbar, C(x)> = <Xbar, x> exactly (the pass is linear in the signal)."""
    case = load_case("directed_weighted")
    adj, k, n = case["adj"], case["k"], case["n"]
    rng = np.random.default_rng(3)
    x0 = rng.standard_normal((n, 2))
    cb = rng.standard_normal((n, 2, 2))
    p = orc.wavelet_parts(adj, k, [0.5, 1.5], x0)
    xbar, _ = wavelet_vjp(adj, k, [0.5, 1.5], x0, 2.0, False, None, cb)
    lhs = float((cb * np.stack(p["S"], axis=1)).sum())
    assert abs(lhs - float((xbar * x0).sum())) <= 1e-10 * max(1.0, abs(lhs))
