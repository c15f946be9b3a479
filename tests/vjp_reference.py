"""Reference gradient of the wavelet pass (test infrastructure only), built on the
float64 forward of ``oracle.wats_oracle``: what the GPU backward is checked against."""
import numpy as np

from oracle import wats_oracle as orc


def wavelet_vjp(adj, k, s, x0, lambda_max, normalize, Hbar, Cbar=None, Tbar=None):
    """Reference gradient of the wavelet pass, float64: ``(Xbar, sbar)`` for the loss
    ``<Hbar, features> + <Cbar, combined> + sum_k <Tbar_k, T_k>``.

    ``Hbar`` is ``[N, S*F]`` (the layout of the features; None: zero), ``Cbar``
    ``[N, S, F]``, ``Tbar`` ``[K+1, N, F]``; ``normalize`` says whether the
    features are row-L1-normalised.  A direct sum over the explicit transposed
    operator ``rescaled_laplacian(adj).T``, not the Clenshaw recurrence:
    ``Xbar = sum_k T_k(M^T) v_k`` with ``v_k = sum_s alpha[s,k] Cbar_s + Tbar_k``,
    and ``sbar_j = -sum_k k alpha[j,k] <Cbar_j, T_k>``.  ``sbar`` has one entry per scale."""
    parts = orc.wavelet_parts(adj, k, s, x0, lambda_max)
    mt = orc.rescaled_laplacian(adj, lambda_max).T.tocsr()
    alpha = parts["alpha"]
    n_scales = alpha.shape[0]
    n, f = parts["X0"].shape
    cb = np.zeros((n, n_scales, f)) if Cbar is None else np.array(Cbar, dtype=np.float64).reshape(n, n_scales, f)
    if Hbar is not None:
        hb = np.asarray(Hbar, dtype=np.float64).reshape(n, n_scales, f)
        for j in range(n_scales):
            if normalize:
                c, h = parts["S"][j], parts["H"][j]
                r = np.abs(c).sum(axis=1, keepdims=True) + 1e-8
                dot = (hb[:, j, :] * h).sum(axis=1, keepdims=True)
                cb[:, j, :] += (hb[:, j, :] - np.sign(c) * dot) / r
            else:
                cb[:, j, :] += hb[:, j, :]
    xbar = np.zeros((n, f))
    for i in range(k + 1):
        v = sum(alpha[j, i] * cb[:, j, :] for j in range(n_scales))
        if Tbar is not None:
            v = v + np.asarray(Tbar[i], dtype=np.float64).reshape(n, f)
        xbar += orc.chebyshev_orders(mt, i, v)[i]        # T_i(M^T) v_i
    sbar = np.array([-sum(i * alpha[j, i] * float((cb[:, j, :] * parts["T"][i]).sum()) for i in range(k + 1))
                     for j in range(n_scales)])
    return xbar, sbar
