"""Reference gradient of the wavelet pass w.r.t. the adjacency and ``lambda_max`` (test
infrastructure only): a float64 restatement of the forward from the dense adjacency, and the dense
``dLoss/dA`` the GPU kernels are checked against.  The companion of ``vjp_reference.wavelet_vjp``
(same loss, same upstream-gradient conventions).  It is a module of its own because it needs a
different forward: ``wavelet_vjp`` is built on the oracle's forward, whose Laplacian entries are
rounded to float32, while the adjacency gradient is checked by finite differences in the adjacency,
which that rounding quantises; ``forward64`` below keeps the whole pass in float64."""
import numpy as np

from oracle import wats_oracle as orc


def forward64(adj, k, s, x0, lambda_max):
    """The wavelet pass restated in float64 end to end from the dense adjacency (the oracle rounds the
    Laplacian entries to float32, which quantises finite differences through it): ``dict(A, d, iso,
    M, X0, T, S, H, alpha)``.  Same semantics as ``orc.wavelet_parts``: ``w_j = sum_{i != j} A_ij``,
    ``d = w^-1/2`` (1 where ``w = 0``), ``L = I' - D A' D`` with the stored diagonal dropped and
    ``I'`` the non-isolated diagonal; ``X0 = log1p(row sums)`` (self loops counted) by default."""
    A = np.asarray(adj.toarray() if hasattr(adj, "toarray") else adj, dtype=np.float64)
    n = A.shape[0]
    off = A - np.diag(np.diag(A))
    w = off.sum(axis=0)
    iso = w == 0
    d = np.where(iso, 1.0, 1.0 / np.sqrt(np.where(iso, 1.0, w)))
    L = np.diag((~iso).astype(np.float64)) - d[:, None] * off * d[None, :]
    M = (2.0 / float(lambda_max)) * L - np.eye(n)
    x0 = np.log1p(A.sum(axis=1)).reshape(-1, 1) if x0 is None else np.asarray(x0, dtype=np.float64)
    if x0.ndim == 1:
        x0 = x0.reshape(-1, 1)
    T = [x0]
    if k > 0:
        T.append(M @ x0)
    for _ in range(2, k + 1):
        T.append(2 * M @ T[-1] - T[-2])
    alpha = orc.heat_coefficients(k, s)
    S = [sum(a[i] * T[i] for i in range(k + 1)) for a in alpha]
    H = [c / (np.abs(c).sum(axis=1, keepdims=True) + 1e-8) for c in S]
    return dict(A=A, d=d, iso=iso, M=M, X0=x0, T=T, S=S, H=H, alpha=alpha)


def adjacency_vjp(adj, k, s, x0, lambda_max, normalize, Hbar, Cbar=None, Tbar=None, with_scale=False):
    """Reference gradient w.r.t. the adjacency and ``lambda_max``, float64: ``(dA [N, N], dlam)`` for the
    loss of :func:`wavelet_vjp` (``x0 = None``: the default signal ``log1p(row sums)``, whose
    dependence on ``A`` is included).  Dense restatement of DESIGN.md section 11: the Clenshaw vectors
    ``lambda_k`` over the explicit ``M^T``, ``g_ij = sum_k m_k <d_i lambda_k[i], d_j T_{k-1}[j]>``,
    ``dA_ij = [i != j] (-a g_ij + gw_j) + grho_i`` with ``gw`` the degree term (0 for an isolated
    node: its ``d`` is held at 1) and ``grho`` the default signal's term;
    ``dlam = -(1/lambda_max) sum_k <lambda_k, T_k + T_{k-2} + m_k T_{k-1}>``.  ``with_scale``: also the
    size of that sum, ``(1/lambda_max) sum_k <|lambda_k|, |T_k| + |T_{k-2}| + m_k |T_{k-1}|>`` (the
    terms cancel to ``m_k <lambda_k, L T_{k-1}>``, small for a smooth signal: a float32 pass can only
    be held to a fraction of this size)."""
    p = forward64(adj, k, s, x0, lambda_max)
    A, d, iso, M, T, alpha = p["A"], p["d"], p["iso"], p["M"], p["T"], p["alpha"]
    n, f = p["X0"].shape
    n_scales = alpha.shape[0]
    cb = np.zeros((n, n_scales, f)) if Cbar is None else np.array(Cbar, dtype=np.float64).reshape(n, n_scales, f)
    if Hbar is not None:
        hb = np.asarray(Hbar, dtype=np.float64).reshape(n, n_scales, f)
        for j in range(n_scales):
            if normalize:
                c, h = p["S"][j], p["H"][j]
                r = np.abs(c).sum(axis=1, keepdims=True) + 1e-8
                dot = (hb[:, j, :] * h).sum(axis=1, keepdims=True)
                cb[:, j, :] += (hb[:, j, :] - np.sign(c) * dot) / r
            else:
                cb[:, j, :] += hb[:, j, :]
    v = [sum(alpha[j, i] * cb[:, j, :] for j in range(n_scales)) for i in range(k + 1)]
    if Tbar is not None:
        v = [v[i] + np.asarray(Tbar[i], dtype=np.float64).reshape(n, f) for i in range(k + 1)]
    lam = [np.zeros((n, f)) for _ in range(k + 3)]          # lam[i] = b_i, zero past K
    for i in range(k, 0, -1):
        lam[i] = v[i] + 2 * M.T @ lam[i + 1] - lam[i + 2]
    xbar = v[0] + (M.T @ lam[1] - lam[2] if k > 0 else 0.0)
    a = 2.0 / float(lambda_max)
    G = sum((1.0 if i == 1 else 2.0) * (d[:, None] * lam[i]) @ (d[:, None] * T[i - 1]).T for i in range(1, k + 1))
    G = np.zeros((n, n)) if k == 0 else G
    off = A - np.diag(np.diag(A))
    R = (off * G).sum(axis=1)
    Q = (off * G).sum(axis=0)
    gw = np.where(iso, 0.0, 0.5 * a * d * d * (R + Q))
    grho = xbar[:, 0] / (1.0 + A.sum(axis=1)) if x0 is None else np.zeros(n)
    dA = -a * G + gw[None, :]
    np.fill_diagonal(dA, 0.0)
    dA += grho[:, None]
    zero = np.zeros((n, f))
    dlam = -sum(float((lam[i] * (T[i] + (T[i - 2] if i >= 2 else zero) + (1.0 if i == 1 else 2.0) * T[i - 1])).sum())
                for i in range(1, k + 1)) / float(lambda_max)
    if not with_scale:
        return dA, dlam
    size = sum(float((np.abs(lam[i]) * (np.abs(T[i]) + (np.abs(T[i - 2]) if i >= 2 else zero) +
                                         (1.0 if i == 1 else 2.0) * np.abs(T[i - 1]))).sum())
               for i in range(1, k + 1)) / float(lambda_max)
    return dA, dlam, size
