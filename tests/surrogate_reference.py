"""Float64 restatement of the structure-gradient surrogate (``csrc/surrogate.cuh``) on the host.

The model is the two-layer row-normalised GCN of the kernel header, on a CSR adjacency plus a
delta list of edge flips (``A' = A + sum of flips``, repeated flips of one entry add):

    d_i = sum_j A'[i,j]  (0 -> 1: the row is "clamped" and takes no gradient through its degree)
    Z1 = D^-1 A' XW + b1,   H1 = relu(Z1),   H2 = D^-1 A' H1,   logits[t] = H2[t] W2^T + b2

and, for an upstream ``u = dLoss/dlogits[t]`` (v = u W2, q_i = A'[t,i] / d_t (v . relu'(Z1[i]))),

    dL/dA[t,m] = (v . H1[m] + q_t . XW[m] - s_t) / d_t,   s_t = v . H2[t] + q_t . (Z1[t] - b1)
    dL/dA[i,t] = (q_i . XW[t] - q_i . (Z1[i] - b1)) / d_i      (i != t; s_t and the second term
                                                              vanish on clamped rows)

Inputs are the float32 arrays the kernels receive (``XW = sur.xw``, ``b1``, ``W2``, ``b2``, the
CSR), promoted to float64, so any difference from the kernels is the kernels' own.  ``relu'(0)``
is 0, as in torch.  ReLU ties: where ``|Z1|`` is within the float32 rounding bound of 0 either
activation is admissible, and when the kernel's own ``Z1`` is given the reference takes its sign
there (``GcnReference.ties`` counts those entries).

Some outputs are identically zero while the float32 terms they are computed from are not: H2 of a
row whose entries were all cancelled by flips (the kernels add a flip after the stored entry it
cancels), and the row gradient of a one-node graph (row normalisation makes the logits invariant
to the scale of row t, so ``sum_m A[t,m] dL/dA[t,m] = 0``; with one node that is the whole row).
No relative bar applies to those; ``h2_terms`` and ``structure_grad_terms`` give the sums of the
absolute values of the terms, against which a float32 result is bounded by its rounding error.
"""
import numpy as np
import scipy.sparse as sp

EPS32 = 2.0 ** -24


def perturbed(adj, deltas=None):
    """``A + flips`` as float64 CSR (duplicates summed; explicit zeros kept, they change nothing)."""
    a = sp.csr_matrix(adj, dtype=np.float64, copy=True)
    if deltas is not None and len(deltas[0]):
        n = a.shape[0]
        r, c, v = (np.asarray(x) for x in deltas)
        a = (a + sp.csr_matrix((v.astype(np.float64), (r, c)), shape=(n, n))).tocsr()
    a.sum_duplicates()
    return a


def absolute_terms(adj, deltas=None):
    """``|A| + sum |flips|`` (float64 CSR) and the number of terms per row: what the kernels sum."""
    a = abs(sp.csr_matrix(adj, dtype=np.float64))
    count = np.diff(a.indptr).astype(np.int64)
    if deltas is not None and len(deltas[0]):
        n = a.shape[0]
        r, c, v = (np.asarray(x) for x in deltas)
        a = (a + sp.csr_matrix((np.abs(v).astype(np.float64), (r, c)), shape=(n, n))).tocsr()
        count += np.bincount(r, minlength=n)
    return a, count


class GcnReference:
    """Forward of the surrogate in float64; ``z1_kernel`` (float32 ``[N, H]``) resolves ReLU ties."""

    def __init__(self, adj, xw, b1, w2, b2, deltas=None, z1_kernel=None):
        self.a = perturbed(adj, deltas)
        self.a_abs, self.terms = absolute_terms(adj, deltas)
        self.xw = np.asarray(xw, np.float64)
        self.b1 = np.asarray(b1, np.float64)
        self.w2 = np.asarray(w2, np.float64)
        self.b2 = np.asarray(b2, np.float64)
        self.deg_raw = np.asarray(self.a.sum(axis=1)).ravel()
        self.clamped = self.deg_raw == 0
        self.deg = np.where(self.clamped, 1.0, self.deg_raw)
        agg = self.a @ self.xw
        self.z1 = agg / self.deg[:, None] + self.b1
        # float32 rounding bound of Z1: a sum of row_len + 1 products, a division and the bias
        row_len = np.diff(self.a.indptr)
        absagg = abs(self.a) @ np.abs(self.xw)
        bound = (row_len[:, None] + 4) * EPS32 * (absagg / self.deg[:, None] + np.abs(self.b1))
        self.active = self.z1 > 0
        self.ties = 0
        if z1_kernel is not None:
            tie = np.abs(self.z1) <= bound
            self.active = np.where(tie, np.asarray(z1_kernel) > 0, self.active)
            self.ties = int(tie.sum())
        self.h1 = np.where(self.active, self.z1, 0.0)

    def h2(self, t):
        row = self.a.getrow(t)
        return (row @ self.h1).ravel() / self.deg[t]

    def h2_terms(self, t):
        """(sum of |terms| of H2[t], number of terms): the float32 sum is within
        ``(count + 2) 2^-24`` of that sum."""
        return (self.a_abs.getrow(t) @ np.abs(self.h1)).ravel() / self.deg[t], int(self.terms[t])

    def logits(self, t):
        return self.h2(t) @ self.w2.T + self.b2

    def all_logits(self):
        return (self.a @ self.h1) / self.deg[:, None] @ self.w2.T + self.b2

    def a_tt(self, t):
        return float(self.a[t, t])

    def structure_grad(self, t, u):
        """(row t, column t) of dLoss/dA for ``u = dLoss/dlogits[t]`` (``[C]``)."""
        u = np.asarray(u, np.float64)
        v = u @ self.w2                                             # [H]
        d_t, clamp_t = self.deg[t], self.clamped[t]
        a_tt = self.a_tt(t)
        q_t = a_tt / d_t * np.where(self.active[t], v, 0.0)
        s_t = 0.0 if clamp_t else v @ self.h2(t) + q_t @ (self.z1[t] - self.b1)
        row = (self.h1 @ v + self.xw @ q_t - s_t) / d_t
        col = np.zeros(self.a.shape[0])
        r = self.a.getrow(t)
        i = r.indices
        q = (r.data / d_t)[:, None] * np.where(self.active[i], v, 0.0)        # q_i, one row per i
        own = np.where(self.clamped[i], 0.0, (q * (self.z1[i] - self.b1)).sum(axis=1))
        col[i] = (q @ self.xw[t] - own) / self.deg[i]
        col[t] = row[t]
        return row, col

    def structure_grad_terms(self, t, u):
        """Sums of |terms| of row and column t of dLoss/dA (same formulas, absolute values)."""
        u = np.abs(np.asarray(u, np.float64))
        v = u @ np.abs(self.w2)
        d_t = self.deg[t]
        q_t = abs(self.a_tt(t)) / d_t * np.where(self.active[t], v, 0.0)
        s_t = v @ np.abs(self.h2(t)) + q_t @ np.abs(self.z1[t] - self.b1)
        row = (np.abs(self.h1) @ v + np.abs(self.xw) @ q_t + s_t) / d_t
        col = np.zeros(self.a.shape[0])
        r = self.a_abs.getrow(t)
        i = r.indices
        q = (r.data / d_t)[:, None] * np.where(self.active[i], v, 0.0)
        col[i] = (q @ np.abs(self.xw[t]) + (q * np.abs(self.z1[i] - self.b1)).sum(axis=1)) / self.deg[i]
        col[t] = row[t]
        return row, col

    def flip_scores(self, row, col, t):
        """The attack's ranking ``(row + col) (1 - 2 A'[t, :])`` (calib_fga.py:880-881)."""
        return (row + col) * (1.0 - 2.0 * self.a.getrow(t).toarray().ravel())
