"""Dense float64 GP posterior (Cholesky), the reference the prediction tests compare against.

Built on the oracle kernel of `oracle/operators.py` (its scaling, the reference's expanded squared distance and
the `eps` under the Matérn square root), so it shares the device's kernel formula entry for entry.  The
reference takes `eps` of the working dtype; `eps=` selects it (float32 for an fp32 run), while the arithmetic
stays float64:

    mean = c + K(X*, X) (K + s I)^{-1} (y - c)
    var  = k(x*, x*) - diag(K(X*, X) (K + s I)^{-1} K(X, X*))   (latent: no noise term)
"""

import numpy as np
import scipy.linalg

from oracle import operators as oracle_ops


EPS64 = float(np.finfo(np.float64).eps)


def _kernel(kind, s2, sigma, eps):
    """`oracle_ops.GramOperator._block`'s kernel of the clamped squared distance, with `eps` given."""
    if kind == "rbf":
        return sigma * np.exp(-s2 / 2)
    s = np.sqrt(s2 + eps)
    return sigma * (1 + s) * np.exp(-s) if kind == "matern32" else sigma * np.exp(-s)


def kernel_matrix(kind, raw_ls, raw_os, A, B, eps=EPS64):
    """K(A, B) in float64 with the oracle's formula (both point sets scaled by the same lengthscales)."""
    ga, gb = oracle_ops.GramOperator(np.asarray(A, np.float64), kind), oracle_ops.GramOperator(np.asarray(B, np.float64), kind)
    xa, _, _ = ga._scaled(np.asarray(raw_ls, np.float64))
    xb, _, _ = gb._scaled(np.asarray(raw_ls, np.float64))
    sigma = oracle_ops.softplus(np.asarray(raw_os, np.float64))
    if eps == EPS64:
        return ga._block(xa, xb, sigma)[0]
    s2 = np.maximum(0.0, np.einsum("id,id->i", xa, xa)[:, None] + np.einsum("jd,jd->j", xb, xb)[None, :] - 2.0 * (xa @ xb.T))
    return _kernel(kind, s2, sigma, eps)


def prior_diag(kind, raw_os, m, eps=EPS64):
    """k(x, x): the kernel formula at s2 = 0."""
    sigma = float(oracle_ops.softplus(np.asarray(raw_os, np.float64)))
    return np.full(m, _kernel(kind, 0.0, sigma, eps))


def posterior(kind, X, y, X_test, *, raw_ls, raw_os, noise, const, eps=EPS64):
    """(mean, latent variance, alpha) at X_test."""
    K = kernel_matrix(kind, raw_ls, raw_os, X, X, eps)
    np.fill_diagonal(K, prior_diag(kind, raw_os, len(X), eps))  # s2 = 0 exactly on the diagonal, as on the device
    Kx = kernel_matrix(kind, raw_ls, raw_os, X_test, X, eps)
    cf = scipy.linalg.cho_factor(K + noise * np.eye(len(X)))
    alpha = scipy.linalg.cho_solve(cf, np.asarray(y, np.float64) - const)
    V = scipy.linalg.cho_solve(cf, Kx.T)
    var = prior_diag(kind, raw_os, len(X_test), eps) - np.einsum("tj,jt->t", Kx, V)
    return const + Kx @ alpha, var, alpha
