"""Closed forms of approximate leave-one-out cross-validation (``ObservationInfluence.approximate_cv``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  numpy, float64: h_n = x_n^T H^{-1} x_n, leverage s_n h_n,
the IJ predictor z_n + w_n r_n h_n, the Newton-step predictor z_n + w_n r_n h_n / (1 - s_n h_n) (NaN where
s_n h_n >= 1 - 2^-40), the held-out losses and their weighted mean; and, to check those closed forms, one Newton
step from theta_hat on the objective without row n and the exact leave-one-out prediction.  ``quad_forms_ld``
states h_n in longdouble (``highprec``) to measure forward errors.
"""
import numpy as np

from . import models
from .highprec import LD, cholesky_ld, solve_lower_ld


NS_SINGULAR = 1.0 - 2.0 ** -40


def quad_forms(X, H):
    """h_n = x_n^T H^{-1} x_n by a dense solve."""
    return np.einsum('nd,dn->n', X, np.linalg.solve(H, X.T))


def loo(X, y, w, theta, family='logistic', l2=0.0):
    """dict(h, leverage, z_ij, z_ns) of the closed forms at theta (the optimum)."""
    cf = models.glm_closed_form(X, y, theta, w, family, l2)
    h = quad_forms(X, cf['hessian'])
    lev = cf['s'] * h
    step = w * cf['r'] * h
    with np.errstate(divide='ignore', invalid='ignore'):
        z_ns = np.where(lev < NS_SINGULAR, cf['z'] + step / (1.0 - lev), np.nan)
    return dict(h=h, leverage=lev, z_ij=cf['z'] + step, z_ns=z_ns)


def glm_loss(z, y, family='logistic'):
    """Negative log-likelihood of y at z up to terms in y only."""
    if family == 'logistic':
        return np.maximum(z, 0.0) + np.log1p(np.exp(-np.abs(z))) - y * z
    if family == 'poisson':
        return np.exp(z) - y * z
    if family == 'gaussian':
        return 0.5 * (y - z) ** 2
    raise ValueError(family)


def mean_loss(loss, w, invalid):
    """(sum w loss / sum w over the rows with w != 0 and not invalid, number of invalid rows)."""
    keep = (w != 0) & ~invalid
    return float(np.sum(w[keep] * loss[keep]) / np.sum(w[keep])), int(np.sum(invalid))


def newton_step_without(X, y, w, theta, n, family='logistic', l2=0.0):
    """x_n^T of one Newton step from theta on the objective with the weight of row n set to zero."""
    w0 = np.array(w, dtype=np.float64)
    w0[n] = 0.0
    cf = models.glm_closed_form(X, y, theta, w0, family, l2)
    return float(X[n] @ (theta - np.linalg.solve(cf['hessian'], cf['grad'])))


def exact_loo(X, y, w, n, family='logistic', l2=0.0):
    """x_n^T theta_hat_{-n}: the optimum without row n, by Newton on the reduced data."""
    keep = np.arange(X.shape[0]) != n
    return float(X[n] @ models.glm_newton(X[keep], y[keep], np.asarray(w)[keep], family, l2))


def quad_forms_ld(H, X):
    """h_n = |L^{-1} x_n|^2 = x_n^T H^{-1} x_n in longdouble (H = L L^T), for the rows of X."""
    L = cholesky_ld(H)
    U = solve_lower_ld(L, np.asarray(X, dtype=LD).T)
    return np.sum(U * U, axis=0)
