"""Closed forms of approximate leave-one-group-out cross-validation (``approximate_cv(groups=...)``), for the tests.

numpy, float64: for groups of consecutive rows R, Q = X_R H^{-1} X_R^T, the IJ predictor z_R + Q u and the
Newton-step predictor z_R + t + Q S^1/2 M^{-1} S^1/2 t; and, to check those closed forms, one Newton step from
theta_hat on the objective without a set of rows and the exact leave-group-out prediction.  The leave-one-out forms
they reduce to at groups of one row are ``oracle.loo``.
"""
import numpy as np

from oracle import models


def group_loo(X, y, w, theta, starts, family='logistic', l2=0.0):
    """dict(h, leverage, z_ij, z_ns) of the leave-one-group-out closed forms at theta (the optimum), for the groups
    of consecutive rows starts[g] .. starts[g+1]-1: with Q = X_R H^{-1} X_R^T, u = (w r)_R, S = diag(s_R) and
    t = Q u, z^IJ = z_R + t and z^NS = z_R + t + Q S^1/2 M^{-1} S^1/2 t for M = I - S^1/2 Q S^1/2 (NaN on the whole
    group when a squared pivot of the Cholesky factor of M is <= 2^-40)."""
    cf = models.glm_closed_form(X, y, theta, w, family, l2)
    Hinv = np.linalg.inv(cf['hessian'])
    N = X.shape[0]
    h, z_ij, z_ns = np.empty(N), np.empty(N), np.empty(N)
    u = w * cf['r']
    for a, b in zip(starts[:-1], starts[1:]):
        Q = X[a:b] @ Hinv @ X[a:b].T
        t = Q @ u[a:b]
        sq = np.sqrt(cf['s'][a:b])
        M = np.eye(b - a) - sq[:, None] * Q * sq[None, :]
        h[a:b] = np.diag(Q)
        z_ij[a:b] = cf['z'][a:b] + t
        piv = _ldl_pivots(M)
        if np.all(piv > 2.0 ** -40):
            z_ns[a:b] = cf['z'][a:b] + t + Q @ (sq * np.linalg.solve(M, sq * t))
        else:
            z_ns[a:b] = np.nan
    return dict(h=h, leverage=cf['s'] * h, z_ij=z_ij, z_ns=z_ns)


def _ldl_pivots(M):
    """The pivots of Gaussian elimination without pivoting of the symmetric M (the squared diagonal of its
    Cholesky factor)."""
    A = np.array(M, dtype=np.float64)
    m = A.shape[0]
    piv = np.empty(m)
    for j in range(m):
        piv[j] = A[j, j]
        if j + 1 < m:
            A[j + 1:, j + 1:] -= np.outer(A[j + 1:, j], A[j, j + 1:]) / A[j, j]
    return piv


def newton_step_without_rows(X, y, w, theta, rows, family='logistic', l2=0.0):
    """X_R of one Newton step from theta on the objective with the weights of the rows R set to zero."""
    w0 = np.array(w, dtype=np.float64)
    w0[rows] = 0.0
    cf = models.glm_closed_form(X, y, theta, w0, family, l2)
    return X[rows] @ (theta - np.linalg.solve(cf['hessian'], cf['grad']))


def exact_lgo(X, y, w, rows, family='logistic', l2=0.0):
    """X_R theta_hat_{-R}: the optimum without the rows R, by Newton on the reduced data."""
    keep = np.ones(X.shape[0], dtype=bool)
    keep[rows] = False
    return X[rows] @ models.glm_newton(X[keep], y[keep], np.asarray(w)[keep], family, l2)
