"""Closed forms of the per-observation influence and the AMIP selection (``vittles_b200.influence_lib``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  numpy, float64:

    psi[k, n] = -resid_n x_n^T H^{-1} a_k          (the rows a_k^T S of the IJ matrix S = -H^{-1} G^T)

the greedy AMIP selection with the product's tie rule (largest score first, ties to the lower index, zero scores
never chosen) and its sequential float64 prefix sum, and Newton on the data with the dropped rows removed.
"""
import numpy as np

from . import models


def psi(X, y, w, theta, A, family='logistic', l2=0.0):
    """(K, N) influence of every observation on the K quantities of interest with gradients A (K, D) at theta."""
    cf = models.glm_closed_form(X, y, theta, w, family, l2)
    V = np.linalg.solve(cf['hessian'], np.atleast_2d(A).T)          # (D, K)
    return -(X @ V).T * cf['r'][None, :]


def amip_greedy(score, value, target, max_drop):
    """dict(n_drop, indices, predicted_value, max_change, direction) for the scores w_n psi_n (dropping A changes
    phi by -sum_{n in A} score_n)."""
    score = np.asarray(score, dtype=np.float64)
    sign = 1.0 if value >= target else -1.0
    key = sign * score
    cand = np.nonzero(key > 0)[0]
    order = cand[np.lexsort((cand, -key[cand]))][:max_drop]
    change = -np.cumsum(score[order])
    pred = value + change
    if value == target:
        n_drop = 0
    else:
        hit = np.nonzero(pred <= target if sign > 0 else pred >= target)[0]
        n_drop = int(hit[0]) + 1 if hit.size else None
    take = order.size if n_drop is None else n_drop
    return dict(n_drop=n_drop, indices=order[:take], predicted_value=float(pred[take - 1]) if take else float(value),
                max_change=float(change[-1]) if order.size else 0.0,
                direction='decrease' if sign > 0 else 'increase')


def refit(X, y, w, drop, family='logistic', l2=0.0):
    """The optimum on the data without the rows ``drop``."""
    keep = np.setdiff1d(np.arange(X.shape[0]), np.asarray(drop, dtype=np.int64))
    return models.glm_newton(X[keep], y[keep], w[keep], family, l2)
