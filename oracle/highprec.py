"""Extended-precision (x87 80-bit ``numpy.longdouble``, eps 1.1e-19) restatement of the infinitesimal-jackknife
solve, used to measure the FORWARD error of float64 algorithms on ill-conditioned Hessians.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Follows ``sensitivity_lib.py:226`` (``-hess_solver(cross)``)
with ``solver_lib.py:27-29`` (Cholesky factor + two triangular solves) in a wider type: neither the reference's
``cho_solve`` nor this build's kernels can be told apart at kappa(H) ~ 1e9 by comparing them with each other (both
carry ~kappa eps of forward error); against this oracle each one's own error is visible.

The second half states the GLM family functions (b^(k), residual, weight) in mpmath at a precision that grows with
|z|: the reference for the per-row arithmetic of ``glm.cu`` in both tails of the linear predictor.
"""
import math

import mpmath
import numpy as np

LD = np.longdouble


def cholesky_ld(H):
    """Lower Cholesky factor of a small SPD matrix in longdouble (column by column)."""
    H = np.array(H, dtype=LD)
    d = H.shape[0]
    L = np.zeros((d, d), dtype=LD)
    for j in range(d):
        v = H[j:, j] - L[j:, :j] @ L[j, :j]
        L[j:, j] = v / np.sqrt(v[0])
    return L


def solve_lower_ld(L, B, transpose=False):
    """L^{-1} B or L^{-T} B by substitution in longdouble."""
    d = L.shape[0]
    X = np.array(B, dtype=LD).reshape(d, -1).copy()
    if not transpose:
        for i in range(d):
            X[i] = (X[i] - L[i, :i] @ X[:i]) / L[i, i]
    else:
        for i in range(d - 1, -1, -1):
            X[i] = (X[i] - L[i + 1:, i] @ X[i + 1:]) / L[i, i]
    return X


def cholesky_ld_batched(B):
    """Lower Cholesky factors of a stack (G, M, M) of small SPD matrices in longdouble, column by column."""
    B = np.asarray(B, dtype=LD)
    M = B.shape[-1]
    L = np.zeros_like(B)
    for j in range(M):
        v = B[:, j:, j] - np.einsum('gik,gk->gi', L[:, j:, :j], L[:, j, :j])
        L[:, j:, j] = v / np.sqrt(v[:, :1])
    return L


def solve_lower_ld_batched(L, B, transpose=False):
    """L_g^{-1} B_g or L_g^{-T} B_g for stacks L (G, M, M) and B (G, M, K) by substitution in longdouble."""
    L = np.asarray(L, dtype=LD)
    X = np.array(B, dtype=LD)
    M = L.shape[-1]
    for i in (range(M - 1, -1, -1) if transpose else range(M)):
        s = (np.einsum('gk,gkc->gc', L[:, i + 1:, i], X[:, i + 1:]) if transpose else
             np.einsum('gk,gkc->gc', L[:, i, :i], X[:, :i]))
        X[:, i] = (X[:, i] - s) / L[:, i, i, None]
    return X


def block_arrow_residual_ld(sa, gi, blocks, cross, hgg, x, b, chunk_entries=1 << 23):
    """b - H x in longdouble for the block-arrow matrix H = [blockdiag(B_g) C; C^T Hgg] placed by the index arrays
    sa (G, M) and gi (Dg,), all float64 numpy arrays; x and b are (d, K).  The cross blocks are converted a chunk of
    blocks at a time, so a C of several GB needs no longdouble copy of itself."""
    x = np.asarray(x, dtype=LD)
    r = np.array(b, dtype=LD)
    G, M = sa.shape
    Dg = gi.shape[0]
    xl, xg = x[sa], x[gi]
    loc = np.empty(xl.shape, dtype=LD)
    glob = np.asarray(hgg, dtype=LD) @ xg
    step = max(1, chunk_entries // (M * max(Dg, 1)))
    for g0 in range(0, G, step):
        sl = slice(g0, g0 + step)
        Cc = np.asarray(cross[sl], dtype=LD)
        loc[sl] = np.asarray(blocks[sl], dtype=LD) @ xl[sl] + Cc @ xg
        glob += Cc.reshape(-1, Dg).T @ xl[sl].reshape(-1, x.shape[1])
    r[sa] -= loc
    r[gi] -= glob
    return r


def logistic_stats_ld(z, y, w):
    """(resid, s) = (sigma(z) - y, w sigma(z) sigma(-z)) of the logistic family in longdouble.  Both are evaluated at
    -|z|, where nothing cancels: 1 - sigma(z) is never formed, so the relative error does not grow like e^z."""
    z, y, w = (np.asarray(a, dtype=LD) for a in (z, y, w))
    e = np.exp(-np.abs(z))
    d = 1 + e
    pos = z >= 0
    sig_p = np.where(pos, 1 / d, e / d)              # sigma(z)
    sig_m = np.where(pos, e / d, 1 / d)              # sigma(-z)
    return (1 - y) * sig_p - y * sig_m, w * e / (d * d)


def logistic_ij_ld(X, y, theta, w, l2=0.0):
    """(H, S = -H^{-1} G^T) of the weighted logistic objective (ridge l2) in longdouble from float64 inputs."""
    X, y, theta, w = (np.asarray(a, dtype=LD) for a in (X, y, theta, w))
    z = X @ theta
    r, s = logistic_stats_ld(z, y, w)
    H = X.T @ (s[:, None] * X) + LD(l2) * np.eye(X.shape[1], dtype=LD)
    G = r[:, None] * X                             # d^2 f / d w_n d theta = (p_n - y_n) x_n
    L = cholesky_ld(H)
    S = -solve_lower_ld(L, solve_lower_ld(L, G.T), transpose=True)
    return H, S


# ----------------------------------------------------------------------------------------------------------------
# The GLM family functions in arbitrary precision (mpmath), independent of the float64 formulas under test.
# b(z) = softplus(z) (logistic), exp(z) (poisson), z^2 / 2 (gaussian).  The working precision is 40 digits plus
# |z| / ln 10, so that 1 - sigma(z) ~ e^-|z| is resolved to 40 digits up to |z| = 750; every value is rounded once to
# float64 (subnormals included).
# ----------------------------------------------------------------------------------------------------------------
def logistic_poly(k):
    """Integer coefficients c_0 .. c_k of P_k, b^(k)(z) = P_k(sigma(z)) for b = softplus:
    P_1(s) = s,  P_{k+1}(s) = P_k'(s) (s - s^2)  (sigma' = sigma - sigma^2)."""
    cur = [0, 1]
    for _ in range(1, k):
        nxt = [0] * (len(cur) + 1)
        for i in range(1, len(cur)):
            nxt[i] += i * cur[i]
            nxt[i + 1] -= i * cur[i]
        cur = nxt
    return cur


def _digits(z):
    return 40 + int(abs(z) / math.log(10)) + 1


def _to_f64(v):
    """mpf -> float64, rounded once (mpmath's float() would round subnormals twice)."""
    if mpmath.isnan(v) or mpmath.isinf(v) or abs(v) >= mpmath.ldexp(1, -1022):
        return float(v)
    return math.ldexp(float(mpmath.nint(mpmath.ldexp(v, 1074))), -1074)


def _bderiv(z, k, family):
    """b^(k)(z) as an mpf at the current working precision (z a finite float)."""
    z = mpmath.mpf(z)
    if family == 'logistic':
        sig = 1 / (1 + mpmath.exp(-z))
        return mpmath.polyval(logistic_poly(k)[::-1], sig)
    if family == 'poisson':
        return mpmath.exp(z)
    if family == 'gaussian':
        return z if k == 1 else (mpmath.mpf(1) if k == 2 else mpmath.mpf(0))
    raise ValueError(family)


def _elementwise(fn, *arrays):
    arrays = np.broadcast_arrays(*(np.asarray(a, dtype=np.float64) for a in arrays))
    out = np.empty(arrays[0].shape)
    for idx in np.ndindex(out.shape):
        args = [float(a[idx]) for a in arrays]
        if math.isnan(args[0]):
            out[idx] = math.nan
            continue
        with mpmath.workdps(_digits(args[0])):
            out[idx] = _to_f64(fn(*args))
    return out


def glm_bderiv_mp(z, k, family):
    """b^(k)(z), k = 1 .. 5, for float64 z (array), correctly rounded to float64."""
    if not 1 <= k <= 5:
        raise ValueError('k = 1 .. 5')
    return _elementwise(lambda zz: _bderiv(zz, k, family), z)


def glm_resid_mp(z, y, family):
    """b'(z) - y, correctly rounded to float64."""
    return _elementwise(lambda zz, yy: _bderiv(zz, 1, family) - mpmath.mpf(yy), z, y)


def glm_weight_mp(z, w, family):
    """s = w b''(z), correctly rounded to float64."""
    return _elementwise(lambda zz, ww: mpmath.mpf(ww) * _bderiv(zz, 2, family), z, w)
