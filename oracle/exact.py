"""Integer-valued designs on which every FP64-grade engine must be EXACT.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  With integer X (|x| <= 2^7), weights that are squares of
small integers (sqrt(s) <= 2^4), small-integer residuals (|r| <= 2^3) and a small-integer stand-in for H^{-1}
(|h| <= 2^3), every product and every partial sum of

    H = X^T diag(s) X          (N <= 2^18 observations)
    S = -Hinv (diag(r) X)^T    (D <= 2^13 features)

is an integer below 2^53, so float64 arithmetic in ANY order gives the exact result.  The INT8 slicing engine is
exact on them too: an operand row of integers of at most 12 bits (sqrt(s) |x| <= 2^11, |h| <= 2^3, |x| <= 2^7) has,
against its power-of-two scale, at most two non-zero balanced base-256 digits, so no digit pair the engine drops is
non-zero, and the residuals enter as a factor of the power-of-two column scale.  A misplaced chunk, tile, digit or
row then shows as a gross error instead of one of 1e-13.
"""
import numpy as np

XMAX = 2 ** 7          # |x_nk|
SQMAX = 2 ** 4         # sqrt(s_n)
RMAX = 2 ** 3          # |resid_n|
HMAX = 2 ** 3          # |Hinv_ij|
MAX_N = 2 ** 18        # observations of a Hessian assembly
MAX_D = 2 ** 13        # features of an apply
EXACT_LIMIT = 2 ** 53


def integer_design(seed, n, d, vmax=XMAX):
    """(n, d) float64 matrix of integers in [-vmax, vmax]."""
    rng = np.random.default_rng(seed)
    return rng.integers(-vmax, vmax + 1, size=(n, d), dtype=np.int64).astype(np.float64)


def square_weights(seed, n, sqmax=SQMAX):
    """(n,) weights k^2, k in [0, sqmax] (zeros included): sqrt(s) is an integer."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, sqmax + 1, size=n, dtype=np.int64)
    return (k * k).astype(np.float64)


def integer_vector(seed, n, vmax=RMAX):
    rng = np.random.default_rng(seed)
    return rng.integers(-vmax, vmax + 1, size=n, dtype=np.int64).astype(np.float64)


def hessian_bound(n):
    """Largest |partial sum| of X^T diag(s) X over n observations."""
    return n * XMAX * XMAX * SQMAX * SQMAX


def apply_bound(d):
    """Largest |partial sum| of Hinv (diag(r) X)^T over d features."""
    return d * HMAX * XMAX * RMAX


def weighted_gram_int(X, s):
    """X^T diag(s) X in Python integers (object arrays: no rounding, no overflow)."""
    Xi = X.astype(np.int64).astype(object)
    si = s.astype(np.int64).astype(object)
    return (Xi * si[:, None]).T.dot(Xi)


def apply_int(Hinv, X, r):
    """-Hinv (diag(r) X)^T in Python integers."""
    Hi = Hinv.astype(np.int64).astype(object)
    G = (X.astype(np.int64).astype(object) * r.astype(np.int64).astype(object)[:, None]).T
    return -Hi.dot(G)
