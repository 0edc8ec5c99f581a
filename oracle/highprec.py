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


# ----------------------------------------------------------------------------------------------------------------
# The per-observation GMM-VB assembly of ``gmm_blocks`` (csrc/blockchol.cu).  Observation n, logits l = [rho_n, 0],
# r = softmax(l), c_k = |x_n - m_k|^2 / 2 - log pi_k, a_k = c_k + log r_k, abar = sum_k r_k a_k, delta_k = a_k - abar:
#   B[j][l] = r_j d_jl (delta_j + 1) - r_j r_l (delta_j + delta_l + 1)      j, l < K-1
#   coef[j][k] = r_j (d_jk - r_k)       (the cross block is coef[j][k] (m_k[t] - x_n[t]))
#   grad_rho_j = r_j delta_j,  obj = abar
# When one responsibility r_dom is close to 1, B_dom,dom, coef_dom,dom and delta_dom are (1 - r_dom)-small, but
# these formulas form them as differences of O(1) numbers: in float64 every digit is lost once the gap between the
# two largest logits passes ~37 (longdouble: ~44).  gmm_blocks_mp evaluates the formulas as written at a precision
# that absorbs the cancellation; gmm_blocks_stable_ld uses forms that do not cancel.
# ----------------------------------------------------------------------------------------------------------------
def _gmm_logits(rho):
    rho = np.asarray(rho, dtype=np.float64)
    return np.concatenate([rho, np.zeros((rho.shape[0], 1))], axis=1)


def gmm_blocks_mp(X, m, rho, log_pi, rows):
    """r, grad_rho, obj_terms, blocks and coef of the observations ``rows`` from the definition, in mpmath, each
    rounded once to float64.  The inputs are taken as the exact float64 values.  The working precision is 50 digits
    plus what the cancellation of 1 - r_dom costs, (top-two logit gap + log(1 + max|c|)) / ln 10."""
    X, m, log_pi = (np.asarray(a, dtype=np.float64) for a in (X, m, log_pi))
    logits = _gmm_logits(rho)
    K, d = m.shape
    M = K - 1
    out = dict(r=np.empty((len(rows), K)), grad_rho=np.empty((len(rows), M)), obj_terms=np.empty(len(rows)),
               blocks=np.empty((len(rows), M, M)), coef=np.empty((len(rows), M, K)))
    for i, n in enumerate(rows):
        top2 = np.sort(logits[n])[-2:]
        csize = float(np.max(np.abs(0.5 * ((X[n] - m) ** 2).sum(1) - log_pi)))
        digits = 50 + int((top2[1] - top2[0] + math.log1p(csize)) / math.log(10)) + 1
        with mpmath.workdps(digits):
            mpf = mpmath.mpf
            lg = [mpf(float(v)) for v in logits[n]]
            mx = max(lg)
            e = [mpmath.exp(v - mx) for v in lg]
            tot = mpmath.fsum(e)
            r = [v / tot for v in e]
            c = [mpmath.fsum((mpf(float(X[n, t])) - mpf(float(m[k, t]))) ** 2 for t in range(d)) / 2
                 - mpf(float(log_pi[k])) for k in range(K)]
            a = [c[k] + (lg[k] - mx - mpmath.log(tot)) for k in range(K)]
            abar = mpmath.fsum(r[k] * a[k] for k in range(K))
            dev = [a[k] - abar for k in range(K)]
            out['r'][i] = [_to_f64(v) for v in r]
            out['grad_rho'][i] = [_to_f64(r[j] * dev[j]) for j in range(M)]
            out['obj_terms'][i] = _to_f64(abar)
            for j in range(M):
                for l in range(M):
                    v = -r[j] * r[l] * (dev[j] + dev[l] + 1)
                    out['blocks'][i, j, l] = _to_f64(v + r[j] * (dev[j] + 1) if j == l else v)
                for k in range(K):
                    out['coef'][i, j, k] = _to_f64(r[j] * ((1 if j == k else 0) - r[k]))
    return out


def gmm_blocks_stable_ld(X, m, rho, log_pi):
    """The same quantities for every observation, in longdouble, in forms that do not cancel (dom = the first
    largest logit; every sum skips the term that is exactly zero):
        q_k = 1 - r_k = sum_{i != k} r_i
        delta_j = sum_i r_i [(c_j - c_i) + (l_j - l_i)]
        B_jj = r_j q_j + r_j delta_j (q_j - r_j),   B_jl = -r_j r_l (1 + delta_j + delta_l)
        coef_jk = r_j q_j (j = k),  -r_j r_k (j != k)
    Longdouble's exponent range also keeps e^-800 normal.  Returns float64 arrays of the outputs of gmm_blocks
    (coef in place of the cross blocks) and, for the error bars, the longdouble c, logits, q and delta."""
    X, m, log_pi = (np.asarray(a, dtype=np.float64) for a in (X, m, log_pi))
    lg = _gmm_logits(rho).astype(LD)
    N, K = lg.shape
    M = K - 1
    off = 1 - np.eye(K, dtype=LD)
    e = np.exp(lg - lg.max(1, keepdims=True))
    tot = e.sum(1, keepdims=True)
    r = e / tot
    q = (e @ off) / tot
    c = np.empty((N, K), dtype=LD)
    for k in range(K):
        c[:, k] = 0.5 * ((X.astype(LD) - m[k].astype(LD)) ** 2).sum(1) - LD(log_pi[k])
    diff = (c[:, :, None] - c[:, None, :]) + (lg[:, :, None] - lg[:, None, :])      # [n, j, i] = a_j - a_i
    delta = np.einsum('ni,nji->nj', r, diff)
    obj = (r * (c + lg - lg.max(1, keepdims=True) - np.log(tot))).sum(1)
    rj, qj, dj = r[:, :M], q[:, :M], delta[:, :M]
    blocks = -(rj[:, :, None] * rj[:, None, :]) * (1 + dj[:, :, None] + dj[:, None, :])
    idx = np.arange(M)
    blocks[:, idx, idx] = rj * qj + rj * dj * (qj - rj)
    coef = -(rj[:, :, None] * r[:, None, :])
    coef[:, idx, idx] = rj * qj
    f64 = lambda a: np.asarray(a, dtype=np.float64)                  # noqa: E731
    return dict(r=f64(r), grad_rho=f64(rj * dj), obj_terms=f64(obj), blocks=f64(blocks), coef=f64(coef),
                c=c, logits=lg, q=q, delta=delta)


GMM_EPS = 2.0 ** -53
GMM_FLOOR = 2.0 ** -1060


def gmm_error_bars(ref, d):
    """Per-entry error bars for gmm_blocks from a first-order error analysis (eps = 2^-53), given the output of
    gmm_blocks_stable_ld for data of dimension d:
        A_n = 1 + max_k |c_k| + max_k |l_k - max l|,   tau_n = 16 (d + K) eps A_n
        floors phi = 2^-1060,  phi_n = 4 phi A_n
        r_k: (8K + |l_k - max l|) eps r_k + phi    (exp amplifies the rounding of its argument l_k - max l)
        grad_rho_j: tau_n r_j q_j + phi_n,   obj: tau_n
        B_jj: tau_n r_j q_j (1 + |delta_j|) + phi_n,   B_jl: tau_n r_j r_l (1 + |delta_j| + |delta_l|) + phi_n
        coef_jk: tau_n |coef_jk| + phi_n     (times |m_k[t] - x_n[t]| for the cross block entry (j, k, t))
    Every bar scales with the entry's own size (r_j q_j, r_j r_l), never with the block's largest entry: a bar
    relative to max |B| is met by formulas that lose every digit of the (1 - r)-small entries.  Only the floors are
    absolute: a responsibility that underflowed to a subnormal or 0 is off by up to 2^-1074, and it is multiplied by
    deviations a_i - a_j of up to 2 A_n.  phi_n stays below 2^-1030, far under every (1 - r) of a gap up to 700."""
    c, lg = np.asarray(ref['c'], dtype=np.float64), np.asarray(ref['logits'], dtype=np.float64)
    r, q, dl = (np.asarray(ref[k], dtype=np.float64) for k in ('r', 'q', 'delta'))
    N, K = r.shape
    M = K - 1
    gap = lg.max(1, keepdims=True) - lg
    A = 1 + np.abs(c).max(1) + gap.max(1)
    tau = 16 * (d + K) * GMM_EPS * A
    t2 = tau[:, None, None]
    rj, qj, dj = r[:, :M], q[:, :M], np.abs(dl[:, :M])
    phi = 4 * GMM_FLOOR * A
    assert np.all(phi < 2.0 ** -1030), 'the underflow floor would cover (1 - r)-small entries'
    p2 = phi[:, None, None]
    blocks = t2 * (rj[:, :, None] * rj[:, None, :]) * (1 + dj[:, :, None] + dj[:, None, :]) + p2
    idx = np.arange(M)
    blocks[:, idx, idx] = tau[:, None] * rj * qj * (1 + dj) + phi[:, None]
    return dict(r=(8 * K + gap) * GMM_EPS * r + GMM_FLOOR, grad_rho=tau[:, None] * rj * qj + phi[:, None],
                obj_terms=tau, blocks=blocks, coef=t2 * np.abs(ref['coef']) + p2, tau=tau, floor=phi)


def gmm_bar_ratios(got, ref, bars, keys=('r', 'grad_rho', 'obj_terms', 'blocks', 'coef')):
    """Per observation, max |got - ref| / bar over the entries of each key (NaN in got gives inf)."""
    out = {}
    for k in keys:
        g = np.asarray(got[k], dtype=np.float64)
        ratio = np.abs(g - ref[k]) / bars[k]
        ratio = np.where(np.isnan(ratio), np.inf, ratio).reshape(g.shape[0], -1)
        out[k] = ratio.max(1)
    return out
