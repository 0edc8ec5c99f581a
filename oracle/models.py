"""Oracle-side model definitions: torch objectives for the generic autodiff path
and numpy closed forms for the benchmark families.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

The reference ships no model code (SURVEY.md section 7, "Configs 3 and 5 are
under-specified"); the objective families below are this build's definitions
(documented in DESIGN.md).  The infinitesimal-jackknife usage - hyperparameter
:= per-observation weights - follows the reference notebook
``docs/source/example_notebooks/mle_weight_sensitivity_example.ipynb:345-371``.
"""
import numpy as np
import torch

# --------------------------------------------------------------------------
# Counter-based synthetic data: numpy twin of vittles_b200/csrc/synth.cu.
# Integer-only up to one final multiply, so host and device agree bit for bit.
# --------------------------------------------------------------------------

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _mix64(x):
    """splitmix64 finaliser on uint64 arrays (wrapping arithmetic)."""
    with np.errstate(over='ignore'):
        x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        x = ((x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        x = ((x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return x ^ (x >> np.uint64(31))


_IH_STD = float(np.sqrt((65536.0 ** 2 - 1.0) / 3.0))   # std of a sum of four U{0..65535}


def synth_design(seed, row0, nrows, ncols, scale=None):
    """Rows ``row0 .. row0+nrows`` of the synthetic design matrix: entries are
    i.i.d. zero-mean, variance ``1/ncols`` (Irwin-Hall(4) of 16-bit lanes of a
    64-bit hash of ``(seed, row, col)``), i.e. ``X ~ N(0,1)/sqrt(D)`` to the
    accuracy that matters for conditioning (SURVEY.md section 8d)."""
    if scale is None:
        scale = 1.0 / (_IH_STD * np.sqrt(float(ncols)))
    rows = np.arange(row0, row0 + nrows, dtype=np.uint64)[:, None]
    cols = np.arange(ncols, dtype=np.uint64)[None, :]
    with np.errstate(over='ignore'):
        ctr = rows * np.uint64(ncols) + cols
        h = _mix64(ctr + _mix64(np.uint64(seed)))
    m = np.uint64(0xFFFF)
    s = ((h & m) + ((h >> np.uint64(16)) & m) + ((h >> np.uint64(32)) & m) + (h >> np.uint64(48))).astype(np.int64)
    return (s - 131070).astype(np.float64) * scale


def synth_uniform(seed, row0, nrows):
    """One U[0,1) per row (53-bit), for Bernoulli responses."""
    rows = np.arange(row0, row0 + nrows, dtype=np.uint64)
    with np.errstate(over='ignore'):
        h = _mix64(rows + _mix64(np.uint64(seed) ^ np.uint64(0xA5A5A5A5A5A5A5A5)))
    return (h >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def synth_theta(seed, ncols):
    """True parameter: entries ~ zero-mean unit-variance (same generator, row = 2^40)."""
    return synth_design(seed ^ 0x5EED, 1 << 40, 1, ncols, scale=1.0 / _IH_STD)[0]


def synth_logistic(seed, n, d, row0=0):
    """(X, y) for config 1/2: ``y ~ Bernoulli(sigmoid(X theta*))``."""
    X = synth_design(seed, row0, n, d)
    theta_star = synth_theta(seed, d)
    p = 1.0 / (1.0 + np.exp(-(X @ theta_star)))
    y = (synth_uniform(seed, row0, n) < p).astype(np.float64)
    return X, y, theta_star


# --------------------------------------------------------------------------
# GLM family: f(theta, w) = sum_n w_n * [ b(z_n) - y_n z_n ],  z = X theta
# --------------------------------------------------------------------------

def glm_objective(X, y, family='logistic', l2=0.0):
    """torch objective ``f(theta, w)`` for the generic autodiff oracle."""
    Xt = torch.as_tensor(np.asarray(X, dtype=np.float64))
    yt = torch.as_tensor(np.asarray(y, dtype=np.float64))

    def f(theta, w):
        z = Xt @ theta
        if family == 'logistic':
            b = torch.nn.functional.softplus(z)
        elif family == 'poisson':
            b = torch.exp(z)
        elif family == 'gaussian':
            b = 0.5 * z * z
        else:
            raise ValueError(family)
        return torch.sum(w * (b - yt * z)) + 0.5 * l2 * torch.sum(theta * theta)
    return f


def _sigmoid_pair(z):
    """(sigma(z), sigma(-z), b''(z) = sigma(z) sigma(-z)), all from e = exp(-|z|): 1 - sigma(z) is never formed, so
    nothing cancels in either tail (p (1 - p) loses e^z of its relative accuracy for z > 0)."""
    z = np.asarray(z, dtype=np.float64)
    e = np.exp(-np.abs(z))
    d = 1.0 + e
    pos = z >= 0
    return np.where(pos, 1.0 / d, e / d), np.where(pos, e / d, 1.0 / d), e / (d * d)


def glm_mean_var(z, family):
    """b'(z), b''(z)."""
    if family == 'logistic':
        p, _, var = _sigmoid_pair(z)
        return p, var
    if family == 'poisson':
        e = np.exp(z)
        return e, e
    if family == 'gaussian':
        return z, np.ones_like(z)
    raise ValueError(family)


def glm_resid(z, y, family):
    """b'(z) - y.  Logistic: (1 - y) sigma(z) - y sigma(-z), equal for every y and free of the cancellation of
    sigma(z) - 1 at y = 1."""
    if family == 'logistic':
        p, q, _ = _sigmoid_pair(z)
        return (1.0 - y) * p - y * q
    return glm_mean_var(z, family)[0] - y


def glm_closed_form(X, y, theta, w, family='logistic', l2=0.0):
    """Closed forms the CUDA kernels implement: gradient, Hessian
    ``X^T diag(w b''(z)) X`` and the (D, N) cross-Hessian whose column n is
    ``(b'(z_n) - y_n) x_n`` (the per-observation gradient)."""
    z = X @ theta
    var = glm_mean_var(z, family)[1]
    r = glm_resid(z, y, family)
    grad = X.T @ (w * r) + l2 * theta
    H = X.T @ ((w * var)[:, None] * X) + l2 * np.eye(X.shape[1])
    cross = (X * r[:, None]).T
    return dict(z=z, r=r, s=w * var, grad=grad, hessian=H, cross_hessian=cross)


def glm_newton(X, y, w, family='logistic', l2=0.0, iters=50, tol=1e-13):
    """Newton's method to the optimum (numpy)."""
    theta = np.zeros(X.shape[1])
    for _ in range(iters):
        cf = glm_closed_form(X, y, theta, w, family, l2)
        step = np.linalg.solve(cf['hessian'], cf['grad'])
        theta = theta - step
        if np.linalg.norm(step) < tol:
            break
    return theta


# --------------------------------------------------------------------------
# Config 5: GLM with a Gaussian prior whose precision and mean are the
# hyperparameter eps = (log tau, mu):
#   f(theta, eps) = sum_n [b(z_n) - y_n z_n] + 0.5 exp(eps0) ||theta - eps1||^2
# --------------------------------------------------------------------------

def hier_glm_objective(X, y, family='logistic'):
    Xt = torch.as_tensor(np.asarray(X, dtype=np.float64))
    yt = torch.as_tensor(np.asarray(y, dtype=np.float64))

    def f(theta, eps):
        z = Xt @ theta
        if family == 'logistic':
            b = torch.nn.functional.softplus(z)
        elif family == 'poisson':
            b = torch.exp(z)
        else:
            b = 0.5 * z * z
        return torch.sum(b - yt * z) + 0.5 * torch.exp(eps[0]) * torch.sum((theta - eps[1]) ** 2)
    return f


def hier_glm_newton(X, y, eps, family='logistic', iters=60, tol=1e-13):
    theta = np.zeros(X.shape[1])
    tau, mu0 = np.exp(eps[0]), eps[1]
    for _ in range(iters):
        z = X @ theta
        m, v = glm_mean_var(z, family)
        grad = X.T @ (m - y) + tau * (theta - mu0)
        H = X.T @ (v[:, None] * X) + tau * np.eye(X.shape[1])
        step = np.linalg.solve(H, grad)
        theta = theta - step
        if np.linalg.norm(step) < tol:
            break
    return theta


# --------------------------------------------------------------------------
# Config 3: Gaussian-mixture mean-field VB with per-observation local
# parameters.  x = (m (K*d), rho_1 .. rho_N (K-1 free logits each)).
#   r_n = softmax([rho_n, 0]);  c_nk = 0.5 ||x_n - m_k||^2 - log pi_k
#   f = sum_n sum_k r_nk (c_nk + log r_nk) + 0.5 * prior_prec * ||m||^2
# --------------------------------------------------------------------------

def gmm_vb_objective(Xobs, K, log_pi=None, prior_prec=1e-2):
    Xt = torch.as_tensor(np.asarray(Xobs, dtype=np.float64))
    N, d = Xt.shape
    lp = torch.zeros(K, dtype=torch.float64) - np.log(K) if log_pi is None else torch.as_tensor(log_pi)

    def f(x):
        m = x[:K * d].reshape(K, d)
        rho = x[K * d:].reshape(N, K - 1)
        logits = torch.cat([rho, torch.zeros(N, 1, dtype=x.dtype)], dim=1)
        logr = torch.log_softmax(logits, dim=1)
        r = torch.exp(logr)
        c = 0.5 * ((Xt[:, None, :] - m[None, :, :]) ** 2).sum(-1) - lp[None, :]
        return torch.sum(r * (c + logr)) + 0.5 * prior_prec * torch.sum(m * m)
    return f


def gmm_vb_sparsity(N, K, d):
    """(G=N, M=K-1) index array of the local blocks; globals are 0..K*d-1."""
    return K * d + np.arange(N * (K - 1)).reshape(N, K - 1)


# --------------------------------------------------------------------------
# Config 4: mean-field normal VB for a multivariate-normal target (the
# reference's own LRVB test model, tests/test_lr_cov_lib.py:30-46), flat
# parameter = (mean (dim), var (dim)).
# --------------------------------------------------------------------------

def mvn_kl_objective(true_mean, true_info):
    tm = torch.as_tensor(np.asarray(true_mean, dtype=np.float64))
    ti = torch.as_tensor(np.asarray(true_info, dtype=np.float64))
    dim = tm.shape[0]

    def f(par):
        mean, var = par[:dim], par[dim:]
        tc = mean - tm
        e_log_p = -0.5 * (torch.sum(torch.diagonal(ti) * var) + tc @ ti @ tc)
        q_ent = 0.5 * torch.sum(torch.log(var))
        return -1 * (q_ent + e_log_p)
    return f


def mvn_kl_closed_form(true_mean, true_info):
    """Optimum and Hessian in closed form: mean = true_mean,
    var = 1/diag(info); H = blockdiag(info, diag(0.5 / var^2))."""
    dim = len(true_mean)
    var = 1.0 / np.diag(true_info)
    H = np.zeros((2 * dim, 2 * dim))
    H[:dim, :dim] = true_info
    H[dim:, dim:] = np.diag(0.5 / var ** 2)
    return np.concatenate([np.asarray(true_mean, dtype=np.float64), var]), H


def gmm_vb_fit(Xobs, K, prior_prec=1e-2, iters=200, seed=0, log_pi=None):
    """Coordinate ascent for the GMM-VB objective (closed-form updates):
    rho_n = optimal logits given m, m_k = sum_n r_nk x_n / (sum_n r_nk + prior).
    Returns the flat parameter at (numerically) the optimum, where the Hessian
    is positive definite."""
    Xobs = np.asarray(Xobs, dtype=np.float64)
    N, d = Xobs.shape
    rng = np.random.RandomState(seed)
    lp = -np.log(K) * np.ones(K) if log_pi is None else np.asarray(log_pi)
    m = Xobs[rng.choice(N, K, replace=False)].copy()
    for _ in range(iters):
        c = 0.5 * ((Xobs[:, None, :] - m[None]) ** 2).sum(-1) - lp[None]
        logits = -(c - c[:, -1:])
        r = np.exp(logits - logits.max(1, keepdims=True))
        r /= r.sum(1, keepdims=True)
        m = (r.T @ Xobs) / (r.sum(0)[:, None] + prior_prec)
    c = 0.5 * ((Xobs[:, None, :] - m[None]) ** 2).sum(-1) - lp[None]
    logits = -(c - c[:, -1:])
    return np.concatenate([m.reshape(-1), logits[:, :K - 1].reshape(-1)])
