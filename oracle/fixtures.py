"""The reference's own test fixtures, re-created without autograd/paragami.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  Each fixture returns
torch objectives (float64) plus the closed-form truths the reference's tests
assert against, so both the oracle and the CUDA path can be pinned to the same
known answers (SURVEY.md section 4 / 8c).
"""
import numpy as np
import torch


# --------------------------------------------------------------------------
# QuadraticModel  (vittles/tests/test_utils.py:23-75)
# --------------------------------------------------------------------------

class QuadraticModel:
    """f = 0.5 theta^T A theta + lam^T theta, A = v v^T + I,
    v = linspace(.1,.3,dim), lam0 = linspace(.5,10,dim), optimum -A^{-1} lam
    (``test_utils.py:33-34,53-69``).  The reference flattens both arguments
    with a lower bound of -20 (``:28-31``) so that, in the "free"
    parametrisation, derivatives of every order are non-zero.  The free
    transform restated here is ``free = log(x - lb)`` (paragami's
    one-sided-bound map; paragami itself is unavailable - the fixture only
    needs *a* smooth bijection, and every truth below is derived from the same
    map, so the checks are self-consistent)."""
    LB = -20.0

    def __init__(self, dim):
        self.dim = dim
        vec = np.linspace(0.1, 0.3, num=dim)
        self.matrix = np.outer(vec, vec) + np.eye(dim)
        self._A = torch.as_tensor(self.matrix)

    # folded <-> flat
    def flatten(self, x, free):
        x = np.asarray(x, dtype=np.float64)
        return np.log(x - self.LB) if free else x.copy()

    def fold(self, x, free):
        x = np.asarray(x, dtype=np.float64)
        return np.exp(x) + self.LB if free else x.copy()

    def _fold_t(self, x, free):
        return torch.exp(x) + self.LB if free else x

    def _flatten_t(self, x, free):
        return torch.log(x - self.LB) if free else x

    def get_default_lambda(self):
        return np.linspace(0.5, 10.0, num=self.dim)

    def get_true_optimal_theta(self, lam):
        return -1 * np.linalg.solve(self.matrix, lam)

    def get_flat_objective(self, theta_free, lambda_free):
        def f(theta_flat, lam_flat):
            theta = self._fold_t(theta_flat, theta_free)
            lam = self._fold_t(lam_flat, lambda_free)
            A = self._A.to(theta.device)
            return 0.5 * theta @ A @ theta + lam @ theta
        return f

    def get_flat_hyper_par_objective(self, theta_free, lambda_free):
        def f(theta_flat, lam_flat):
            return self._fold_t(lam_flat, lambda_free) @ self._fold_t(theta_flat, theta_free)
        return f

    def get_flat_true_optimal_theta(self, theta_free, lambda_free):
        """torch map lam_flat -> theta_flat (closed form), differentiable."""
        def opt(lam_flat):
            lam = self._fold_t(lam_flat, lambda_free)
            theta = -1 * torch.linalg.solve(self._A.to(lam.device), lam)
            return self._flatten_t(theta, theta_free)
        return opt

    def get_default_flat_values(self, theta_free, lambda_free):
        lam0 = self.get_default_lambda()
        theta0 = self.get_true_optimal_theta(lam0)
        return self.flatten(theta0, theta_free), self.flatten(lam0, lambda_free)


# --------------------------------------------------------------------------
# Block quadratic  (vittles/tests/test_sparse_hessian_lib.py:15-113)
# --------------------------------------------------------------------------

def _psd_from_free(free6):
    """3x3 PSD matrix from 6 free numbers: Cholesky factor with a log diagonal
    (the shape of paragami's PSDSymmetricMatrixPattern free map)."""
    L = torch.zeros(3, 3, dtype=free6.dtype, device=free6.device)
    idx = torch.tril_indices(3, 3, device=free6.device)
    L = L.index_put((idx[0], idx[1]), free6)
    d = torch.diagonal(L)
    L = L - torch.diag(d) + torch.diag(torch.exp(d))
    return L @ L.T


def block_quadratic(num_groups=10, group_size=3, with_scales=False, seed=42):
    """f(x) = 0.5 [scale] sum_n a_n^T M_n a_n with per-group parameters
    (a_n (3), M_n (6 free)) -> block size 9 (``test_sparse_hessian_lib.py:21-31``)
    and, optionally, two global positive ``scales`` multiplying everything
    (``:67-73``).  Flat layout: all vectors, then all matrices, then the
    scales - so each block's indices are NOT contiguous, as upstream."""
    assert group_size == 3
    rng = np.random.RandomState(seed)
    G = num_groups
    nvec, nmat = G * 3, G * 6
    x = rng.normal(size=nvec + nmat + (2 if with_scales else 0))
    if with_scales:
        x[-2:] = np.log(rng.uniform(0.5, 2.0, size=2))
    inds = np.array([list(range(3 * g, 3 * g + 3)) + list(range(nvec + 6 * g, nvec + 6 * g + 6))
                     for g in range(G)])
    global_inds = np.arange(nvec + nmat, nvec + nmat + 2) if with_scales else np.array([], dtype=int)

    def f(xf):
        a = xf[:nvec].reshape(G, 3)
        mats = torch.stack([_psd_from_free(xf[nvec + 6 * g: nvec + 6 * g + 6]) for g in range(G)])
        val = 0.5 * torch.einsum('nij,ni,nj', mats, a, a)
        if with_scales:
            val = val * torch.prod(torch.exp(xf[-2:]))
        return val
    return f, x, inds, global_inds


# --------------------------------------------------------------------------
# MVN target for linear-response covariances (tests/test_lr_cov_lib.py:20-61)
# --------------------------------------------------------------------------

def mvn_lr_fixture(dim=4):
    """true_cov = dim*I + m m^T, m = arange(dim) (``:26-28``); optimum
    mean = m, var = 1/diag(info) (``:60-61``); LR covariance of the mean is
    exactly ``true_cov`` (``:90-93``)."""
    true_mean = np.arange(0, dim).astype(np.float64)
    true_cov = dim * np.eye(dim) + np.outer(true_mean, true_mean)
    true_info = np.linalg.inv(true_cov)
    return true_mean, true_cov, true_info


# --------------------------------------------------------------------------
# Weighted least squares with weights as the hyperparameter
# (tests/test_sensitivity_lib.py:838-901)
# --------------------------------------------------------------------------

def wls_fixture(n_obs=10, dim=2, seed=7):
    rng = np.random.RandomState(seed)
    theta_true = np.array([0.5, -0.1])[:dim]
    x = rng.random_sample((n_obs, dim))
    y = x @ theta_true + rng.normal(size=n_obs)
    xt, yt = torch.as_tensor(x), torch.as_tensor(y)

    def objective(theta, w):
        resid = yt - xt @ theta
        return torch.sum(w * resid ** 2)

    def run_regression(w):
        """torch closed form, differentiable in w."""
        xtx = torch.einsum('n,ni,nj->ij', w, xt, xt)
        xty = torch.einsum('n,ni,n->i', w, xt, yt)
        return torch.linalg.solve(xtx, xty)
    return objective, run_regression, x, y


# --------------------------------------------------------------------------
# GMM-VB observations assigned with confidence (the regime of a fitted mixture
# whose clusters are separated)
# --------------------------------------------------------------------------

GMM_GAPS = (0, 1, 20, 36, 37, 38, 60, 300, 700, 740, 800)


def gmm_confident(seed, N, K, d, spacing=48.0):
    """X (N, d), m (K, d), rho (N, K-1), log_pi (K,) and, per observation, the component built to dominate (``dom``)
    and the gap between its logit and the runner-up's (``gap``); ``vb`` marks the observations with logits at the
    VB optimum.

    Centers are ``spacing`` apart: m_k = spacing / sqrt(2) e_k when d >= K, else m_k = spacing k e_0 (on a line).
    Observation n takes in turn a dominant component (the first, the last free logit or the implicit K-th), a gap
    from GMM_GAPS and whether two logits tie at the top.
      * even n (``vb``): x_n lies on the segment from m_dom to a runner-up m_b where c_b - c_dom = gap, plus unit
        noise in the directions no center spans; rho_j = -(c_j - c_K), so that a_k = c_k + log r_k is the same for
        every k and only the complements 1 - r carry the local block.  A tie is the midpoint (gap 0).
      * odd n: top logit T, runner-up T - gap (T for a tie, which may be the implicit 0), the others T - gap - U(0, 8).
    Gaps >= 745 underflow the runner-up's responsibility."""
    rng = np.random.default_rng(seed)
    lp = 0.3 * rng.normal(size=K)
    log_pi = lp - np.log(np.sum(np.exp(lp)))
    m = np.zeros((K, d))
    if d >= K:
        m[np.arange(K), np.arange(K)] = spacing / np.sqrt(2.0)
        free_axes = np.arange(K, d)
    else:
        m[:, 0] = spacing * np.arange(K)
        free_axes = np.arange(1, d)
    positions = sorted({0, K - 2, K - 1})
    combos = [(p, g, tie) for p in positions for g in GMM_GAPS for tie in (False, True)]
    dom = np.empty(N, dtype=np.int64)
    gap = np.empty(N)
    vb = np.arange(N) % 2 == 0
    X = np.zeros((N, d))
    offsets = np.zeros((N, K))
    for n in range(N):
        a, g, tie = combos[(n // 2 + 7 * (n % 2)) % len(combos)]
        g = 0.0 if tie else float(g)
        others = [k for k in range(K) if k != a]
        if vb[n]:
            b = (a + 1 if a + 1 < K else a - 1) if d < K else others[rng.integers(K - 1)]
            u = (m[b] - m[a]) / spacing
            t = (0.5 * spacing ** 2 + (log_pi[a] - log_pi[b]) - g) / spacing
            X[n] = m[a] + t * u
            X[n, free_axes] = rng.normal(size=len(free_axes))
        else:
            b = others[rng.integers(K - 1)]
            offsets[n] = g + rng.uniform(0.0, 8.0, size=K)
            offsets[n, a] = 0.0
            offsets[n, b] = g
        dom[n], gap[n] = a, g
    c = 0.5 * ((X[:, None, :] - m[None]) ** 2).sum(-1) - log_pi[None]
    logits = np.where(vb[:, None], -(c - c[:, -1:]), offsets[:, -1:] - offsets)
    return X, m, logits[:, :K - 1].copy(), log_pi, dict(dom=dom, gap=gap, vb=vb)
