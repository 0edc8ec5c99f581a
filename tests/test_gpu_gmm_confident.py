"""GPU tests of ``gmm_blocks`` (``csrc/blockchol.cu``) on observations assigned with confidence, the normal case of a
fitted mixture whose clusters are separated: logit gaps of tens to hundreds, where 1 - r rounds to 0 in float64.

Every output of every observation is held to per-entry error bars (``highprec.gmm_error_bars``, scaled by r_j q_j
and r_j r_l, not by the largest entry of the block) around the longdouble reference that does not cancel
(``highprec.gmm_blocks_stable_ld``, itself checked against mpmath in ``test_gmm_reference_host.py``).  Neither the
longdouble closed form nor float64 autodiff is a reference in this regime.  Downstream, the block-arrow solver must
factor the Hessian of a fitted two-cluster model and solve with a componentwise small residual."""
import numpy as np
import pytest
import torch

from oracle import fixtures, highprec, models

pytestmark = pytest.mark.gpu

EPS = highprec.GMM_EPS
KD = [(K, d) for K in (2, 3, 17, 32) for d in (1, 33)] + [(32, 257)]


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


@pytest.fixture(scope='module')
def n_wrap(vt):
    """Observations of one launch past twice its grid cap: grid_for(N, 1, 8) caps the grid at 8 CTAs per SM."""
    return 2 * 8 * vt.ops.device_info()['sm_count'] + 3


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64), device='cuda')


def _describe(meta, n):
    return 'row {}'.format(n) if meta is None else 'row {} (dominant {}, gap {}, vb {})'.format(
        n, meta['dom'][n], meta['gap'][n], meta['vb'][n])


def _check_within_bars(out, X, m, rho, log_pi, what, meta=None):
    """The outputs of gmm_blocks in ``out`` against the stable longdouble reference within the per-entry bars; the
    cross blocks entry by entry on the device, a chunk of observations at a time."""
    N, d = X.shape
    K = m.shape[0]
    for key, v in out.items():
        assert not bool(torch.isnan(v).any()), '{}: NaN in {}'.format(what, key)
    ref = highprec.gmm_blocks_stable_ld(X, m, rho, log_pi)
    bars = highprec.gmm_error_bars(ref, d)
    host = {k: out[k].cpu().numpy() for k in ('r', 'grad_rho', 'obj_terms', 'blocks') if k in out}
    for key, rat in highprec.gmm_bar_ratios(host, ref, bars, keys=tuple(host)).items():
        n = int(np.argmax(rat))
        assert rat[n] <= 1, '{}: {} of {} is {:.3g} x its bar'.format(what, key, _describe(meta, n), rat[n])
    # cross[n, j, k*d + t] = coef[n, j, k] (m_k[t] - x_n[t]), bar (tau_n |coef| + phi_n) |m_k[t] - x_n[t]|
    coef, cbar = _dev(ref['coef']), _dev(bars['coef'])
    Xd, md = _dev(X), _dev(m)
    step = max(1, (1 << 24) // ((K - 1) * K * d))
    for n0 in range(0, N, step):
        dm = md[None] - Xd[n0:n0 + step, None, :]
        got = out['cross'][n0:n0 + step].view(-1, K - 1, K, d)
        err = (got - coef[n0:n0 + step, :, :, None] * dm[:, None]).abs()
        bar = cbar[n0:n0 + step, :, :, None] * dm.abs()[:, None]
        bad = ~(err <= bar)
        if bool(bad.any()):
            n = n0 + int(bad.reshape(bad.shape[0], -1).any(1).nonzero()[0, 0])
            worst = float((err[n - n0] / bar[n - n0]).nan_to_num(nan=np.inf).max())
            raise AssertionError('{}: cross block of {} is {:.3g} x its bar'.format(what, _describe(meta, n), worst))


@pytest.mark.parametrize('K,d', KD)
def test_gmm_blocks_confident_observations(vt, n_wrap, K, d):
    """One launch past twice the grid cap.  Each observation has a dominant component (the first, the last free
    logit or the implicit K-th), a gap from 0 to 800 (36 / 37 / 38 straddle 1 - r rounding to 0 in float64, >= 745
    underflows the runner-up) and possibly a tie at the top; half at the VB optimum, where only the complements
    1 - r carry the local block."""
    X, m, rho, log_pi, meta = fixtures.gmm_confident(K * 1000 + d, n_wrap, K, d)
    assert set(meta['gap'][meta['vb']]) == set(meta['gap'][~meta['vb']]) == set(map(float, fixtures.GMM_GAPS))
    assert set(meta['dom']) == {0, K - 2, K - 1}
    out = vt.ops.gmm_blocks(_dev(X), _dev(m), _dev(rho), _dev(log_pi))
    _check_within_bars(out, X, m, rho, log_pi, 'K {} d {}'.format(K, d), meta)


@pytest.mark.parametrize('K,d', [(2, 1), (3, 33), (32, 33)])
def test_gmm_blocks_overlap_regime_within_the_bars(vt, n_wrap, K, d):
    """The overlapping clusters of the edge tests (every responsibility in [1e-3, 1 - 1e-3]) meet the same bars."""
    from test_gpu_block_arrow import _gmm_data
    X, m, rho, log_pi = _gmm_data(K * 7 + d, n_wrap, K, d)
    out = vt.ops.gmm_blocks(_dev(X), _dev(m), _dev(rho), _dev(log_pi))
    _check_within_bars(out, X, m, rho, log_pi, 'overlap K {} d {}'.format(K, d))


def test_gmm_vb_two_separated_clusters_factor_and_solve(vt, n_wrap):
    """Centers at +-6 on one axis, d = 2, unit noise, fitted by coordinate ascent: most logit gaps are past 37.  The
    assembled Hessian is within the bars of the reference, the block-arrow solver factors it, and its solutions of
    two right-hand sides have, on every local row, a residual of a few eps of |H||x| + |b| (longdouble residual);
    against the reference Hessian, plus what the bars allow the assembly.  The global rows meet the normwise bound
    of test_gmm_vb_medium_block_arrow_solve."""
    N, K, d, prior = n_wrap, 2, 2, 0.5
    rng = np.random.default_rng(20261021)
    X = rng.normal(size=(N, d))
    X[:, 0] += np.where(rng.random(N) < 0.5, -6.0, 6.0)
    x = models.gmm_vb_fit(X, K, prior_prec=prior)
    m, rho = x[:K * d].reshape(K, d), x[K * d:].reshape(N, K - 1)
    gaps = np.abs(rho[:, 0])
    assert np.mean(gaps > 37) >= 0.9 and gaps.max() < 700, (np.mean(gaps > 37), gaps.max())
    log_pi = np.full(K, -np.log(K))
    obj = vt.objectives.GMMVBObjective(X, K, prior_prec=prior)
    sa = obj.sparsity_array()
    h = vt.SparseBlockHessian(obj, sa).get_hessian(x)
    _check_within_bars(dict(blocks=h.blocks, cross=h.cross), X, m, rho, log_pi, 'fitted two-cluster Hessian')
    ref = highprec.gmm_blocks_stable_ld(X, m, rho, log_pi)
    bars = highprec.gmm_error_bars(ref, d)
    rsum = np.asarray(ref['r'], dtype=np.longdouble).sum(0)
    hgg_ref = np.diag(np.repeat(np.asarray(rsum + prior, dtype=np.float64), d))
    np.testing.assert_allclose(h.hgg.cpu().numpy(), hgg_ref, rtol=1e-12, atol=0)

    solve = vt.solver_lib.get_sparse_cholesky_solver(h)                     # LinAlgError if a block is not PD
    B = rng.normal(size=(obj.dim, 2))
    sol = np.asarray(solve(B))
    assert np.all(np.isfinite(sol))
    gi = np.arange(K * d)
    dm = m[None] - X[:, None, :]                                             # (N, K, d)
    cross_ref = (ref['coef'][:, :, :, None] * dm[:, None]).reshape(N, K - 1, K * d)
    cross_bar = (bars['coef'][:, :, :, None] * np.abs(dm)[:, None]).reshape(N, K - 1, K * d)
    zero = np.zeros_like(B)
    hk = (h.blocks.cpu().numpy(), h.cross.cpu().numpy(), h.hgg.cpu().numpy())
    for name, (blocks, cross, hgg), slack in (
            ('assembled', hk, None),
            ('reference', (ref['blocks'], cross_ref, hgg_ref), (bars['blocks'], cross_bar, np.zeros_like(hgg_ref)))):
        res = np.abs(highprec.block_arrow_residual_ld(sa, gi, blocks, cross, hgg, sol, B))
        size = -highprec.block_arrow_residual_ld(sa, gi, np.abs(blocks), np.abs(cross), np.abs(hgg), np.abs(sol), zero)
        bound = 64 * EPS * (size + np.abs(B))
        if slack is not None:
            bound = bound - highprec.block_arrow_residual_ld(sa, gi, *slack, np.abs(sol), zero)
        loc = sa.reshape(-1)
        ratio = (res[loc] / bound[loc]).astype(np.float64)
        i = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
        assert ratio[i] <= 1, '{} Hessian: local row {} rhs {} residual {:.3g} x its bound'.format(
            name, loc[i[0]], i[1], ratio[i])
        hmax = max(np.abs(blocks).max(), np.abs(cross).max(), np.abs(hgg).max())
        assert res[gi].max() < 1e-9 * hmax * np.abs(sol).max(), name
