"""CPU tests of the GMM-VB references for observations assigned with confidence (``oracle/highprec.py``): the
longdouble forms that do not cancel against the definition in mpmath, and the per-entry error bars of
``gmm_error_bars`` against the formulas they have to tell apart, restated in float64 as ``gmm_blocks`` evaluates
them (``csrc/blockchol.cu``).  No GPU needed."""
import numpy as np
import pytest

from oracle import fixtures, highprec

CASES = [(2, 1), (2, 33), (3, 1), (3, 33), (17, 1), (32, 33)]


def _data(K, d, N=660):
    return fixtures.gmm_confident(K * 100 + d, N, K, d)


def _rows(ref, rows):
    return {k: v[rows] for k, v in ref.items()}


def _kernel_f64(X, m, rho, log_pi, stable):
    """The per-observation arithmetic of gmm_blocks in float64: ``stable`` False restates the formulas
    r_j (delta_j + 1) - r_j^2 (2 delta_j + 1), r_j (1 - r_j) and delta = a - abar; True the forms of the kernel's
    header (complements and deviations as sums over the other components)."""
    N, K = rho.shape[0], m.shape[0]
    M = K - 1
    lg = np.concatenate([rho, np.zeros((N, 1))], axis=1)
    mx = lg.max(1, keepdims=True)
    e = np.exp(lg - mx)
    tot = e.sum(1, keepdims=True)
    r = e / tot
    c = 0.5 * ((X[:, None, :] - m[None]) ** 2).sum(-1) - log_pi[None]
    a = c + ((lg - mx) - np.log(tot))
    abar = (r * a).sum(1)
    idx = np.arange(M)
    if stable:
        dom = np.argmax(lg, axis=1)
        is_dom = np.arange(K)[None] == dom[:, None]
        q = np.where(is_dom, np.where(is_dom, 0.0, e).sum(1, keepdims=True) * r, 1.0 - r)
        da = (c - c[np.arange(N), dom][:, None]) + (lg - mx)
        dev = da - np.where(is_dom, 0.0, r * da).sum(1, keepdims=True)
        rj, qj, dj = r[:, :M], q[:, :M], dev[:, :M]
        blocks = -(rj[:, :, None] * rj[:, None, :]) * (dj[:, :, None] + dj[:, None, :] + 1.0)
        blocks[:, idx, idx] = rj * qj + rj * dj * (qj - rj)
        coef = -(rj[:, :, None] * r[:, None, :])
        coef[:, idx, idx] = rj * qj
    else:
        dev = a - abar[:, None]
        rj, dj = r[:, :M], dev[:, :M]
        blocks = -(rj[:, :, None] * rj[:, None, :]) * (dj[:, :, None] + dj[:, None, :] + 1.0)
        blocks[:, idx, idx] += rj * (dj + 1.0)
        coef = rj[:, :, None] * (np.eye(M, K)[None] - r[:, None, :])
    return dict(r=r, grad_rho=rj * dj, obj_terms=abar, blocks=blocks, coef=coef)


@pytest.mark.parametrize('K,d', CASES)
def test_stable_longdouble_reference_matches_mpmath(K, d):
    """About 100 observations per case over the whole grid of gaps, dominant positions and ties, at the VB optimum
    and off it: the longdouble reference is within 1/100 of the bars of the definition evaluated in mpmath."""
    X, m, rho, log_pi, meta = _data(K, d)
    ref = highprec.gmm_blocks_stable_ld(X, m, rho, log_pi)
    bars = highprec.gmm_error_bars(ref, d)
    rows = np.arange(0, X.shape[0], 6 if K < 32 else 12)
    assert set(meta['gap'][rows]) == set(float(g) for g in fixtures.GMM_GAPS)
    mp = highprec.gmm_blocks_mp(X, m, rho, log_pi, rows)
    ratios = highprec.gmm_bar_ratios(mp, _rows(ref, rows), _rows(bars, rows))
    for key, rat in ratios.items():
        i = int(np.argmax(rat))
        assert rat[i] <= 0.01, '{} K {} d {}: row {} (gap {}) at {:.3g} of the bar'.format(
            key, K, d, rows[i], meta['gap'][rows[i]], rat[i])


def _free_dominant(meta, rho, lo, hi):
    """Observations whose largest logit is a free one (not the implicit 0) and unique, with lo <= gap <= hi."""
    lg = np.concatenate([rho, np.zeros((rho.shape[0], 1))], axis=1)
    top = np.sort(lg, axis=1)
    return (np.argmax(lg, axis=1) < rho.shape[1]) & (top[:, -1] - top[:, -2] >= lo) & (top[:, -1] - top[:, -2] <= hi)


@pytest.mark.parametrize('K,d', CASES)
def test_longdouble_closed_form_misses_the_bars_of_confident_rows(K, d):
    """The longdouble closed form the overlap-regime tests use (``_gmm_closed_form_ld``) is no reference here: at
    every observation whose dominant component is a free logit with a gap of 40 or more it is outside the bars (its
    11 extra bits postpone the cancellation from a gap of ~37 to ~44, no further)."""
    from test_gpu_block_arrow import _gmm_closed_form_ld
    X, m, rho, log_pi, meta = _data(K, d)
    ref = highprec.gmm_blocks_stable_ld(X, m, rho, log_pi)
    bars = highprec.gmm_error_bars(ref, d)
    old = _gmm_closed_form_ld(X, m, rho, log_pi)
    ratios = highprec.gmm_bar_ratios(old, ref, bars, keys=('grad_rho', 'blocks', 'coef'))
    worst = np.maximum.reduce(list(ratios.values()))
    sel = _free_dominant(meta, rho, 40, 700)
    assert sel.sum() >= 20
    assert np.all(worst[sel] > 1), np.flatnonzero(sel & (worst <= 1))


@pytest.mark.parametrize('K,d', CASES)
def test_bars_separate_the_cancelling_formulas_from_the_stable_ones(K, d):
    """The kernel's arithmetic restated in float64: the formulas that cancel are outside the bars at every
    observation whose dominant component is a free logit with a gap of 38 to 700, and the stable forms are inside
    them at every observation, underflowed responsibilities included."""
    X, m, rho, log_pi, meta = _data(K, d)
    ref = highprec.gmm_blocks_stable_ld(X, m, rho, log_pi)
    bars = highprec.gmm_error_bars(ref, d)
    new = _kernel_f64(X, m, rho, log_pi, stable=True)
    for key, rat in highprec.gmm_bar_ratios(new, ref, bars).items():
        i = int(np.argmax(rat))
        assert rat[i] <= 1, '{} K {} d {}: row {} (gap {}, vb {}) at {:.3g} x the bar'.format(
            key, K, d, i, meta['gap'][i], meta['vb'][i], rat[i])
    old = _kernel_f64(X, m, rho, log_pi, stable=False)
    worst = np.maximum.reduce(list(highprec.gmm_bar_ratios(old, ref, bars, keys=('grad_rho', 'blocks')).values()))
    sel = _free_dominant(meta, rho, 38, 700)
    assert sel.sum() >= 20
    assert np.all(worst[sel] > 1), np.flatnonzero(sel & (worst <= 1))
    if K == 2:       # at the VB optimum the one local entry is r (1 - r) > 0; the cancelling formula's is often <= 0
        opt = sel & meta['vb']
        assert np.all(ref['blocks'][opt, 0, 0] > 0) and np.all(new['blocks'][opt, 0, 0] > 0)
        assert np.mean(old['blocks'][opt, 0, 0] <= 0) > 0.2
