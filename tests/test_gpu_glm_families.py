"""GPU tests of the per-row GLM family arithmetic of ``glm.cu`` (``StatsOp``: resid = b'(z) - y, s = w b''(z),
sqrt(s); ``b_deriv``: the coefficients w b^(q+1)(z) of ``vt_glm_dirderiv``) over the whole linear-predictor range.

The reference is the mpmath statement of the three families (``oracle/highprec.py``), which shares no formula with
the kernels.  With X = I (n <= 2048) the statistics pass returns z = theta exactly and each entry of the directional
derivative along all-ones directions is one coefficient, so the kernels' own per-row values are probed one by one:
every product with 0 or 1 is exact and the reductions add zeros to a single value.  Then: the logistic model on
(-X, 1 - y) is the model on (X, y) with the labels coded the other way, so every FP64 output must be the same bits;
and on separable data (every row 16 .. 36 from the margin) Hessian, IJ matrix, influence and directional derivatives
must hold the parity bar against references built from the mpmath weights and residuals."""
import math

import numpy as np
import pytest
import scipy.linalg
import torch

from conftest import assert_close
from oracle import highprec, influence as oinf

pytestmark = pytest.mark.gpu

FAMILIES = ['logistic', 'poisson', 'gaussian']
REL = 2e-15
TINY = 2.0 ** -1073                        # two units of the last subnormal place
YS = (0.0, 1.0, 0.3)
WS = (1.0, 0.37, 2.5, 0.0)


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _host(t):
    return t.detach().cpu().numpy()


def _grid():
    """+-0, +-1e-300, a dense sweep of [-40, 40], the zeros of b^(4) and b^(5) (|z| ~ 2.29, 1.32) and the far tails
    where sigma(-|z|), exp(z) and their products leave the normal range or overflow."""
    special = [0.0, 1e-300, 1.3169579, 2.2924317, 36.7, 37.0, 100.0, 700.0, 708.4, 709.78, 745.2, 750.0]
    sweep = np.linspace(-40.0, 40.0, 1601)
    return np.concatenate([sweep, special, [-v for v in special]])


@pytest.fixture(scope='module')
def grid():
    return _grid()


@pytest.fixture(scope='module')
def refs(grid):
    """Per family: the mpmath b^(k) (k = 1..5), resid for every y and s for every w on the grid."""
    out = {}
    for fam in FAMILIES:
        d = {'b': {k: highprec.glm_bderiv_mp(grid, k, fam) for k in range(1, 6)}}
        d['resid'] = {y: highprec.glm_resid_mp(grid, y, fam) for y in YS}
        d['s'] = {w: highprec.glm_weight_mp(grid, w, fam) for w in WS}
        out[fam] = d
    return out


def _check(actual, ref, what, rel=REL, scale=None, mask=None):
    """|actual - ref| <= rel * scale + 2^-1073 (scale = |ref| by default); where ref is +-inf actual must equal it."""
    actual, ref = np.asarray(actual, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    m = np.ones(ref.shape, dtype=bool) if mask is None else mask
    inf = m & np.isinf(ref)
    assert np.array_equal(actual[inf], ref[inf]), '{}: infinite entries differ'.format(what)
    fin = m & np.isfinite(ref)
    scale = np.abs(ref) if scale is None else np.broadcast_to(scale, ref.shape)
    err = np.abs(actual[fin] - ref[fin])
    tol = rel * scale[fin] + TINY
    bad = ~(err <= tol)
    if bad.any():
        i = np.argmax(np.where(bad, err / tol, 0.0))
        raise AssertionError('{}: {} of {} entries off; worst at z-index {}: {!r} vs {!r} (err/tol {:.3g})'.format(
            what, int(bad.sum()), int(fin.sum()), int(np.nonzero(fin)[0][i]), float(actual[fin][i]),
            float(ref[fin][i]), float(err[i] / tol[i])))


# --------------------------------------------------------------------------- a. pointwise probes, X = I ----
@pytest.mark.parametrize('family', FAMILIES)
def test_stats_pointwise_vs_mpmath(vt, family, grid, refs):
    """glm_stats on X = I, theta = z: resid and s of every row against mpmath, for y in {0, 1, 0.3} and
    w in {1, 0.37, 2.5, 0}, on both instances of the pass (with and without the fused column maxima)."""
    n = grid.size
    assert n <= 2048
    X = torch.eye(n, dtype=torch.float64, device='cuda')
    zt = _dev(grid)
    r = refs[family]
    b1 = np.abs(r['b'][1])
    for colmax in (False, True):
        for y in YS:
            for w in WS:
                st = vt.ops.glm_stats(X, zt, torch.full((n,), y, dtype=torch.float64, device='cuda'),
                                      torch.full((n,), w, dtype=torch.float64, device='cuda'), family,
                                      want_grad=False, want_colmax=colmax)
                tag = '{} y={} w={} colmax={}'.format(family, y, w, colmax)
                z, resid, s = (_host(t) for t in st[:3])
                assert np.all(z == grid), tag + ': z != theta'
                if family == 'gaussian':
                    assert np.array_equal(resid, r['resid'][y]), tag + ': resid not exact'
                    assert np.array_equal(s, r['s'][w]), tag + ': s not exact'
                else:
                    if family == 'logistic' and y != 0.3:
                        _check(resid, r['resid'][y], tag + ' resid')
                    else:                                # b'(z) ~ y cancels: relative to |b'| + y
                        _check(resid, r['resid'][y], tag + ' resid', scale=b1 + y)
                    # poisson, w = 0, z >= 710: 0 * inf is NaN (the mpmath reference says 0)
                    ok = ~((family == 'poisson') & (w == 0.0) & (grid >= 710.0))
                    _check(s, r['s'][w], tag + ' s', mask=ok)
                    if family == 'poisson':
                        big = grid >= 710.0
                        assert np.all(np.isposinf(resid[big])), tag + ': resid not +inf from z = 710 on'
                        if w > 0:
                            assert np.all(np.isposinf(s[big])), tag + ': s not +inf from z = 710 on'
                if not colmax:
                    continue
                sq, cmax = st[4]
                assert np.array_equal(_host(sq), np.sqrt(s), equal_nan=True), tag + ': sq != sqrt(s)'
                normal = np.abs(r['s'][w]) >= 2.0 ** -1022
                _check(_host(sq), np.sqrt(r['s'][w]), tag + ' sqrt(s)', mask=normal & np.isfinite(r['s'][w]))
                cm = _host(cmax).view(np.uint64)
                if torch.isfinite(st[2]).all():
                    # column c holds max_n sqrt(s_n) |x_nc| = sqrt(s_c): its high word (the binade and top 20 bits)
                    hi = _host(sq).view(np.uint64) & np.uint64(0xFFFFFFFF00000000)
                    assert np.array_equal(cm, hi), tag + ': column maxima != high words of sqrt(s)'
                else:                                    # a non-finite weight poisons every column (0 * inf)
                    assert np.all(cm >= np.uint64(0x7FF0000000000000)), tag + ': non-finite weight not propagated'


@pytest.mark.parametrize('family', FAMILIES)
def test_dirderiv_coefficients_pointwise_vs_mpmath(vt, family, grid, refs):
    """glm_dirderiv(I, z, ones((q, n)), w): out[n] = w_n b^(q+1)(z_n), q = 1..4, against mpmath.  Logistic:
    relative 2e-15 from |z| = 3 on, 1e-14 of the largest |b^(k)| inside; poisson relative; gaussian exact."""
    zz = grid[grid <= 708.4] if family == 'poisson' else grid   # one non-finite coefficient would poison every column
    sel = np.isin(grid, zz)
    n = zz.size
    X = torch.eye(n, dtype=torch.float64, device='cuda')
    zt = _dev(zz)
    for q in range(1, 5):
        k = q + 1
        bk = refs[family]['b'][k][sel]
        for w in WS:
            out = _host(vt.ops.glm_dirderiv(X, zt, torch.ones((q, n), dtype=torch.float64, device='cuda'),
                                            torch.full((n,), w, dtype=torch.float64, device='cuda'), family))
            ref = w * bk                                  # (one more rounding than the kernel's w * b)
            tag = '{} q={} w={}'.format(family, q, w)
            if family == 'gaussian':
                assert np.array_equal(out, ref), tag + ': not exact'
            elif family == 'poisson':
                _check(out, ref, tag)
            else:
                far = np.abs(zz) >= 3.0
                _check(out, ref, tag + ' |z|>=3', mask=far)
                _check(out, ref, tag + ' |z|<3', rel=1e-14, scale=np.max(np.abs(ref)), mask=~far)


@pytest.mark.parametrize('family', FAMILIES)
def test_nan_linear_predictor_propagates(vt, family):
    """A NaN z gives a NaN resid, and (where they depend on z) a NaN s, sqrt(s), column maximum and coefficient."""
    X1 = torch.ones((1, 1), dtype=torch.float64, device='cuda')
    nan = torch.full((1,), math.nan, dtype=torch.float64, device='cuda')
    w = torch.full((1,), 0.37, dtype=torch.float64, device='cuda')
    for q in range(1, 5):
        c = vt.ops.glm_dirderiv(X1, nan, torch.ones((q, 1), dtype=torch.float64, device='cuda'), w, family)
        if family == 'gaussian':
            assert float(c) == (0.37 if q == 1 else 0.0)
        else:
            assert torch.isnan(c).all(), '{} q={}: coefficient not NaN'.format(family, q)
    # statistics: with X = I, 0 * NaN makes every row's z NaN
    n = 16
    X = torch.eye(n, dtype=torch.float64, device='cuda')
    theta = torch.linspace(-3, 3, n, dtype=torch.float64, device='cuda')
    theta[5] = math.nan
    y = torch.full((n,), 1.0, dtype=torch.float64, device='cuda')
    wn = torch.full((n,), 0.37, dtype=torch.float64, device='cuda')
    for colmax in (False, True):
        st = vt.ops.glm_stats(X, theta, y, wn, family, want_grad=False, want_colmax=colmax)
        assert torch.isnan(st[0]).all() and torch.isnan(st[1]).all(), family + ': z / resid not NaN'
        if family == 'gaussian':
            assert torch.equal(st[2], wn)
            continue
        assert torch.isnan(st[2]).all(), family + ': s not NaN'
        if colmax:
            sq, cmax = st[4]
            assert torch.isnan(sq).all() and torch.isnan(cmax.view(torch.float64)).all(), family + ': colmax'


# --------------------------------------------------------------------------- b. label-mirror invariance ----
def _mirror_problem(n, d, seed):
    """Rows spread over z in [-40, 40] (a random perpendicular part plus the wanted component along theta)."""
    rng = np.random.default_rng(seed)
    theta = rng.normal(size=d)
    u = theta / np.linalg.norm(theta)
    G = rng.normal(size=(n, d))
    t = rng.uniform(-40.0, 40.0, size=n)
    X = G - np.outer(G @ u, u) + np.outer(t / np.linalg.norm(theta), u)
    y = (rng.uniform(size=n) < 1.0 / (1.0 + np.exp(-np.clip(t, -700, 700)))).astype(np.float64)
    w = rng.uniform(0.5, 1.5, size=n)
    return X, y, w, theta


@pytest.mark.parametrize('precision', ['f64', 'f64_ozaki'])
def test_label_mirror_invariance(vt, precision):
    """(X, y) and (-X, 1 - y) are the same logistic model.  s and the gradient are the same bits, resid is exactly
    negated, and so are (f64) the Hessian, dopt_dhyper and the directional derivatives of orders 1..4: every sign flip
    cancels.  On the INT8 engine balanced digits are not sign-symmetric (-128 has no positive twin), so Hessian and
    dopt_dhyper are held to the parity bar there."""
    n, d, l2 = 3000, 40, 0.5
    X, y, w, theta = _mirror_problem(n, d, seed=11)
    z = X @ theta
    assert z.min() < -35 and z.max() > 35
    a = vt.objectives.GLMObjective(X, y, l2=l2, precision=precision)
    b = vt.objectives.GLMObjective(-X, 1.0 - y, l2=l2, precision=precision)
    sa, sb = a.vt_stats(theta, w, for_hessian=True), b.vt_stats(theta, w, for_hessian=True)
    assert torch.equal(sa['s'], sb['s']), 's differs'
    assert torch.equal(sa['resid'], -sb['resid']), 'resid not negated'
    assert torch.equal(sa['grad'], sb['grad']), 'gradient differs'
    pa = vt.HyperparameterSensitivityLinearApproximation(a, theta, w)
    pb = vt.HyperparameterSensitivityLinearApproximation(b, theta, w)
    same = torch.equal if precision == 'f64' else None
    for what, u, v in (('Hessian', a.vt_hessian(theta, w), b.vt_hessian(theta, w)),
                       ('Hessian at opt', pa.get_hessian_at_opt(), pb.get_hessian_at_opt()),
                       ('dopt_dhyper', pa.get_dopt_dhyper(), pb.get_dopt_dhyper())):
        u, v = torch.as_tensor(u), torch.as_tensor(v)
        if same is not None:
            assert same(u, v), '{} differs ({} entries)'.format(what, int((u != v).sum()))
        else:
            assert_close(u, v, what=what + ' (f64_ozaki)')
    rng = np.random.default_rng(12)
    dirs = [rng.normal(size=d) / math.sqrt(d) for _ in range(4)]
    for m in range(1, 5):
        da = a.vt_directional_derivative(theta, w, dirs[:m], [])
        db = b.vt_directional_derivative(theta, w, dirs[:m], [])
        assert torch.equal(da, db), 'directional derivative m={} differs'.format(m)


# ------------------------------------------------------------------------ c. separable data end to end ----
def _separable(n, d, seed):
    """y = 1 rows with z in [16, 36], y = 0 rows their mirror.  theta = 4 e_0, so z = 4 x_0 exactly; the other
    columns are Gaussian, scaled by e^((z - 16) / 2) so that every row carries about the same weight s |x|^2 and
    H stays well conditioned although s spans e^-16 .. e^-36."""
    rng = np.random.default_rng(seed)
    h = n // 2
    zh = rng.uniform(16.0, 36.0, size=h)
    Xh = np.empty((h, d))
    Xh[:, 0] = zh / 4.0
    Xh[:, 1:] = rng.normal(size=(h, d - 1)) * np.exp((zh - 16.0) / 2.0)[:, None]
    X = np.concatenate([Xh, -Xh])
    y = np.concatenate([np.ones(h), np.zeros(h)])
    theta = np.zeros(d)
    theta[0] = 4.0
    return X, y, theta


@pytest.mark.parametrize('d,precision', [(64, 'f64'), (512, 'f64_ozaki')])
def test_separable_logistic_end_to_end(vt, d, precision):
    n = 4096
    X, y, theta = _separable(n, d, seed=d)
    w = np.ones(n)
    z = X @ theta
    assert np.array_equal(z[:n // 2], 4.0 * X[:n // 2, 0]) and z[:n // 2].min() >= 16 and z[:n // 2].max() <= 36
    s_ref = highprec.glm_weight_mp(z, w, 'logistic')
    r_ref = highprec.glm_resid_mp(z, y, 'logistic')
    Hd = X.T @ (s_ref[:, None] * X)
    l2 = 1e-3 * float(np.min(np.diag(Hd)))          # small enough not to mask the weights
    H_ref = Hd + l2 * np.eye(d)
    assert np.linalg.cond(H_ref) <= 1e4
    obj = vt.objectives.GLMObjective(X, y, l2=l2, precision=precision)
    if precision == 'f64_ozaki':
        assert 'colmax' in obj.vt_stats(theta, w, for_hessian=True)      # the fused column-maxima pass runs
    st = obj.vt_stats(theta, w)
    _check(_host(st['s']), s_ref, 's (separable)')
    _check(_host(st['resid']), r_ref, 'resid (separable)')
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    assert_close(sens.get_hessian_at_opt(), H_ref, what='Hessian d={} {}'.format(d, precision))
    S = np.asarray(torch.as_tensor(sens.get_dopt_dhyper()).cpu())
    if d <= 64:
        S_ref = highprec.logistic_ij_ld(X, y, theta, w, l2=l2)[1].astype(np.float64)
    else:
        S_ref = -scipy.linalg.cho_solve(scipy.linalg.cho_factor(H_ref), (X * r_ref[:, None]).T)
    assert_close(S, S_ref, what='dopt_dhyper d={} {}'.format(d, precision))
    rng = np.random.default_rng(d + 1)
    A = rng.normal(size=(3, d))
    psi = vt.ObservationInfluence(obj, theta, w).influence(A)
    assert_close(psi, oinf.psi(X, y, w, theta, A, 'logistic', l2), what='influence d={} {}'.format(d, precision))
    Xd, zd = _dev(X), _dev(z)
    for q in range(1, 5):
        V = rng.normal(size=(q, d)) / math.sqrt(d)
        out = vt.ops.glm_dirderiv(Xd, zd, _dev(V), None, 'logistic')
        ref = X.T @ (highprec.glm_bderiv_mp(z, q + 1, 'logistic') * np.prod(X @ V.T, axis=1))
        assert_close(out, ref, what='glm_dirderiv q={} d={}'.format(q, d))
