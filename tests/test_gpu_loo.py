"""GPU tests of approximate leave-one-out cross-validation: the quadratic forms h_n = |Linv x_n|^2 on both engines
(exact on integer data at every block edge and over several INT8 chunks, padded and offset layouts, bitwise
repeatable), the one-pass triangular solves in every regime of the Cholesky solve, and the API of
``ObservationInfluence`` (leverage, both predictors, held-out losses) against the numpy closed forms of
``oracle/loo.py`` and against refits."""
import warnings

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import exact, loo as oloo, models
from test_gpu_dispatch_edges import (_launches, _parity, _regime_K, _rnd, _sentinel_block,
                                     _sentinels_intact, apply_chunk_rows, solve_regime)

pytestmark = pytest.mark.gpu

ENGINES = ['f64', 'f64_ozaki']


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


@pytest.fixture(scope='module')
def sms(vt):
    return vt.ops.device_info()['sm_count']


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _int_lower(D, seed):
    """Lower-triangular integer Linv, |entries| <= 8."""
    return torch.tril(_dev(exact.integer_design(seed, D, D, vmax=exact.HMAX)))


def _int_rows(N, D, seed):
    """Integer design, |x| <= 16: |Linv x| <= 2^7 D, so every square and every sum of D squares stays below 2^53
    up to D = 4096, and float64 arithmetic in any order is exact."""
    return _dev(exact.integer_design(seed, N, D, vmax=16))


def _ref(Linv, X):
    return ((X @ Linv.T) ** 2).sum(1)


# ------------------------------------------------------------------ exactness ----
@pytest.mark.parametrize('engine', ENGINES)
@pytest.mark.parametrize('D', [1, 7, 127, 128, 129, 511, 512, 513, 1024, 1025, 2048, 2049, 4096])
def test_quad_forms_exact_on_integers(vt, engine, D):
    Linv = _int_lower(D, 10 + D)
    for N in (1, 63, 64, 65):
        X = _int_rows(N, D, 20 + N)
        h = vt.ops.quad_forms(Linv, X, precision=engine)
        assert torch.equal(h, _ref(Linv, X)), (engine, D, N)


@pytest.mark.parametrize('D', [1024, 1025, 2048])
def test_int8_quad_forms_over_many_chunks(vt, sms, D):
    """Three chunks and a ragged fourth.  D <= 1024: the converter warps slice chunk c + 1 during the GEMM of chunk c
    (one slicing launch for Linv, one for chunk 0, then GEMM + finish per chunk); wider rows: a slicing launch per
    chunk."""
    ch = apply_chunk_rows(10 ** 9, D, sms)
    N = 3 * ch + ch // 3 + 5
    nch = 4
    Linv = _int_lower(D, 30 + D)
    X = _int_rows(N, D, 31 + D)
    vt.ops.quad_forms(Linv, X[:64], precision='f64_ozaki')              # workspace and module loads
    h, launches = _launches(vt, lambda: vt.ops.quad_forms(Linv, X, precision='f64_ozaki'))
    assert launches == (2 + 2 * nch if D <= 1024 else 1 + 3 * nch), launches
    assert torch.equal(h, _ref(Linv, X))
    assert torch.equal(vt.ops.quad_forms(Linv, X, precision='f64'), h)


# -------------------------------------------------------------------- layouts ----
@pytest.mark.parametrize('engine', ENGINES)
@pytest.mark.parametrize('D', [129, 1024, 1025])
def test_quad_forms_layouts_and_repeatability(vt, engine, D):
    N = 3000
    g = torch.Generator(device='cuda').manual_seed(D)
    Linv = torch.tril(torch.randn(D, D, device='cuda', dtype=torch.float64, generator=g)) / D ** 0.5
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g)
    base = vt.ops.quad_forms(Linv, X, precision=engine)
    assert torch.equal(vt.ops.quad_forms(Linv, X, precision=engine), base), 'two calls'
    for pad in (1, 2):                                                  # ld = D + 1, D + 2
        Xp = torch.zeros(N, D + pad, device='cuda', dtype=torch.float64)
        Xp[:, :D] = X
        assert torch.equal(vt.ops.quad_forms(Linv, Xp[:, :D], precision=engine), base), ('pad', pad)
    Xo = torch.zeros(N, D + 1, device='cuda', dtype=torch.float64)     # base 8 bytes off 16-byte alignment
    Xo[:, 1:] = X
    assert torch.equal(vt.ops.quad_forms(Linv, Xo[:, 1:], precision=engine), base), 'offset base'
    big, view = _sentinel_block(1, N, 9, 5)
    out = view.reshape(-1)
    vt.ops.quad_forms(Linv, X, precision=engine, out=out)
    assert torch.equal(out, base) and _sentinels_intact(big, (5, 5 + N))
    _parity(base, _ref(Linv, X), what='{} D={}'.format(engine, D))


def test_quad_forms_argument_checks(vt):
    D, N = 8, 10
    Linv = torch.tril(_rnd(D, D, seed=1))
    X = _rnd(N, D, seed=2)
    for p in ('tf32', 'tf32x3'):
        with pytest.raises(ValueError):
            vt.ops.quad_forms(Linv, X, precision=p)
    for bad in (Linv[:, :7], Linv[:7, :7], _rnd(D + 1, D + 1, seed=3).tril()):
        with pytest.raises(ValueError):
            vt.ops.quad_forms(bad, X)
    up = Linv.clone()
    up[2, 5] = 1e-300
    with pytest.raises(ValueError):
        vt.ops.quad_forms(up, X)
    for out in (torch.empty(N + 1, dtype=torch.float64, device='cuda'),
                torch.empty(2 * N, dtype=torch.float64, device='cuda')[::2],
                torch.empty(N, 1, dtype=torch.float64, device='cuda')):
        with pytest.raises(ValueError):
            vt.ops.quad_forms(Linv, X, out=out)


# --------------------------------------------------------------------- solves ----
@pytest.mark.parametrize('D,kind', [(300, 'chain'), (1024, 'chain'), (1024, 'chain+1'), (2049, 'ragged'),
                                    (1024, 'inplace'), (300, 'inplace')])
def test_trsm_lower_in_every_regime(vt, sms, D, kind):
    K = 300 if (D == 300 and kind == 'inplace') else _regime_K(kind, D, sms)
    want = {'chain': 'chain', 'chain+1': 'oop512', 'ragged': 'oop512', 'inplace': 'inplace256'}[kind]
    assert solve_regime(D, K, sms) == want
    A = _rnd(D, D + 5, seed=D)
    H = A @ A.T / D + torch.eye(D, device='cuda', dtype=torch.float64)
    f = vt.ops.potrf(H)
    L = torch.tril(f.L)
    B = _rnd(D, K, seed=K)
    Y = f.solve_lower(B)
    _parity(Y, torch.linalg.solve_triangular(L, B, upper=False), atol_scale=1e-11, what='forward')
    Z = f.solve_lower(B, transpose=True)
    _parity(Z, torch.linalg.solve_triangular(L.T, B, upper=True), atol_scale=1e-11, what='backward')
    assert torch.equal(f.solve_lower(Y, transpose=True), f.solve(B)), 'forward then backward = potrs'
    Li = f.inverse_factor()
    assert bool((torch.triu(Li, 1) == 0).all())
    _parity(Li, torch.linalg.solve_triangular(L, torch.eye(D, device='cuda', dtype=torch.float64), upper=False),
            atol_scale=1e-11, what='inverse factor')


# ------------------------------------------------------------------------ API ----
def _problem(family, n, d, seed):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, d)) / np.sqrt(d)
    X[:, 0] = 1.0
    theta0 = rng.normal(size=d)
    z0 = X @ theta0
    if family == 'logistic':
        y = (rng.uniform(size=n) < 1 / (1 + np.exp(-z0))).astype(np.float64)
    elif family == 'poisson':
        y = rng.poisson(np.exp(np.clip(z0, -5, 3))).astype(np.float64)
    else:
        y = z0 + rng.normal(size=n)
    w = rng.uniform(0.5, 2.0, size=n)
    w[::11] = 0.0
    return X, y, w


def _influence(vt, X, y, w, family, l2, precision='auto'):
    theta = models.glm_newton(X, y, w, family, l2)
    obj = vt.objectives.GLMObjective(_dev(X), _dev(y), family=family, l2=l2, precision=precision)
    return vt.ObservationInfluence(obj, _dev(theta), weights=_dev(w)), theta


@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
@pytest.mark.parametrize('l2', [0.0, 0.1])
def test_api_against_the_oracle(vt, family, l2):
    X, y, w = _problem(family, 400, 6, seed=len(family) + int(10 * l2))
    oi, theta = _influence(vt, X, y, w, family, l2)
    ref = oloo.loo(X, y, w, theta, family, l2)
    assert_close(oi.leverage(), ref['leverage'], what='leverage')
    assert_close(oi.loo_linear_predictor('ij'), ref['z_ij'], what='z_ij')
    assert_close(oi.loo_linear_predictor('ns'), ref['z_ns'], what='z_ns')
    for method, z in (('ns', ref['z_ns']), ('ij', ref['z_ij'])):
        res = oi.approximate_cv(method)
        loss = oloo.glm_loss(z, y, family)
        ml, nbad = oloo.mean_loss(loss, w, np.isnan(z))
        assert res.method == method and res.n_invalid == nbad == 0
        assert_close(res.z_loo, z, what='z_loo ' + method)
        assert_close(res.loss, loss, what='loss ' + method)
        assert_close(res.leverage, ref['leverage'], what='leverage ' + method)
        assert_close(np.array([res.mean_loss]), np.array([ml]), what='mean_loss ' + method)
    z_ij = oi.loo_linear_predictor('ij').cpu().numpy()
    for n in (0, 5, 11, 399):                                   # row 11 has weight zero
        pred = oi.predict_opt_par_without([n]).cpu().numpy()
        assert_close(np.array([z_ij[n]]), np.array([X[n] @ pred]), what='IJ row {}'.format(n))


def test_gaussian_newton_step_is_exact_leave_one_out(vt):
    X, y, w = _problem('gaussian', 300, 5, seed=4)
    oi, _ = _influence(vt, X, y, w, 'gaussian', 0.1)
    z = oi.loo_linear_predictor('ns').cpu().numpy()
    exact_z = np.array([oloo.exact_loo(X, y, w, n, 'gaussian', 0.1) for n in range(300)])
    assert_close(z, exact_z, what='PRESS')


def test_singular_leave_one_out_row(vt):
    """Feature 5 is nonzero in row 7 only and l2 = 0: without row 7 the Hessian is singular."""
    X, y, w = _problem('gaussian', 200, 6, seed=5)
    X[:, 5] = 0.0
    X[7, 5] = 1.5
    w[7] = 1.0
    oi, theta = _influence(vt, X, y, w, 'gaussian', 0.0)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter('always')
        res = oi.approximate_cv('ns')
    assert len([r for r in rec if issubclass(r.category, UserWarning)]) == 1
    z = res.z_loo.cpu().numpy()
    assert np.isnan(z[7]) and np.isnan(res.loss.cpu().numpy()[7]) and res.n_invalid == 1
    assert np.isfinite(np.delete(z, 7)).all()
    ref = oloo.loo(X, y, w, theta, 'gaussian', 0.0)
    keep = np.arange(200) != 7
    assert_close(z[keep], ref['z_ns'][keep], what='other rows')
    ml, nbad = oloo.mean_loss(oloo.glm_loss(ref['z_ns'], y, 'gaussian'), w, np.isnan(ref['z_ns']))
    assert nbad == 1
    assert_close(np.array([res.mean_loss]), np.array([ml]), what='mean_loss')


def test_method_is_checked_before_device_work(vt):
    X, y, w = _problem('logistic', 100, 4, seed=6)
    oi, _ = _influence(vt, X, y, w, 'logistic', 0.1)
    for bad in ('NS', 'exact', None):
        with pytest.raises(ValueError):
            oi.approximate_cv(bad)
        with pytest.raises(ValueError):
            oi.loo_linear_predictor(bad)
    assert oi._h is None


# --------------------------------------------------------------- bench width ----
def test_bench_width_both_engines_and_memory(vt):
    """D = 1024, N = 2e5: 'auto' takes the INT8 engine.  Both engines against the torch closed form and each other.
    The engines' workspaces do not grow with N (the INT8 one is ~0.55 GB of digits for two chunks); beyond them,
    approximate_cv allocates O(N) vectors and L^{-1}, nothing of size D x N."""
    N, D = 200000, 1024
    assert vt.ops.resolve_precision('auto', N, D) == 'f64_ozaki'
    lib = vt._cabi.load()
    assert lib.vt_quad_forms_ozaki_workspace_bytes(N, D, 7) == lib.vt_quad_forms_ozaki_workspace_bytes(10 ** 7, D, 7)
    g = torch.Generator(device='cuda').manual_seed(9)
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g) / D ** 0.5
    theta = torch.randn(D, device='cuda', dtype=torch.float64, generator=g) * 0.3
    y = (torch.rand(N, device='cuda', dtype=torch.float64, generator=g) < torch.sigmoid(X @ theta)).double()
    w = torch.rand(N, device='cuda', dtype=torch.float64, generator=g) + 0.5
    results = {}
    for precision in ('auto', 'f64'):
        vt.ops.free_workspaces()
        obj = vt.objectives.GLMObjective(X, y, family='logistic', l2=1.0, precision=precision)
        oi = vt.ObservationInfluence(obj, theta, weights=w)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        res = oi.approximate_cv('ns')
        torch.cuda.synchronize()
        grown = torch.cuda.max_memory_allocated() - base
        ws = sum(b.numel() * 8 for (k, _), b in vt.ops._workspaces.items() if k in ('qf', 'qf_ozaki'))
        assert grown - ws < 8 * D * N / 4, (precision, grown, ws)
        results[precision] = (res, oi)
    (ra, oa), (rf, of) = results['auto'], results['f64']
    Li = oa.factor.inverse_factor()
    h_ref = ((X @ Li.T) ** 2).sum(1)
    _parity(oa._h, h_ref, what='h auto')
    _parity(of._h, h_ref, what='h f64')
    _parity(oa._h, of._h, what='h engines')
    _parity(ra.z_loo, rf.z_loo, what='z_loo engines')
    assert ra.n_invalid == rf.n_invalid == 0
    assert abs(ra.mean_loss - rf.mean_loss) <= 1e-8 * abs(rf.mean_loss)


# ---------------------------------------------------------------- conditioning ----
@pytest.mark.parametrize('kappa', [1e2, 1e6, 1e9])
@pytest.mark.parametrize('engine', ENGINES)
def test_forward_error_against_extended_precision(vt, kappa, engine):
    D, N = 64, 200
    rng = np.random.default_rng(int(np.log10(kappa)))
    Q, _ = np.linalg.qr(rng.normal(size=(D, D)))
    H = (Q * np.logspace(0, np.log10(kappa), D)) @ Q.T
    H = 0.5 * (H + H.T)
    X = rng.normal(size=(N, D))
    ref = oloo.quad_forms_ld(H, X)
    f = vt.ops.potrf(_dev(H))
    h = vt.ops.quad_forms(f.inverse_factor(), _dev(X), precision=engine).cpu().numpy()
    err = float(np.max(np.abs((h - ref) / ref)))
    err_np = float(np.max(np.abs((oloo.quad_forms(X, H) - ref) / ref)))
    # (a floor of a few ulps: at kappa = 1e2 both errors are at the rounding level)
    assert err <= 10 * err_np + 64 * 2.0 ** -53, (engine, kappa, err, err_np)
