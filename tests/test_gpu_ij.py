"""GPU parity: Hessian assembly, Cholesky solve and the infinitesimal-jackknife
apply (SURVEY.md section 8a rows 1, 5, 6, 7) against the oracle and the golden
fixtures produced by the unmodified reference.  Everything goes through the
C ABI (``libvittles_b200.so``)."""
import numpy as np
import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


def _dev(a):
    return torch.as_tensor(np.asarray(a, dtype=np.float64), device='cuda')


def test_synth_matches_oracle_bitwise(vt):
    from oracle import models
    for (seed, row0, n, d) in [(20261017, 0, 1000, 10), (5, 12345, 257, 33), (9, 10**7 - 100, 100, 1024)]:
        Xd = vt.ops.synth_design(seed, row0, n, d, 'cuda')
        Xo = models.synth_design(seed, row0, n, d)
        assert np.array_equal(Xd.cpu().numpy(), Xo)
    th = vt.ops.synth_theta(77, 64, 'cuda')
    assert np.array_equal(th.cpu().numpy(), models.synth_theta(77, 64))


def test_config1_logistic_ij_vs_golden(vt, golden):
    """BASELINE config 1: logistic regression D=10, N=1000, IJ weight
    sensitivity through HyperparameterSensitivityLinearApproximation +
    Cholesky; golden values come from the reference class itself."""
    from oracle import models
    g = golden('logistic_ij_cfg1')
    seed, n, d = int(g['seed']), int(g['n']), int(g['d'])
    X, y, _ = models.synth_logistic(seed, n, d)
    obj = vt.objectives.GLMObjective(X, y, family='logistic')
    w = np.ones(n)
    sens = vt.HyperparameterSensitivityLinearApproximation(
        objective_fun=obj, opt_par_value=g['theta'], hyper_par_value=w, validate_optimum=True, grad_tol=1e-8)
    S = sens.get_dopt_dhyper()
    assert isinstance(S, np.ndarray) and S.shape == (d, n)
    assert_close(sens.get_hessian_at_opt(), g['hessian'], what='H')
    assert_close(S, g['sens'], what='dopt_dhyper')
    assert_close(sens.predict_opt_par_from_hyper_par(g['w1']), g['pred'], what='prediction')
    # same thing with device tensors in, device tensors out
    sens_d = vt.HyperparameterSensitivityLinearApproximation(obj, _dev(g['theta']), _dev(w))
    assert sens_d.get_dopt_dhyper().is_cuda
    assert_close(sens_d.get_dopt_dhyper(), g['sens'])


def test_config1_generic_autodiff_path(vt, golden):
    """The same problem through a plain torch callable: torch.func derivatives,
    GPU Cholesky solve of the (D, N) cross-Hessian."""
    from oracle import models
    g = golden('logistic_ij_cfg1')
    X, y, _ = models.synth_logistic(int(g['seed']), int(g['n']), int(g['d']))
    Xd, yd = _dev(X), _dev(y)

    def objective(theta, w):
        z = Xd @ theta
        return torch.sum(w * (torch.nn.functional.softplus(z) - yd * z))
    sens = vt.HyperparameterSensitivityLinearApproximation(
        objective, g['theta'], np.ones(int(g['n'])), validate_optimum=True)
    assert_close(sens.get_dopt_dhyper(), g['sens'])
    assert_close(sens.get_hessian_at_opt(), g['hessian'])


def test_poisson_ridge_weighted_vs_golden(vt, golden):
    g = golden('poisson_ij')      # odd D = 7: exercises the unaligned (8-byte) staging paths
    obj = vt.objectives.GLMObjective(g['X'], g['y'], family='poisson', l2=float(g['l2']))
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, g['theta'], g['w'], validate_optimum=True)
    assert_close(sens.get_hessian_at_opt(), g['hessian'])
    assert_close(sens.get_dopt_dhyper(), g['sens'])


def test_validate_optimum_raises(vt, golden):
    g = golden('logistic_ij_cfg1')
    from oracle import models
    X, y, _ = models.synth_logistic(int(g['seed']), int(g['n']), int(g['d']))
    obj = vt.objectives.GLMObjective(X, y)
    with pytest.raises(ValueError):
        vt.HyperparameterSensitivityLinearApproximation(obj, g['theta'] + 0.1, np.ones(1000), validate_optimum=True)
    with pytest.raises(ValueError):     # wrong Hessian shape (sensitivity_lib.py:386-387)
        vt.HyperparameterSensitivityLinearApproximation(obj, g['theta'], np.ones(1000), hessian_at_opt=np.eye(3))


@pytest.mark.parametrize('n,d,family', [(5000, 130, 'logistic'), (3001, 257, 'logistic'), (4096, 1024, 'logistic'),
                                        (777, 64, 'gaussian')])
def test_ij_against_closed_form_oracle(vt, n, d, family):
    """Sizes that cross tile boundaries (D = 130, 257: ragged 128-tiles; D = 1024:
    the benchmark width, several split-K parts)."""
    from oracle import models
    rng = np.random.RandomState(n + d)
    X = models.synth_design(11, 0, n, d)
    theta = 0.5 * rng.normal(size=d)
    if family == 'logistic':
        y = (rng.uniform(size=n) < 1 / (1 + np.exp(-X @ theta))).astype(np.float64)
    else:
        y = X @ theta + rng.normal(size=n)
    w = rng.uniform(0.5, 1.5, size=n)
    cf = models.glm_closed_form(X, y, theta, w, family, l2=0.1)
    obj = vt.objectives.GLMObjective(X, y, family=family, l2=0.1)
    st = obj.vt_stats(_dev(theta), _dev(w))
    assert_close(st['z'], cf['z'], rtol=1e-10)
    assert_close(st['resid'], cf['r'], rtol=1e-9, atol_scale=1e-13)
    assert_close(st['grad'], cf['grad'], rtol=1e-9)
    H = obj.vt_hessian(_dev(theta), _dev(w), st)
    assert_close(H, cf['hessian'], rtol=1e-10)
    assert torch.equal(H, H.T)
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    S_ref = -np.linalg.solve(cf['hessian'], cf['cross_hessian'])
    assert_close(sens.get_dopt_dhyper(), S_ref, what='S')
    w1 = w * rng.uniform(0.0, 2.0, size=n)
    assert_close(sens.predict_opt_par_from_hyper_par(w1), theta + S_ref @ (w1 - w), rtol=1e-8)


def test_hessian_bitwise_reproducible(vt):
    from oracle import models
    X = _dev(models.synth_design(3, 0, 20000, 256))
    s = torch.rand(20000, dtype=torch.float64, device='cuda')
    H1 = vt.ops.syrk_weighted(X, s)
    H2 = vt.ops.syrk_weighted(X, s)
    assert torch.equal(H1, H2)


def test_linear_function_derivatives(vt, golden):
    """get_opt_par_function: value, refusal away from lambda_0, first derivatives
    in both modes, NotImplementedError for second order
    (tests/test_sensitivity_lib.py:556-598)."""
    g = golden('linear_quadratic')
    from oracle.fixtures import QuadraticModel
    model = QuadraticModel(3)
    obj = model.get_flat_objective(True, True)
    theta0, lam0 = g['t1l1_theta0'], g['t1l1_lam0']
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta0, lam0, validate_optimum=True)
    S = g['t1l1_sens']
    get_opt_par = sens.get_opt_par_function()
    assert_close(get_opt_par(lam0), theta0)
    with pytest.raises(ValueError):
        get_opt_par(lam0 + 1)
    lam_t = _dev(lam0).requires_grad_(True)

    def fun_of_opt(lam):
        return torch.exp(torch.sum(get_opt_par(lam) + 0.1))
    val = fun_of_opt(lam_t)
    grad, = torch.autograd.grad(val, lam_t, create_graph=True)
    assert_close(grad, S.T @ np.full(3, float(val)), rtol=1e-9)
    with pytest.raises(NotImplementedError):
        torch.autograd.grad(grad.sum(), lam_t)
    import torch.autograd.forward_ad as fwAD
    delta = np.random.RandomState(0).uniform(size=3)
    with fwAD.dual_level():
        dual = fwAD.make_dual(_dev(lam0), _dev(delta))
        tangent = fwAD.unpack_dual(fun_of_opt(dual)).tangent
    assert_close(tangent, delta @ S.T @ np.full(3, float(val)), rtol=1e-9)


@pytest.mark.parametrize('key', ['t0l0', 't0l1', 't1l0', 't1l1'])
def test_quadratic_model_vs_golden(vt, golden, key):
    """tests/test_sensitivity_lib.py:454-613 (all free/not-free combinations)."""
    g = golden('linear_quadratic')
    from oracle.fixtures import QuadraticModel
    model = QuadraticModel(3)
    tf_, lf = key[1] == '1', key[3] == '1'
    obj = model.get_flat_objective(tf_, lf)
    theta0, lam0 = g[key + '_theta0'], g[key + '_lam0']
    for use_hess in (False, True):
        for use_cross in (False, True):
            for use_hyper in (False, True):
                kw = {}
                if use_hess:
                    kw['hessian_at_opt'] = g[key + '_hess']
                if use_cross:
                    kw['cross_hess_at_opt'] = -g[key + '_hess'] @ g[key + '_sens']
                if use_hyper:
                    kw['hyper_par_objective_fun'] = model.get_flat_hyper_par_objective(tf_, lf)
                sens = vt.HyperparameterSensitivityLinearApproximation(
                    obj, theta0, lam0, validate_optimum=True, **kw)
                assert_close(sens.get_dopt_dhyper(), g[key + '_sens'], rtol=1e-8, atol_scale=1e-11)
                assert_close(sens.get_dopt_dhyper(), g[key + '_true_jac'], rtol=1e-7, atol_scale=1e-10)
                assert_close(sens.predict_opt_par_from_hyper_par(lam0 + 0.001), g[key + '_pred'], rtol=1e-9)


@pytest.mark.parametrize('key', ['t0l0', 't0l1', 't1l0', 't1l1'])
def test_quadratic_model_through_patterns_vs_golden(vt, golden, key):
    """The reference's QuadraticModel test set-up (``tests/test_utils.py:23-75``: NumericArrayPattern(lb=-20) +
    FlattenFunctionInput) written with ``vittles_b200.patterns`` instead of paragami, through
    HyperparameterSensitivityLinearApproximation on the GPU, against the golden values the unmodified reference
    produced for the same four free / not-free combinations (``tests/test_sensitivity_lib.py:454-613``)."""
    pg = vt.patterns
    g = golden('linear_quadratic')
    dim = 3
    theta_free, lambda_free = key[1] == '1', key[3] == '1'
    theta_pattern = pg.NumericArrayPattern(shape=(dim,), lb=-20.0)
    lambda_pattern = pg.NumericArrayPattern(shape=(dim,), lb=-20.0)
    vec = np.linspace(0.1, 0.3, num=dim)
    matrix = np.outer(vec, vec) + np.eye(dim)

    def get_objective(theta, lam):
        A = torch.as_tensor(matrix, device=theta.device)
        return 0.5 * theta @ A @ theta + lam @ theta
    objective = pg.FlattenFunctionInput(get_objective, free=[theta_free, lambda_free], argnums=[0, 1],
                                        patterns=[theta_pattern, lambda_pattern])
    lam0_folded = np.linspace(0.5, 10.0, num=dim)
    theta0_folded = -1 * np.linalg.solve(matrix, lam0_folded)
    theta0 = theta_pattern.flatten(theta0_folded, theta_free)
    lam0 = lambda_pattern.flatten(lam0_folded, lambda_free)
    assert_close(theta0, g[key + '_theta0'], rtol=1e-13)
    assert_close(lam0, g[key + '_lam0'], rtol=1e-13)
    sens = vt.HyperparameterSensitivityLinearApproximation(objective, theta0, lam0, validate_optimum=True)
    assert_close(sens.get_hessian_at_opt(), g[key + '_hess'], rtol=1e-9, atol_scale=1e-12)
    assert_close(sens.get_dopt_dhyper(), g[key + '_sens'], rtol=1e-8, atol_scale=1e-11)
    assert_close(sens.predict_opt_par_from_hyper_par(lam0 + 0.001), g[key + '_pred'], rtol=1e-9)


def test_streamed_host_input_matches_resident(vt):
    """Pinned host X goes through the chunked-copy path (copies overlapped with
    the statistics + Hessian sweep); results must equal the resident path.  With odd D and n = 4100 the chunk that
    starts at row 1025 begins 8 bytes off the 16-byte alignment: the statistics pass stages it with plain loads."""
    from oracle import models
    for n, d in ((4096, 64), (4100, 65)):
        X, y, _ = models.synth_logistic(3, n, d)
        w = np.random.RandomState(0).uniform(0.5, 1.5, size=n)
        theta = models.glm_newton(X, y, w, l2=0.2)
        Xh = torch.as_tensor(X).pin_memory()
        obj_s = vt.objectives.GLMObjective(Xh, y, l2=0.2, stream_chunks=8)
        assert obj_s._host_src is not None
        if d % 2:
            assert any((obj_s.X[r0:].data_ptr() % 16) == 8 for r0 in (n * c // 8 for c in range(8)))
        sens_s = vt.HyperparameterSensitivityLinearApproximation(obj_s, theta, w, validate_optimum=True)
        assert not obj_s._pending and obj_s._host_src is None
        sens_r = vt.HyperparameterSensitivityLinearApproximation(vt.objectives.GLMObjective(X, y, l2=0.2), theta, w)
        assert_close(sens_s.get_hessian_at_opt(), sens_r.get_hessian_at_opt(), rtol=1e-12)
        assert_close(sens_s.get_dopt_dhyper(), sens_r.get_dopt_dhyper(), rtol=1e-9, atol_scale=1e-13)
        cf = models.glm_closed_form(X, y, theta, w, l2=0.2)
        assert_close(sens_s.get_dopt_dhyper(), -np.linalg.solve(cf['hessian'], cf['cross_hessian']))


@pytest.mark.parametrize('kappa', [1e2, 1e6, 1e9])
def test_conditioning_sweep(vt, kappa):
    """Forward error of the IJ sensitivities against an extended-precision oracle (oracle/highprec.py) as the Hessian
    becomes ill conditioned.  The reference substitutes with the Cholesky factor (``solver_lib.py:29``); the fused
    path multiplies by an explicit inverse only while a lower bound on kappa(H) keeps kappa eps far below the parity
    tolerance and substitutes otherwise - at every kappa its error must be comparable to the error scipy's
    ``cho_solve`` (the reference's own algorithm, float64) makes on the same inputs."""
    import scipy.linalg
    from oracle import models, highprec
    n, d = 3000, 40
    X, y, _ = models.synth_logistic(41, n, d)
    X = X * np.sqrt(d) * np.logspace(0, -0.5 * np.log10(kappa), d)[None, :]       # column scales: kappa(H) ~ kappa
    w = np.ones(n)
    theta = models.glm_newton(X, y, w, iters=100)
    H_ld, S_ld = highprec.logistic_ij_ld(X, y, theta, w)
    S_ref = np.asarray(S_ld, dtype=np.float64)
    true_kappa = np.linalg.cond(np.asarray(H_ld, dtype=np.float64))
    assert 0.05 * kappa < true_kappa < 200 * kappa
    cf = models.glm_closed_form(X, y, theta, w)
    S_scipy = -scipy.linalg.cho_solve(scipy.linalg.cho_factor(cf['hessian']), cf['cross_hessian'])

    def err(S):      # row-wise: the rows of S live on very different scales here
        return float(np.max(np.max(np.abs(np.asarray(S) - S_ref), axis=1) / np.max(np.abs(S_ref), axis=1)))
    e_scipy = err(S_scipy)
    obj = vt.objectives.GLMObjective(X, y, family='logistic')
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    e_ours = err(sens.get_dopt_dhyper())
    assert sens.hessian_cond_lower_bound <= 1.01 * true_kappa
    assert sens.used_explicit_inverse == (sens.hessian_cond_lower_bound <= 1e6)
    if kappa >= 1e9:
        assert not sens.used_explicit_inverse               # substitution, like the reference
    if kappa <= 1e2:
        assert sens.used_explicit_inverse
    floor = 50 * np.finfo(np.float64).eps
    assert e_ours <= 10 * max(e_scipy, floor), (kappa, e_ours, e_scipy)
    # the parity bar itself holds whenever kappa eps allows it at all
    if kappa <= 1e6:
        assert_close(sens.get_dopt_dhyper(), S_scipy, rtol=1e-8, atol_scale=1e-9, what='kappa {:g}'.format(kappa))


def test_default_engine_at_bench_width_vs_oracle(vt):
    """The DEFAULT path (precision='auto') at the width of BASELINE config 2 (D = 1024) and N = 2e5 observations:
    'auto' resolves to the INT8 error-free-slicing engine here, and the whole (D, N) result meets the rtol 1e-8
    parity bar against the oracle's closed form + the reference's cho_factor / cho_solve."""
    from oracle import models, solver_lib as osl
    n, d = 200_000, 1024
    assert vt.ops.resolve_precision('auto', n, d) == 'f64_ozaki'
    assert vt.ops.resolve_precision('auto', 1000, 10) == 'f64'
    X, y, _ = models.synth_logistic(20261017, n, d)
    w = np.ones(n)
    Xd, yd, wd = _dev(X), _dev(y), _dev(w)
    obj = vt.objectives.GLMObjective(Xd, yd, family='logistic')
    assert obj.precision == 'auto'
    theta = torch.zeros(d, dtype=torch.float64, device='cuda')
    for _ in range(30):                                     # Newton on the same kernels
        st = obj.vt_stats(theta, wd)
        step = vt.ops.potrf(obj.vt_hessian(theta, wd, st)).solve(st['grad'])
        theta = theta - step
        if float(torch.linalg.vector_norm(step)) < 1e-12:
            break
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, wd, validate_optimum=True, grad_tol=1e-8)
    cf = models.glm_closed_form(X, y, theta.cpu().numpy(), w)
    S_ref = -1 * osl.get_cholesky_solver(cf['hessian'])(cf['cross_hessian'])
    assert_close(sens.get_hessian_at_opt(), cf['hessian'], rtol=1e-9, what='H (auto engine)')
    assert_close(sens.get_dopt_dhyper(), S_ref, rtol=1e-8, atol_scale=1e-12, what='dopt_dhyper (auto engine, D=1024)')
    # the explicit DMMA engine on the same inputs
    obj64 = vt.objectives.GLMObjective(Xd, yd, family='logistic', precision='f64')
    sens64 = vt.HyperparameterSensitivityLinearApproximation(obj64, theta, wd)
    assert_close(sens64.get_dopt_dhyper(), S_ref, rtol=1e-8, atol_scale=1e-12, what='dopt_dhyper (f64 DMMA, D=1024)')


def test_large_results_reach_the_host_through_pinned_staging(vt, monkeypatch):
    """get_dopt_dhyper() on numpy / CPU inputs returns the (D, N) matrix on the host (``sensitivity_lib.py:230-231``):
    large results go through one pinned buffer, or - when the host cannot pin that much - through two pinned
    staging buffers into pageable memory.  Both paths are exercised here with small thresholds."""
    from vittles_b200 import _arrays
    g = torch.Generator(device='cuda').manual_seed(0)
    t = torch.randn(37, 1001, device='cuda', dtype=torch.float64, generator=g)
    ref = t.cpu()
    monkeypatch.setattr(_arrays, 'PINNED_STAGING_MIN_BYTES', 1024)
    out = _arrays.to_host(t)
    assert not out.is_cuda and out.is_pinned() and torch.equal(out, ref)
    assert torch.equal(_arrays.to_host(t.T), ref.T)                           # non-contiguous source
    monkeypatch.setattr(_arrays, 'STAGING_BYTES', 8 * 5000)                   # 8 chunks, ragged tail
    staged = _arrays._to_host_staged(t)
    assert not staged.is_cuda and staged.shape == ref.shape and torch.equal(staged, ref)
    assert isinstance(_arrays.as_kind(t, 'numpy'), np.ndarray)
