"""GPU parity: ParametricSensitivityTaylorExpansion, the fused directional
derivative / Hessian-vector-product kernels and get_cg_solver over them
(SURVEY.md section 8a rows 4, 8-11; BASELINE config 5 family)."""
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


def test_term_tables_match_reference(vt, golden):
    from vittles_b200 import sensitivity_lib as sl
    g = golden('taylor')
    terms = [sl._get_taylor_base_terms()]
    for k in range(1, 5):
        nxt = []
        for t in terms[-1]:
            nxt += t.differentiate()
        terms.append(sl._consolidate_terms(nxt))
    for k in range(5):
        table = g['table_order{}'.format(k + 1)]
        ref = {(int(r[1]), tuple(int(x) for x in r[2:2 + k + 1])): r[0] for r in table}
        mine = {(t.eps_order, tuple(t.eta_orders)): t.prefactor for t in terms[k]}
        assert mine == ref


def test_quadratic_taylor_vs_golden(vt, golden):
    """tests/test_sensitivity_lib.py:616-726: orders 1-3 with a given Hessian,
    an autodiff Hessian and a custom CG solver."""
    from oracle.fixtures import QuadraticModel
    g = golden('taylor')
    model = QuadraticModel(3)
    obj = model.get_flat_objective(True, True)
    eta0, eps0, eps1 = g['q_eta0'], g['q_eps0'], g['q_eps1']
    for hess0 in (g['q_hess0'], None):
        te = vt.ParametricSensitivityTaylorExpansion.optimization_objective(
            objective_function=obj, input_val0=eta0, hyper_val0=eps0, order=3, hess0=hess0)
        assert te.get_max_order() == 3
        derivs = te.evaluate_input_derivs(eps1 - eps0)
        for k in range(3):
            assert_close(derivs[k], g['q_derivs'][k], rtol=1e-8, atol_scale=1e-10)
            assert_close(derivs[k], g['q_true'][k], rtol=1e-6, atol_scale=1e-8)
        assert_close(te.evaluate_taylor_series(eps1), g['q_series'], rtol=1e-9)
        d = g['q_derivs']
        assert_close(te.evaluate_taylor_series(eps1, max_order=1), eta0 + d[0], rtol=1e-9)
        assert_close(te.evaluate_taylor_series(eps1, max_order=2), eta0 + d[0] + d[1] / 2, rtol=1e-9)
        terms = te.evaluate_taylor_series_terms(eps1, max_order=3)
        assert_close(np.sum(terms, axis=0), g['q_series'], rtol=1e-9)
    hess_d = _dev(g['q_hess0'])
    solver = vt.solver_lib.get_cg_solver(lambda v: hess_d @ v, dim=3, cg_opts={'tol': 1e-13})
    te_cg = vt.ParametricSensitivityTaylorExpansion(
        estimating_equation=torch.func.grad(obj, argnums=0), input_val0=_dev(eta0), hyper_val0=_dev(eps0),
        order=3, hess_solver=solver)
    derivs = te_cg.evaluate_input_derivs(_dev(eps1 - eps0))
    for k in range(3):
        assert derivs[k].is_cuda
        assert_close(derivs[k], g['q_derivs'][k], rtol=1e-7, atol_scale=1e-9)
    with pytest.raises(ValueError):
        te_cg.evaluate_taylor_series(eps1, max_order=4)
    with pytest.raises(ValueError):
        te_cg.print_terms(k=7)


def test_structured_prior_taylor_vs_golden(vt, golden):
    """Config-5 family (GLM + Gaussian prior, eps = (log tau, mu)), order 3:
    fused directional-derivative kernels + GPU Cholesky vs the reference class
    run on autodiff."""
    from oracle import models
    g = golden('taylor')
    X, y, _ = models.synth_logistic(int(g['h_seed']), int(g['h_n']), int(g['h_d']))
    obj = vt.objectives.GLMPriorObjective(X, y, family='logistic')
    te = vt.ParametricSensitivityTaylorExpansion.optimization_objective(
        objective_function=obj, input_val0=g['h_theta0'], hyper_val0=g['h_eps0'], order=3)
    derivs = te.evaluate_input_derivs(g['h_eps1'] - g['h_eps0'])
    for k in range(3):
        assert_close(derivs[k], g['h_derivs'][k], rtol=1e-8, atol_scale=1e-10, what='d{}'.format(k + 1))
    assert_close(te.evaluate_taylor_series(g['h_eps1']), g['h_series'], rtol=1e-9)
    assert_close(obj.vt_hessian(_dev(g['h_theta0']), _dev(g['h_eps0'])), g['h_hess'], rtol=1e-10)
    # the same expansion with get_cg_solver over the fused Hessian-vector product
    hvp = obj.vt_hvp_fn(g['h_theta0'], g['h_eps0'])
    te_cg = vt.ParametricSensitivityTaylorExpansion(
        estimating_equation=obj, input_val0=g['h_theta0'], hyper_val0=g['h_eps0'], order=3,
        hess_solver=vt.solver_lib.get_cg_solver(hvp, int(g['h_d']), cg_opts={'tol': 1e-13}))
    derivs_cg = te_cg.evaluate_input_derivs(g['h_eps1'] - g['h_eps0'])
    for k in range(3):
        assert_close(derivs_cg[k], g['h_derivs'][k], rtol=1e-7, atol_scale=1e-9)


@pytest.mark.parametrize('n,d', [(3000, 96), (2500, 1024), (1200, 2048), (999, 33)])
def test_dirderiv_and_hvp_kernels_vs_oracle(vt, n, d):
    """vt_glm_hvp / vt_glm_dirderiv against the oracle's nested forward-mode
    JVPs of the autodiff gradient, incl. D = 2048 (config 5 width) and odd D."""
    from oracle import models, sensitivity as osens
    rng = np.random.RandomState(d)
    X = models.synth_design(5, 0, n, d)
    theta = 0.7 * rng.normal(size=d)
    y = (rng.uniform(size=n) < 0.5).astype(np.float64)
    eps = np.array([0.3, -0.1])
    obj = vt.objectives.GLMPriorObjective(X, y)
    g_torch = torch.func.grad(models.hier_glm_objective(X, y), argnums=0)
    dirs = [rng.normal(size=d) / np.sqrt(d) * 3 for _ in range(4)]
    de = [np.array([0.2, 0.5]), np.array([-0.4, 0.1])]
    for m, ne in [(0, 0), (1, 0), (2, 0), (3, 0), (4, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 1)]:
        ours = obj.vt_directional_derivative(theta, eps, dirs[:m], de[:ne])
        ref = osens.directional_derivative(g_torch, theta, eps, dirs[:m], de[:ne])
        assert_close(ours, ref, rtol=1e-8, atol_scale=1e-11, what='m={} n={}'.format(m, ne))
    hv = obj.vt_hvp_fn(theta, eps)(dirs[0])
    assert_close(hv, osens.directional_derivative(g_torch, theta, eps, dirs[:1], []), rtol=1e-9, atol_scale=1e-12)


def test_poisson_dirderiv_vs_oracle(vt):
    """The Poisson family's fused directional derivatives of orders 3-5 (q = 2..4 directions: b^(k) = exp for every
    k) against the oracle's nested forward-mode JVPs."""
    from oracle import models, sensitivity as osens
    n, d = 2000, 48
    rng = np.random.RandomState(4)
    X = models.synth_design(6, 0, n, d)
    theta = 0.7 * rng.normal(size=d)
    y = rng.poisson(np.exp(X @ theta)).astype(np.float64)
    eps = np.array([0.3, -0.1])
    obj = vt.objectives.GLMPriorObjective(X, y, family='poisson')
    g_torch = torch.func.grad(models.hier_glm_objective(X, y, family='poisson'), argnums=0)
    dirs = [rng.normal(size=d) / np.sqrt(d) * 3 for _ in range(4)]
    for m in (2, 3, 4):
        ours = obj.vt_directional_derivative(theta, eps, dirs[:m], [])
        ref = osens.directional_derivative(g_torch, theta, eps, dirs[:m], [])
        assert_close(ours, ref, rtol=1e-8, atol_scale=1e-11, what='poisson m={}'.format(m))


def test_weights_taylor_wls(vt):
    """tests/test_sensitivity_lib.py:838-901: order-4 expansion in the
    observation weights of a weighted least-squares fit, against nested JVPs of
    the closed-form solution; structured (gaussian GLM) and generic paths."""
    from oracle import fixtures
    objective, run_regression, x, y = fixtures.wls_fixture()
    n_obs = len(y)
    w1 = np.ones(n_obs)
    dw = np.random.RandomState(1).uniform(size=n_obs) - 0.5
    w1t, dwt = torch.as_tensor(w1), torch.as_tensor(dw)
    theta0 = run_regression(w1t).numpy()
    exact = run_regression(w1t + dwt).numpy()
    # truth: the oracle's Taylor terms (pinned to the reference in tests/test_oracle.py)
    from oracle import sensitivity as osens, solver_lib as osl
    g = torch.func.grad(objective, argnums=0)
    H = torch.func.hessian(objective, argnums=0)(torch.as_tensor(theta0), w1t).numpy()
    truths = osens.taylor_input_derivs(g, theta0, w1, dw, 4, osl.get_cholesky_solver(H))
    series = theta0 + truths[0] + truths[1] / 2 + truths[2] / 6 + truths[3] / 24
    assert np.linalg.norm(series - exact) < 0.05 * np.linalg.norm(theta0 + truths[0] - exact)
    # structured: 0.5 * sum w (z - y)^2  ==  gaussian GLM up to a term independent of theta
    obj = vt.objectives.GLMObjective(x, y, family='gaussian')
    te = vt.ParametricSensitivityTaylorExpansion.optimization_objective(obj, theta0, w1, order=4)
    assert_close(te.evaluate_taylor_series(w1 + dw), series, rtol=1e-8)
    derivs = te.evaluate_input_derivs(dw)
    for k in range(4):
        assert_close(derivs[k], truths[k], rtol=1e-7, atol_scale=1e-9)
    # generic torch objective on the device, truncated orders as in the reference test
    xd, yd = _dev(x), _dev(y)

    def objective_d(theta, w):
        return torch.sum(w * (yd - xd @ theta) ** 2)
    with pytest.warns(UserWarning):
        te2 = vt.ParametricSensitivityTaylorExpansion.optimization_objective(
            objective_d, theta0, w1, order=4, max_hyper_order=1, max_input_order=2)
    assert_close(te2.evaluate_taylor_series(w1 + dw), series, rtol=1e-8)
    with pytest.warns(UserWarning):
        te3 = vt.ParametricSensitivityTaylorExpansion.optimization_objective(
            objective_d, theta0, w1, order=3, forward_mode=False, max_hyper_order=1, max_input_order=2)
    assert_close(te3.evaluate_taylor_series(w1 + dw, max_order=3),
                 theta0 + truths[0] + truths[1] / 2 + truths[2] / 6, rtol=1e-8)


def test_cg_glm_iteration_parity(vt):
    """get_cg_solver over the fused HVP follows scipy's legacy-tolerance CG
    iterate for iterate: same matvec count, same answer, on a D=2048 problem."""
    from oracle import models, solver_lib as osl
    n, d = 6000, 2048
    X = models.synth_design(8, 0, n, d)
    y = (np.random.RandomState(0).uniform(size=n) < 0.5).astype(np.float64)
    theta = np.zeros(d)
    eps = np.array([np.log(0.5), 0.0])
    obj = vt.objectives.GLMPriorObjective(X, y)
    hvp = obj.vt_hvp_fn(theta, eps)
    H = X.T @ (0.25 * X) + 0.5 * np.eye(d)
    b = np.random.RandomState(1).normal(size=d)
    solve = vt.solver_lib.get_cg_solver(hvp, d)                # default legacy tol 1e-5
    x_gpu = solve(b)
    x_ref, info, nmv = osl.cg_reference_iterates(lambda v: H @ v, b, rtol=1e-5)
    assert info == 0 and solve.last_iterations == nmv
    assert_close(x_gpu, x_ref, rtol=1e-7, atol_scale=1e-9)
    x_tight = vt.solver_lib.get_cg_solver(hvp, d, {'tol': 1e-13})(b)
    assert_close(x_tight, np.linalg.solve(H, b), rtol=1e-8, atol_scale=1e-10)
