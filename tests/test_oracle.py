"""CPU: the oracle against (a) the golden outputs of the unmodified reference
(tests/golden/*.npz, made by oracle/make_golden.py) and (b) the closed-form
truths the reference's own tests assert (SURVEY.md section 4 / 8c)."""
import warnings

import numpy as np
import pytest
import scipy as sp
import scipy.sparse
import torch

from conftest import assert_close
import oracle
from oracle import models, fixtures


def test_solver_lib_oracle_vs_golden(golden):
    g = golden('solver_lib')
    o = oracle.solver_lib
    h, v, V = g['h'], g['v'], g['V']
    assert_close(o.get_dense_cholesky_solver(h)(v), g['dense_v'], rtol=1e-12)
    assert_close(o.get_cholesky_solver(h)(V), g['dense_V'], rtol=1e-12)
    hs = sp.sparse.csc_matrix(h)
    assert_close(o.get_cholesky_solver(hs)(v), g['sparse_v'], rtol=1e-12)
    assert_close(o.get_sparse_cholesky_solver(hs)(V), g['sparse_V'], rtol=1e-12)
    assert_close(o.get_cg_solver(lambda x: h @ x, 10)(v), g['cg_v'], rtol=1e-12)
    with pytest.warns(UserWarning):
        assert_close(o.get_cg_solver(lambda x: hs @ x, 10, {'maxiter': 1})(v), g['cg_maxiter1_v'], rtol=1e-12)
    with pytest.raises(ValueError):
        o.get_sparse_cholesky_solver(h)
    # the reference test's own assertion: everything equals np.linalg.solve to 6 decimals
    truth = np.linalg.solve(h, v)
    for k in ('dense_v', 'sparse_v', 'cg_v'):
        np.testing.assert_array_almost_equal(g[k], truth)
    x, info, nmv = o.cg_reference_iterates(lambda x: h @ x, v, rtol=1e-5)
    assert info == 0 and nmv == int(g['cg_v_iters'])
    assert_close(x, g['cg_v'], rtol=1e-10)


@pytest.mark.parametrize('key', ['t0l0', 't0l1', 't1l0', 't1l1'])
def test_linear_quadratic_oracle_vs_golden(golden, key):
    g = golden('linear_quadratic')
    model = fixtures.QuadraticModel(3)
    tf_, lf = key[1] == '1', key[3] == '1'
    res = oracle.sensitivity.linear_sensitivity(
        model.get_flat_objective(tf_, lf), g[key + '_theta0'], g[key + '_lam0'], validate_optimum=True)
    assert_close(res['sens'], g[key + '_sens'], rtol=1e-12)
    assert_close(res['hessian'], g[key + '_hess'], rtol=1e-12)
    np.testing.assert_array_almost_equal(res['sens'], g[key + '_true_jac'])       # reference :551-554
    pred = oracle.sensitivity.predict_from_hyper(g[key + '_theta0'], g[key + '_lam0'], res['sens'],
                                                 g[key + '_lam0'] + 0.001)
    assert_close(pred, g[key + '_pred'], rtol=1e-12)
    if not tf_ and not lf:
        # linear in lambda: the prediction is exact (reference :528-531)
        true1 = model.get_true_optimal_theta(g[key + '_lam0'] + 0.001)
        np.testing.assert_array_almost_equal(pred, true1)


def test_logistic_ij_oracle_vs_golden(golden):
    g = golden('logistic_ij_cfg1')
    seed, n, d = int(g['seed']), int(g['n']), int(g['d'])
    X, y, _ = models.synth_logistic(seed, n, d)
    assert np.array_equal(X[:4], g['X_head']) and np.array_equal(y[:16], g['y_head'])
    w = np.ones(n)
    cf = models.glm_closed_form(X, y, g['theta'], w)
    assert np.linalg.norm(cf['grad']) < 1e-8
    assert_close(cf['hessian'], g['hessian'], rtol=1e-11)
    assert_close(-np.linalg.solve(cf['hessian'], cf['cross_hessian']), g['sens'], rtol=1e-9, atol_scale=1e-12)
    res = oracle.sensitivity.linear_sensitivity(models.glm_objective(X, y), g['theta'], w)
    assert_close(res['sens'], g['sens'], rtol=1e-11, atol_scale=1e-13)
    assert_close(oracle.sensitivity.predict_from_hyper(g['theta'], w, res['sens'], g['w1']), g['pred'], rtol=1e-11)
    g2 = golden('poisson_ij')
    cf2 = models.glm_closed_form(g2['X'], g2['y'], g2['theta'], g2['w'], 'poisson', float(g2['l2']))
    assert_close(-np.linalg.solve(cf2['hessian'], cf2['cross_hessian']), g2['sens'], rtol=1e-9, atol_scale=1e-12)


def test_taylor_oracle_vs_golden(golden):
    g = golden('taylor')
    tabs = oracle.sensitivity.taylor_term_table(5)
    for k in range(5):
        ref = {(int(r[1]), tuple(int(x) for x in r[2:2 + k + 1])): r[0] for r in g['table_order{}'.format(k + 1)]}
        assert {(e, tuple(o)): p for p, e, o in tabs[k]} == ref
    # SURVEY.md section 3.2: 1, 3, 6, 11 right-hand-side terms for orders 1-4
    assert [sum(1 for p, e, o in t if o[-1] == 0) for t in tabs[:4]] == [1, 3, 6, 11]
    model = fixtures.QuadraticModel(3)
    gq = torch.func.grad(model.get_flat_objective(True, True), argnums=0)
    solve = oracle.solver_lib.get_cholesky_solver(g['q_hess0'])
    d = oracle.sensitivity.taylor_input_derivs(gq, g['q_eta0'], g['q_eps0'], g['q_eps1'] - g['q_eps0'], 3, solve)
    for k in range(3):
        assert_close(d[k], g['q_derivs'][k], rtol=1e-11, atol_scale=1e-13)
        np.testing.assert_array_almost_equal(d[k], g['q_true'][k])                 # reference :697-703
        np.testing.assert_array_almost_equal(g['q_derivs_cg'][k], g['q_true'][k], decimal=4)
    X, y, _ = models.synth_logistic(int(g['h_seed']), int(g['h_n']), int(g['h_d']))
    gh = torch.func.grad(models.hier_glm_objective(X, y), argnums=0)
    dh = oracle.sensitivity.taylor_input_derivs(gh, g['h_theta0'], g['h_eps0'], g['h_eps1'] - g['h_eps0'], 3,
                                                oracle.solver_lib.get_cholesky_solver(g['h_hess']))
    for k in range(3):
        assert_close(dh[k], g['h_derivs'][k], rtol=1e-10, atol_scale=1e-13)
    # the order-3 series is much closer to the re-optimised optimum than order 1
    e1 = np.linalg.norm(g['h_theta0'] + g['h_derivs'][0] - g['h_theta1'])
    e3 = np.linalg.norm(g['h_series'] - g['h_theta1'])
    assert e3 < 0.2 * e1


def test_sparse_hessian_oracle_vs_golden(golden):
    g = golden('sparse_hessian')
    f, x, inds, _ = fixtures.block_quadratic(10, 3, with_scales=False)
    assert_close(oracle.sparse_hessian.block_hessian(f, g['bq_x'], inds).toarray(), g['bq_block_hess'], rtol=1e-12,
                 atol_scale=1e-14)
    h0 = torch.func.hessian(f)(torch.as_tensor(g['bq_x'])).numpy()
    np.testing.assert_array_almost_equal(g['bq_block_hess'], h0)                   # reference :53
    f2, x2, inds2, ginds2 = fixtures.block_quadratic(10, 3, with_scales=True)
    assert_close(oracle.sparse_hessian.full_hessian(f2, g['bqs_x'], inds2).toarray(), g['bqs_full_hess'],
                 rtol=1e-12, atol_scale=1e-14)
    assert_close(oracle.sparse_hessian.global_hessian(f2, g['bqs_x'], inds2, ginds2).toarray(),
                 g['bqs_global_hess'], rtol=1e-12, atol_scale=1e-14)
    with pytest.raises(ValueError):
        oracle.sparse_hessian.check_sparsity_array(np.array([[0, 1], [1, 2]]))
    with pytest.raises(ValueError):
        oracle.sparse_hessian.global_hessian(f2, g['bqs_x'], inds2, np.array([0]))
    K = int(g['gmm_K'])
    fg = models.gmm_vb_objective(g['gmm_X'], K)
    inds = models.gmm_vb_sparsity(g['gmm_X'].shape[0], K, g['gmm_X'].shape[1])
    assert_close(oracle.sparse_hessian.full_hessian(fg, g['gmm_x'], inds).toarray(), g['gmm_hess'], rtol=1e-11,
                 atol_scale=1e-13)
    assert_close(np.linalg.solve(g['gmm_hess'], g['gmm_b']), g['gmm_solve'], rtol=1e-8, atol_scale=1e-10)


def test_lr_cov_oracle_vs_golden(golden):
    g = golden('lr_cov')
    f = models.mvn_kl_objective(g['true_mean'], g['true_info'])
    cov = oracle.lr_cov.lr_covariance(f, g['opt'], lambda par: par[:4])
    assert_close(cov, g['cov'], rtol=1e-11)
    np.testing.assert_array_almost_equal(g['true_cov'], cov)                      # reference :93
    opt, H = models.mvn_kl_closed_form(g['true_mean'], g['true_info'])
    assert_close(H, g['hessian'], rtol=1e-10, atol_scale=1e-13)
    hess, solve = oracle.lr_cov.base_values(f, g['opt'], validate=True, grad_tol=1e-12)
    j = oracle.lr_cov.moment_jacobian(lambda par: par[:4], g['opt'])
    assert_close(oracle.lr_cov.lr_covariance_from_jacobians(solve, 8, j[0:2], j[2:4]), g['cross01_23'], rtol=1e-10,
                 atol_scale=1e-12)
    for a, b in [(j.T, j), (j, j.T), (j[:, :, None], j), (j, j[:, :, None])]:
        with pytest.raises(ValueError):
            oracle.lr_cov.lr_covariance_from_jacobians(solve, 8, a, b)
    with pytest.raises(ValueError):
        oracle.lr_cov.base_values(f, g['opt'] + 0.01, validate=True, grad_tol=1e-12)


def test_bivariate_oracle_vs_golden(golden):
    """CrossSensitivity / OptimumChecker restatement vs the unmodified reference
    (bivariate_sensitivity_lib.py:57-115,118-205)."""
    import torch
    from oracle import bivariate
    g = golden('bivariate')
    xt, yt = torch.as_tensor(g['x']), torch.as_tensor(g['y'])

    def w_obj(theta, w):
        return 0.5 * torch.sum(w * (yt - torch.exp(xt @ theta)) ** 2)

    def pert_obj(theta, lam, w):
        return w_obj(theta, w) - torch.dot(lam, theta)

    def solver(v):
        return np.linalg.solve(g['hess_base'], v)
    w_base = np.ones(len(g['y']))
    cross, di1, di2 = bivariate.cross_sensitivity(torch.func.grad(pert_obj, argnums=0), solver, g['theta_base'],
                                                  g['lam_base'], w_base, -g['lam_base'], g['new_w'] - w_base)
    assert_close(di1, g['di1'], rtol=1e-10)
    assert_close(di2, g['di2'], rtol=1e-10)
    assert_close(cross, g['cross'], rtol=1e-10)
    oc = bivariate.optimum_checker(torch.func.grad(w_obj, argnums=0), solver, g['theta_base'], w_base, g['new_w'])
    for k in ('newton_step', 'dinput_dhyper', 'correction', 'evaluate'):
        assert_close(oc[k], g['oc_' + k], rtol=1e-10, atol_scale=1e-11)
    # the reference test's own check: the Lagrange direction reproduces a Newton step
    assert_close(oc['newton_step'], -np.linalg.solve(g['hess_base'], g['lam_base']), rtol=1e-10)


def test_synth_generator_statistics():
    X = models.synth_design(1, 0, 4000, 64)
    assert abs(X.mean()) < 2e-3 and abs(X.var() * 64 - 1.0) < 0.02
    a = models.synth_design(9, 100, 50, 16)
    b = models.synth_design(9, 0, 150, 16)[100:]
    assert np.array_equal(a, b)                      # any row range is reproducible
    u = models.synth_uniform(3, 0, 10000)
    assert 0.0 <= u.min() and u.max() < 1.0 and abs(u.mean() - 0.5) < 0.02


@pytest.mark.parametrize('nslices', [5, 6, 7])
def test_int8_slicing_model_is_error_free_and_bounded(nslices):
    """The arithmetic model of the INT8 engine (oracle/slicing.py): the balanced base-256 digits reproduce every
    operand to 8 S - 1 bits of its row scale, every accumulator stays inside INT32 at K = 1024 (the model asserts it),
    and the recombined product is within the analytic bound of the float64 product - without a GPU."""
    from oracle import slicing
    rng = np.random.RandomState(7)
    a = rng.normal(size=(40, 1024)) * np.exp(3 * rng.normal(size=(40, 1)))
    b = rng.normal(size=(24, 1024)) * np.exp(3 * rng.normal(size=(24, 1)))
    a[3] = 0.0
    d, sc = slicing.slice_rows(a, nslices)
    assert d.dtype == np.int8 and np.abs(d[0].astype(np.int64)).max() <= 65      # |x| / scale < 1: top digit <= 64 + carry
    assert np.all(np.frexp(sc)[0] == 0.5) and np.all(sc > np.max(np.abs(a), axis=1))
    resid = np.max(np.abs(a - slicing.reconstruct(d, sc)), axis=1)
    assert np.all(resid <= sc * 2.0 ** (-(8 * nslices - 1)) * (1 + 2.0 ** -40))   # round to nearest: half a unit
    # the digits are an exact positional representation of q = rint(x 2^(8S-2) / scale)
    q = sum(d[s].astype(np.int64) << (8 * (nslices - 1 - s)) for s in range(nslices))
    assert np.array_equal(q, np.rint(np.ldexp(a, (8 * nslices - 2 - np.frexp(sc)[1] + 1)[:, None])).astype(np.int64))
    out = slicing.sliced_gemm(a, b, nslices)
    exact = a @ b.T
    sa, sb = sc, slicing.slice_rows(b, nslices)[1]
    bound = slicing.error_bound(a.shape[1], nslices) * sa[:, None] * sb[None, :] + 1e-15 * np.abs(exact)
    assert np.all(np.abs(out - exact) <= bound)
    if nslices >= 6:
        np.testing.assert_allclose(out, exact, rtol=1e-8, atol=1e-12 * np.max(np.abs(exact)))


def test_int8_slicing_model_extreme_digits():
    """Every digit -128 (the largest magnitude a balanced digit takes) at the largest K a split-K part may have
    (16384 + one k-block): the INT32 accumulators of the model (asserted inside digits_gemm) do not overflow."""
    from oracle import slicing
    S, K = 7, 16384 + 128
    d = np.full((S, 2, K), -128, dtype=np.int8)
    out = slicing.digits_gemm(d, np.ones(2), d, np.ones(2))
    x = -2.0 * sum(2.0 ** (-8 * s) for s in range(S))                 # 2^-6 sum_s (-128) 2^-8s
    dropped = sum((2 * S - 1 - l) * 2.0 ** (2 - 8 * l) for l in range(S, 2 * S - 1))
    np.testing.assert_allclose(out, K * (x * x - dropped), rtol=1e-15)


def test_extended_precision_oracle_agrees_with_scipy_when_well_conditioned():
    """oracle/highprec.py (longdouble Cholesky solve) against the reference's cho_factor / cho_solve on a
    well-conditioned logistic problem: they agree to float64 rounding, and the longdouble residual is ~1e-19."""
    import scipy.linalg
    from oracle import models, highprec
    n, d = 400, 12
    X, y, _ = models.synth_logistic(3, n, d)
    w = np.ones(n)
    theta = models.glm_newton(X, y, w)
    H_ld, S_ld = highprec.logistic_ij_ld(X, y, theta, w)
    cf = models.glm_closed_form(X, y, theta, w)
    S = -scipy.linalg.cho_solve(scipy.linalg.cho_factor(cf['hessian']), cf['cross_hessian'])
    np.testing.assert_allclose(np.asarray(S_ld, dtype=np.float64), S, rtol=1e-10, atol=1e-13 * np.abs(S).max())
    G_ld = ((1 / (1 + np.exp(-(X.astype(np.longdouble) @ theta.astype(np.longdouble)))) - y)[:, None] * X).T
    resid = np.abs(H_ld @ S_ld + G_ld).max() / np.abs(G_ld).max()
    assert float(resid) < 1e-17


def test_integer_designs_are_exact_in_float64_and_in_the_int8_model():
    """oracle/exact.py: on the integer designs float64 is exact (numpy's BLAS product equals the Python-integer
    product), the largest shapes the GPU tests use stay below 2^53, and the INT8 engine's arithmetic model reproduces
    the exact product too - so the GPU tests may demand torch.equal of every engine."""
    from oracle import exact, slicing
    assert exact.hessian_bound(exact.MAX_N) < exact.EXACT_LIMIT
    assert exact.apply_bound(exact.MAX_D) < exact.EXACT_LIMIT
    for n, d in [(300, 37), (1001, 64)]:
        X = exact.integer_design(1, n, d)
        s = exact.square_weights(2, n)
        r = exact.integer_vector(3, n)
        Hinv = exact.integer_design(4, d, d, vmax=exact.HMAX)
        assert np.abs(X).max() == exact.XMAX and np.abs(r).max() == exact.RMAX and np.all(np.sqrt(s) % 1 == 0)
        H = (X * s[:, None]).T @ X
        S = -Hinv @ (X * r[:, None]).T
        assert np.array_equal(H.astype(np.int64).astype(object), exact.weighted_gram_int(X, s))
        assert np.array_equal(S.astype(np.int64).astype(object), exact.apply_int(Hinv, X, r))
        # the engine's model: the transposed weighted operand of the Hessian, the residual folded into the scale
        W = (X * np.sqrt(s)[:, None]).T.copy()
        dW, sW = slicing.slice_rows(W, 7)
        assert np.array_equal(slicing.digits_gemm(dW, sW, dW, sW), H)
        assert np.all(dW[2:] == 0)                            # two digits carry every entry: nothing is dropped
        dH, sH = slicing.slice_rows(Hinv, 7)
        dX, sX = slicing.slice_rows(X, 7)
        assert np.array_equal(-slicing.digits_gemm(dH, sH, dX, sX * r), S)
