#!/usr/bin/env python3
"""Generate ``tests/golden/*.npz`` by running the UNMODIFIED reference.

TEST INFRASTRUCTURE ONLY.  It needs a checkout of the reference
(rgiordan/vittles, the directory that holds the ``vittles`` package); the
tests do not, which is why the outputs are committed:

    python oracle/make_golden.py PATH/TO/VITTLES_CHECKOUT

How the reference runs here: ``autograd`` and ``paragami`` are not installed,
so ``oracle/refshim`` provides ``torch.func``-backed stand-ins for the handful
of names the reference imports, and ``scipy.sparse.linalg.cg`` is wrapped to
accept the removed ``atol='legacy'`` (``solver_lib.py:93``) with its documented
meaning (``rtol=tol, atol=0``).  The reference's SOURCE is untouched: every
golden value below is produced by ``vittles.*`` code imported from that
checkout.  Each case is also evaluated with the oracle restatement
and the two must agree to 1e-12 relative before anything is written.
"""
import os
import sys
import warnings

import numpy as np
import scipy as sp
import scipy.sparse
import scipy.sparse.linalg
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(ROOT, 'tests', 'golden')
if len(sys.argv) != 2:
    sys.exit('usage: python oracle/make_golden.py PATH/TO/VITTLES_CHECKOUT')
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(HERE, 'refshim'))
sys.path.insert(0, REF)

# ---- environment shim for the removed scipy keyword (not a source change) ----
_scipy_cg = sp.sparse.linalg.cg


def _cg_legacy(A, b, x0=None, tol=None, maxiter=None, M=None, callback=None, atol=None, rtol=None):
    if atol == 'legacy' or atol is None:
        atol = 0.0
    if rtol is None:
        rtol = 1e-5 if tol is None else tol
    return _scipy_cg(A, b, x0=x0, rtol=rtol, atol=atol, maxiter=maxiter, M=M, callback=callback)


sp.sparse.linalg.cg = _cg_legacy

import vittles  # noqa: E402  (the reference, from REF)
from vittles import solver_lib as ref_solver_lib  # noqa: E402
from vittles import sensitivity_lib as ref_sens  # noqa: E402

import oracle  # noqa: E402
from oracle import models, fixtures, bivariate  # noqa: E402,F401

assert vittles.__file__.startswith(REF + os.sep), vittles.__file__


def close(a, b, what, rtol=1e-12):
    a, b = np.asarray(a), np.asarray(b)
    scale = max(np.max(np.abs(b)), 1e-300)
    err = np.max(np.abs(a - b)) / scale
    assert err < rtol, '{}: oracle vs reference rel err {}'.format(what, err)
    return err


def save(name, **arrays):
    path = os.path.join(OUT, name + '.npz')
    np.savez_compressed(path, **arrays)
    print('wrote', os.path.relpath(path, ROOT), {k: np.asarray(v).shape for k, v in arrays.items()})


# --------------------------------------------------------------------------
def golden_solver():
    """tests/test_solver_lib.py:11-43 inputs (seed 101, d=10)."""
    np.random.seed(101)
    d = 10
    h = np.random.random((d, d))
    h = h + h.T + d * np.eye(d)
    v = np.random.random(d)
    V = np.random.random((d, 4))
    hs = sp.sparse.csc_matrix(h)
    out = dict(h=h, v=v, V=V)
    out['dense_v'] = ref_solver_lib.get_dense_cholesky_solver(h)(v)
    out['dense_V'] = ref_solver_lib.get_cholesky_solver(h)(V)
    out['sparse_v'] = ref_solver_lib.get_cholesky_solver(hs)(v)
    out['sparse_V'] = ref_solver_lib.get_sparse_cholesky_solver(hs)(V)
    out['cg_v'] = ref_solver_lib.get_cg_solver(lambda x: h @ x, d)(v)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        out['cg_maxiter1_v'] = ref_solver_lib.get_cg_solver(lambda x: hs @ x, d, cg_opts={'maxiter': 1})(v)
        assert any(issubclass(x.category, UserWarning) for x in w)
    out['cg_tol_v'] = ref_solver_lib.get_cg_solver(lambda x: h @ x, d, cg_opts={'tol': 1e-12})(v)
    # the reference's own assertion: all equal np.linalg.solve to 6 decimals
    truth = np.linalg.solve(h, v)
    for k in ['dense_v', 'sparse_v', 'cg_v']:
        np.testing.assert_array_almost_equal(out[k], truth)
    # oracle agreement
    o = oracle.solver_lib
    close(o.get_dense_cholesky_solver(h)(v), out['dense_v'], 'dense_v')
    close(o.get_cholesky_solver(h)(V), out['dense_V'], 'dense_V')
    close(o.get_cholesky_solver(hs)(V), out['sparse_V'], 'sparse_V')
    close(o.get_cg_solver(lambda x: h @ x, d)(v), out['cg_v'], 'cg_v')
    close(o.get_cg_solver(lambda x: h @ x, d, {'tol': 1e-12})(v), out['cg_tol_v'], 'cg_tol_v')
    x_it, info, nmv = o.cg_reference_iterates(lambda x: h @ x, v, rtol=1e-5)
    close(x_it, out['cg_v'], 'cg iterates restatement', rtol=1e-10)
    out['cg_v_iters'] = np.array(nmv)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        close(o.get_cg_solver(lambda x: hs @ x, d, {'maxiter': 1})(v), out['cg_maxiter1_v'], 'cg_maxiter1')
    save('solver_lib', **out)


# --------------------------------------------------------------------------
def golden_linear_quadratic():
    """tests/test_sensitivity_lib.py:454-613 on QuadraticModel(dim=3)."""
    model = fixtures.QuadraticModel(3)
    out = {}
    for tf_ in (False, True):
        for lf in (False, True):
            theta0, lam0 = model.get_default_flat_values(tf_, lf)
            obj = model.get_flat_objective(tf_, lf)
            sens = vittles.HyperparameterSensitivityLinearApproximation(
                objective_fun=obj, opt_par_value=theta0, hyper_par_value=lam0, validate_optimum=True)
            key = 't{}l{}'.format(int(tf_), int(lf))
            out[key + '_theta0'] = theta0
            out[key + '_lam0'] = lam0
            out[key + '_sens'] = sens.get_dopt_dhyper()
            out[key + '_hess'] = sens.get_hessian_at_opt()
            out[key + '_pred'] = sens.predict_opt_par_from_hyper_par(lam0 + 0.001)
            # the reference test's truth: jacobian of the closed-form optimum (:551-554)
            truth = torch.func.jacrev(model.get_flat_true_optimal_theta(tf_, lf))(torch.as_tensor(lam0)).numpy()
            np.testing.assert_array_almost_equal(truth, out[key + '_sens'])
            out[key + '_true_jac'] = truth
            # with the hyper-only objective (:496-504)
            sens2 = vittles.HyperparameterSensitivityLinearApproximation(
                objective_fun=obj, opt_par_value=theta0, hyper_par_value=lam0,
                hyper_par_objective_fun=model.get_flat_hyper_par_objective(tf_, lf))
            close(sens2.get_dopt_dhyper(), out[key + '_sens'], key + ' hyper-only objective')
            o = oracle.sensitivity.linear_sensitivity(obj, theta0, lam0, validate_optimum=True)
            close(o['sens'], out[key + '_sens'], key + ' sens')
            close(o['hessian'], out[key + '_hess'], key + ' hess')
    save('linear_quadratic', **out)


def golden_logistic_ij():
    """Config 1: logistic regression D=10, N=1000, IJ weight sensitivity via the
    reference class with autodiff Hessian and cross-Hessian (weights are the
    hyperparameter, notebook :345-371)."""
    seed, n, d = 20261017, 1000, 10
    X, y, _ = models.synth_logistic(seed, n, d)
    w = np.ones(n)
    theta = models.glm_newton(X, y, w)
    obj = models.glm_objective(X, y)
    sens = vittles.HyperparameterSensitivityLinearApproximation(
        objective_fun=obj, opt_par_value=theta, hyper_par_value=w, validate_optimum=True, grad_tol=1e-8)
    S = sens.get_dopt_dhyper()
    H = sens.get_hessian_at_opt()
    assert S.shape == (d, n)
    cf = models.glm_closed_form(X, y, theta, w)
    close(cf['hessian'], H, 'logistic closed-form H')
    close(-np.linalg.solve(cf['hessian'], cf['cross_hessian']), S, 'logistic closed-form S')
    o = oracle.sensitivity.linear_sensitivity(obj, theta, w, validate_optimum=True)
    close(o['sens'], S, 'logistic oracle S')
    w1 = w.copy()
    w1[::7] = 0.0
    pred = sens.predict_opt_par_from_hyper_par(w1)
    save('logistic_ij_cfg1', seed=np.array(seed), n=np.array(n), d=np.array(d), theta=theta,
         hessian=H, sens=S, w1=w1, pred=pred, X_head=X[:4], y_head=y[:16])
    # A second family + ridge, smaller, full compare
    X2, _, th2 = models.synth_logistic(seed + 1, 300, 7)
    y2 = np.random.RandomState(3).poisson(np.exp(X2 @ th2)).astype(np.float64)
    w2 = np.random.RandomState(4).uniform(0.5, 1.5, size=300)
    theta2 = models.glm_newton(X2, y2, w2, family='poisson', l2=0.3)
    obj2 = models.glm_objective(X2, y2, family='poisson', l2=0.3)
    sens2 = vittles.HyperparameterSensitivityLinearApproximation(
        objective_fun=obj2, opt_par_value=theta2, hyper_par_value=w2, validate_optimum=True)
    cf2 = models.glm_closed_form(X2, y2, theta2, w2, 'poisson', 0.3)
    close(-np.linalg.solve(cf2['hessian'], cf2['cross_hessian']), sens2.get_dopt_dhyper(), 'poisson S')
    save('poisson_ij', X=X2, y=y2, w=w2, theta=theta2, l2=np.array(0.3),
         hessian=sens2.get_hessian_at_opt(), sens=sens2.get_dopt_dhyper())


# --------------------------------------------------------------------------
def _ref_term_table(order):
    terms = [ref_sens._get_taylor_base_terms()]
    for k in range(1, order):
        nxt = []
        for t in terms[-1]:
            nxt += t.differentiate()
        terms.append(ref_sens._consolidate_terms(nxt))
    return terms


def golden_taylor():
    """tests/test_sensitivity_lib.py:616-726 (orders 1-3, Cholesky and CG) and
    the term tables of orders 1-5."""
    out = {}
    # term tables: compare the signature->prefactor maps
    ref_tabs = _ref_term_table(5)
    my_tabs = oracle.sensitivity.taylor_term_table(5)
    for k in range(5):
        ref_map = {}
        for t in ref_tabs[k]:
            key = (t.eps_order, tuple(t.eta_orders))
            ref_map[key] = ref_map.get(key, 0.0) + t.prefactor
        my_map = {(e, tuple(o)): p for p, e, o in my_tabs[k]}
        assert ref_map == my_map, (k, ref_map, my_map)
        flat = []
        for (e, o), p in sorted(ref_map.items()):
            flat.append([p, e] + list(o) + [0] * (5 - len(o)))
        out['table_order{}'.format(k + 1)] = np.array(flat, dtype=np.float64)
    print('term counts per order (reference, as listed):', [len(t) for t in ref_tabs])

    model = fixtures.QuadraticModel(3)
    eta0, eps0 = model.get_default_flat_values(True, True)
    obj = model.get_flat_objective(True, True)
    hess0 = torch.func.hessian(obj, argnums=0)(torch.as_tensor(eta0), torch.as_tensor(eps0)).numpy()
    eps1 = eps0 + 1e-1
    te = vittles.ParametricSensitivityTaylorExpansion.optimization_objective(
        objective_function=obj, input_val0=eta0, hyper_val0=eps0, order=3, hess0=hess0)
    derivs = te.evaluate_input_derivs(eps1 - eps0)
    series = te.evaluate_taylor_series(eps1)
    # the reference test's truth (:680-703)
    opt = model.get_flat_true_optimal_theta(True, True)
    j1 = torch.func.jacfwd(opt)
    j2 = torch.func.jacfwd(j1)
    j3 = torch.func.jacfwd(j2)
    e0t, de = torch.as_tensor(eps0), torch.as_tensor(eps1 - eps0)
    d1 = torch.einsum('ij,j', j1(e0t), de).numpy()
    d2 = torch.einsum('ijk,j,k', j2(e0t), de, de).numpy()
    d3 = torch.einsum('ijkl,j,k,l', j3(e0t), de, de, de).numpy()
    np.testing.assert_array_almost_equal(d1, derivs[0])
    np.testing.assert_array_almost_equal(d2, derivs[1])
    np.testing.assert_array_almost_equal(d3, derivs[2])
    # custom CG solver (:642-652)
    import autograd
    te_cg = vittles.ParametricSensitivityTaylorExpansion(
        estimating_equation=autograd.grad(obj, argnum=0), input_val0=eta0, hyper_val0=eps0, order=3,
        hess_solver=ref_solver_lib.get_cg_solver(lambda v: hess0 @ v, dim=3))
    derivs_cg = te_cg.evaluate_input_derivs(eps1 - eps0)
    g = torch.func.grad(obj, argnums=0)
    o_derivs = oracle.sensitivity.taylor_input_derivs(
        g, eta0, eps0, eps1 - eps0, 3, oracle.solver_lib.get_cholesky_solver(hess0))
    for k in range(3):
        close(o_derivs[k], derivs[k], 'quadratic taylor d{}'.format(k + 1))
    close(oracle.sensitivity.taylor_series(g, eta0, eps0, eps1, 3, oracle.solver_lib.get_cholesky_solver(hess0)),
          series, 'quadratic taylor series')
    out.update(q_eta0=eta0, q_eps0=eps0, q_eps1=eps1, q_hess0=hess0, q_derivs=np.array(derivs),
               q_derivs_cg=np.array(derivs_cg), q_series=series, q_true=np.array([d1, d2, d3]))

    # Config-5 family at a small size: prior hyperparameter eps = (log tau, mu)
    seed, n, d = 77, 400, 8
    X, y, _ = models.synth_logistic(seed, n, d)
    eps0h = np.array([np.log(2.0), 0.1])
    theta0 = models.hier_glm_newton(X, y, eps0h)
    objh = models.hier_glm_objective(X, y)
    eps1h = eps0h + np.array([0.3, -0.2])
    teh = vittles.ParametricSensitivityTaylorExpansion.optimization_objective(
        objective_function=objh, input_val0=theta0, hyper_val0=eps0h, order=3)
    dh = teh.evaluate_input_derivs(eps1h - eps0h)
    sh = teh.evaluate_taylor_series(eps1h)
    gh = torch.func.grad(objh, argnums=0)
    Hh = torch.func.hessian(objh, argnums=0)(torch.as_tensor(theta0), torch.as_tensor(eps0h)).numpy()
    oh = oracle.sensitivity.taylor_input_derivs(gh, theta0, eps0h, eps1h - eps0h, 3,
                                                oracle.solver_lib.get_cholesky_solver(Hh))
    for k in range(3):
        close(oh[k], dh[k], 'hier taylor d{}'.format(k + 1))
    # the expansion should track the true re-optimised parameter
    theta1 = models.hier_glm_newton(X, y, eps1h)
    assert np.linalg.norm(sh - theta1) < 0.2 * np.linalg.norm(theta0 + dh[0] - theta1)
    out.update(h_seed=np.array(seed), h_n=np.array(n), h_d=np.array(d), h_eps0=eps0h, h_eps1=eps1h,
               h_theta0=theta0, h_hess=Hh, h_derivs=np.array(dh), h_series=sh, h_theta1=theta1)
    save('taylor', **out)


# --------------------------------------------------------------------------
def golden_sparse_hessian():
    """tests/test_sparse_hessian_lib.py:15-113 and a small GMM-VB (config 3 family)."""
    out = {}
    f, x, inds, _ = fixtures.block_quadratic(10, 3, with_scales=False)
    sh = vittles.SparseBlockHessian(f, inds)
    hb = np.array(sh.get_block_hessian(x).todense())
    h0 = torch.func.hessian(f)(torch.as_tensor(x)).numpy()
    np.testing.assert_array_almost_equal(hb, h0)          # the reference's assertion (:53)
    close(oracle.sparse_hessian.block_hessian(f, x, inds).toarray(), hb, 'block hessian')
    out.update(bq_x=x, bq_inds=inds, bq_block_hess=hb)

    f2, x2, inds2, ginds2 = fixtures.block_quadratic(10, 3, with_scales=True)
    sh2 = vittles.SparseBlockHessian(f2, inds2)
    hfull = np.array(sh2.get_hessian(x2).todense())
    h02 = torch.func.hessian(f2)(torch.as_tensor(x2)).numpy()
    np.testing.assert_array_almost_equal(hfull, h02)       # (:113)
    hg = np.array(sh2.get_global_hessian(x2, global_inds=ginds2).todense())
    close(oracle.sparse_hessian.full_hessian(f2, x2, inds2).toarray(), hfull, 'full hessian')
    close(oracle.sparse_hessian.global_hessian(f2, x2, inds2, ginds2).toarray(), hg, 'global hessian')
    out.update(bqs_x=x2, bqs_inds=inds2, bqs_ginds=ginds2, bqs_full_hess=hfull, bqs_global_hess=hg)

    # GMM-VB small: N=12, K=3, d=2
    N, K, d = 12, 3, 2
    rng = np.random.RandomState(5)
    centers = rng.normal(size=(K, d)) * 3
    Xobs = centers[rng.randint(K, size=N)] + rng.normal(size=(N, d))
    fg = models.gmm_vb_objective(Xobs, K)
    xg = models.gmm_vb_fit(Xobs, K)                      # at the VB optimum: H is positive definite
    assert np.linalg.norm(torch.func.grad(fg)(torch.as_tensor(xg)).numpy()) < 1e-8
    indsg = models.gmm_vb_sparsity(N, K, d)
    shg = vittles.SparseBlockHessian(fg, indsg)
    hgm = np.array(shg.get_hessian(xg).todense())
    h0g = torch.func.hessian(fg)(torch.as_tensor(xg)).numpy()
    np.testing.assert_array_almost_equal(hgm, h0g)
    close(oracle.sparse_hessian.full_hessian(fg, xg, indsg).toarray(), hgm, 'gmm hessian')
    b = rng.normal(size=len(xg))
    sol = ref_solver_lib.get_cholesky_solver(sp.sparse.csc_matrix(shg.get_hessian(xg)))(b)
    close(np.linalg.solve(h0g, b), sol, 'gmm sparse solve', rtol=1e-9)
    out.update(gmm_X=Xobs, gmm_K=np.array(K), gmm_x=xg, gmm_hess=hgm, gmm_b=b, gmm_solve=sol)
    save('sparse_hessian', **out)


# --------------------------------------------------------------------------
def golden_lr_cov():
    """tests/test_lr_cov_lib.py:16-135 (dim 4, not-free parametrisation)."""
    true_mean, true_cov, true_info = fixtures.mvn_lr_fixture(4)
    f = models.mvn_kl_objective(true_mean, true_info)
    opt, Hcf = models.mvn_kl_closed_form(true_mean, true_info)
    lr = vittles.LinearResponseCovariances(objective_fun=f, opt_par_value=opt, validate_optimum=True, grad_tol=1e-12)

    def mean_fun(par):
        return par[:4]
    cov = lr.get_lr_covariance(mean_fun)
    np.testing.assert_array_almost_equal(true_cov, cov)     # the reference's assertion (:93)
    close(Hcf, lr.get_hessian_at_opt(), 'mvn closed-form H')
    jac = lr.get_moment_jacobian(mean_fun)
    cross = lr.get_lr_covariance_from_jacobians(jac[0:2], jac[2:4])
    close(oracle.lr_cov.lr_covariance(f, opt, mean_fun), cov, 'lr cov')
    save('lr_cov', true_mean=true_mean, true_cov=true_cov, true_info=true_info, opt=opt,
         hessian=lr.get_hessian_at_opt(), cov=cov, jac=jac, cross01_23=cross)


# --------------------------------------------------------------------------
def golden_bivariate():
    """tests/test_bivariate_sensitivity_lib.py:15-260 on a seeded version of its model
    (y ~ N(exp(x theta), 1), weights as the second hyperparameter), at an
    incompletely optimised theta, plus a Poisson GLM for the structured path."""
    import autograd
    from vittles.bivariate_sensitivity_lib import CrossSensitivity, OptimumChecker
    rng = np.random.RandomState(2024)
    dim, n_obs = 10, 200
    theta_true = rng.random_sample(dim) - 0.5
    x = rng.random_sample((n_obs, dim))
    x = x - np.mean(x, axis=0)
    y = np.exp(x @ theta_true) + rng.normal(size=n_obs)
    xt, yt = torch.as_tensor(x), torch.as_tensor(y)

    def w_obj(theta, w):
        resid = yt - torch.exp(xt @ theta)
        return 0.5 * torch.sum(w * resid ** 2)

    def pert_obj(theta, lam, w):
        return w_obj(theta, w) - torch.dot(lam, theta)

    w_base = np.ones(n_obs)
    theta = np.zeros(dim)
    grad_f = torch.func.grad(w_obj, argnums=0)
    hess_f = torch.func.hessian(w_obj, argnums=0)
    for _ in range(50):
        theta = theta - np.linalg.solve(hess_f(torch.as_tensor(theta), torch.as_tensor(w_base)).numpy(),
                                        grad_f(torch.as_tensor(theta), torch.as_tensor(w_base)).numpy())
    assert np.linalg.norm(grad_f(torch.as_tensor(theta), torch.as_tensor(w_base)).numpy()) < 1e-10
    theta_base = theta + 0.02 * (rng.random_sample(dim) - 0.5)          # "stopped early"
    hess_base = hess_f(torch.as_tensor(theta_base), torch.as_tensor(w_base)).numpy()
    lam_base = grad_f(torch.as_tensor(theta_base), torch.as_tensor(w_base)).numpy()
    new_w = np.ones(n_obs)
    new_w[1] = 0
    new_w[17] = 2.5
    dw = new_w - w_base
    dlambda = -1 * lam_base

    def solver(v):
        return np.linalg.solve(hess_base, v)
    g3 = autograd.jacobian(pert_obj, argnum=0)
    g3_t = torch.func.grad(pert_obj, argnums=0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        cs = CrossSensitivity(estimating_equation=g3, solver=solver, input_base=theta_base,
                              hyper1_base=lam_base, hyper2_base=w_base)
    di1, di2 = cs.get_di1(dlambda), cs.get_di2(dw)
    cross = cs.evaluate(dlambda, dw)
    o_cross, o_di1, o_di2 = oracle.bivariate.cross_sensitivity(g3_t, solver, theta_base, lam_base, w_base, dlambda, dw)
    close(o_di1, di1, 'bivariate di1')
    close(o_di2, di2, 'bivariate di2')
    close(o_cross, cross, 'bivariate cross')
    # the reference test's own assertions (:243-257)
    g2 = autograd.jacobian(w_obj, argnum=0)
    g2_t = torch.func.grad(w_obj, argnums=0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        oc = OptimumChecker(estimating_equation=g2, solver=solver, input_base=theta_base, hyper_base=w_base)
    newton_step = -1 * np.linalg.solve(hess_base, lam_base)
    np.testing.assert_array_almost_equal(newton_step, oc.get_newton_step())
    oc_out = dict(newton_step=oc.get_newton_step(), dinput_dhyper=oc.get_dinput_dhyper(dw),
                  correction=oc.correction(new_w), evaluate=oc.evaluate(new_w))
    o_oc = oracle.bivariate.optimum_checker(g2_t, solver, theta_base, w_base, new_w)
    for k in oc_out:
        close(o_oc[k], oc_out[k], 'optimum checker ' + k)
    out = dict(x=x, y=y, theta_base=theta_base, hess_base=hess_base, lam_base=lam_base, new_w=new_w,
               di1=di1, di2=di2, cross=cross, **{'oc_' + k: v for k, v in oc_out.items()})

    # Poisson GLM (structured objective family of this build) away from its optimum
    Xp = models.synth_design(31, 0, 300, 6)
    yp = rng.poisson(np.exp(Xp @ (0.5 * models.synth_theta(31, 6)))).astype(np.float64)
    wp = rng.uniform(0.5, 1.5, size=300)
    fp = models.glm_objective(Xp, yp, family='poisson', l2=0.2)
    thp = models.glm_newton(Xp, yp, wp, family='poisson', l2=0.2) + 0.01 * (rng.random_sample(6) - 0.5)
    Hp = torch.func.hessian(fp, argnums=0)(torch.as_tensor(thp), torch.as_tensor(wp)).numpy()
    new_wp = wp * rng.uniform(0.8, 1.2, size=300)

    def solver_p(v):
        return np.linalg.solve(Hp, v)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        ocp = OptimumChecker(estimating_equation=autograd.jacobian(fp, argnum=0), solver=solver_p,
                             input_base=thp, hyper_base=wp)
    ocp_out = dict(newton_step=ocp.get_newton_step(), dinput_dhyper=ocp.get_dinput_dhyper(new_wp - wp),
                   correction=ocp.correction(new_wp), evaluate=ocp.evaluate(new_wp))
    o_ocp = oracle.bivariate.optimum_checker(torch.func.grad(fp, argnums=0), solver_p, thp, wp, new_wp)
    for k in ocp_out:
        close(o_ocp[k], ocp_out[k], 'poisson optimum checker ' + k)
    out.update(p_X=Xp, p_y=yp, p_w=wp, p_l2=np.array(0.2), p_theta=thp, p_hess=Hp, p_new_w=new_wp,
               **{'p_oc_' + k: v for k, v in ocp_out.items()})
    save('bivariate', **out)


if __name__ == '__main__':
    os.makedirs(OUT, exist_ok=True)
    torch.set_default_dtype(torch.float64)
    golden_solver()
    golden_linear_quadratic()
    golden_logistic_ij()
    golden_taylor()
    golden_sparse_hessian()
    golden_lr_cov()
    golden_bivariate()
    print('all golden fixtures written; oracle == reference on every case')
