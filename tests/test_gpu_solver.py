"""GPU parity: solver_lib (SURVEY.md section 8a rows 1-4) and the GEMM engine."""
import warnings

import numpy as np
import pytest
import scipy as sp
import scipy.linalg
import scipy.sparse
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


def _dev(a):
    return torch.as_tensor(np.asarray(a, dtype=np.float64), device='cuda')


def test_solver_lib_vs_golden(vt, golden):
    """tests/test_solver_lib.py:11-43 inputs; golden outputs from the reference."""
    g = golden('solver_lib')
    h, v, V = g['h'], g['v'], g['V']
    sl = vt.solver_lib
    assert_close(sl.get_dense_cholesky_solver(h)(v), g['dense_v'])
    assert_close(sl.get_cholesky_solver(h)(V), g['dense_V'])
    h_chol = sp.linalg.cho_factor(h)
    assert_close(sl.get_dense_cholesky_solver(None, h_chol)(v), g['dense_v'], rtol=1e-9)
    hs = sp.sparse.csc_matrix(h)
    assert_close(sl.get_cholesky_solver(hs)(v), g['sparse_v'])
    assert_close(sl.get_sparse_cholesky_solver(hs)(V), g['sparse_V'])
    with pytest.raises(ValueError):
        sl.get_sparse_cholesky_solver(h)
    # CG: default legacy tolerance 1e-5 -> same iterates as scipy, same iteration count
    cg = sl.get_cg_solver(lambda x: h @ x, 10)
    assert_close(cg(v), g['cg_v'], rtol=1e-8, atol_scale=1e-10)
    assert cg.last_iterations == int(g['cg_v_iters'])
    assert_close(sl.get_cg_solver(lambda x: hs @ x, 10, cg_opts={'tol': 1e-12})(v), g['cg_tol_v'], rtol=1e-8,
                 atol_scale=1e-10)
    with pytest.warns(UserWarning, match='CG exited with error code 1'):
        out = sl.get_cg_solver(lambda x: hs @ x, 10, cg_opts={'maxiter': 1})(v)
    assert_close(out, g['cg_maxiter1_v'], rtol=1e-8, atol_scale=1e-10)
    # device tensors in -> device tensors out, matvec called with device tensors
    hd = _dev(h)
    xd = sl.get_cg_solver(lambda x: hd @ x, 10, {'tol': 1e-13})(_dev(v))
    assert xd.is_cuda
    assert_close(xd, np.linalg.solve(h, v), rtol=1e-8)


def test_not_positive_definite_raises(vt):
    h = np.eye(5)
    h[3, 3] = -1.0
    with pytest.raises(np.linalg.LinAlgError):
        vt.solver_lib.get_dense_cholesky_solver(h)


@pytest.mark.parametrize('d,k', [(1, 1), (7, 3), (128, 5), (129, 130), (300, 1), (1024, 64), (1500, 257), (1023, 9),
                                 (1025, 1300), (2049, 1100)])
def test_cholesky_vs_scipy(vt, d, k):
    rng = np.random.RandomState(d * 7 + k)
    a = rng.normal(size=(d, d + 5))
    h = a @ a.T / d + np.eye(d)
    B = rng.normal(size=(d, k))
    solve = vt.solver_lib.get_cholesky_solver(h)
    ref = sp.linalg.cho_solve(sp.linalg.cho_factor(h), B)
    assert_close(solve(B), ref, rtol=1e-8, atol_scale=1e-11)
    assert_close(solve(B[:, 0]), ref[:, 0], rtol=1e-8, atol_scale=1e-11)
    L = torch.tril(solve.factor.L).cpu().numpy()
    assert_close(L, np.linalg.cholesky(h), rtol=1e-9, atol_scale=1e-12)


@pytest.mark.parametrize('tile', [0, 64, 128])
@pytest.mark.parametrize('am,bm', [('KC', 'KC'), ('KC', 'KS'), ('KS', 'KC'), ('KS', 'KS')])
@pytest.mark.parametrize('m,n,k', [(1, 1, 1), (5, 7, 3), (128, 128, 16), (130, 257, 1000), (300, 64, 4100)])
def test_gemm_engine(vt, am, bm, m, n, k, tile):
    rng = np.random.RandomState(m + n + k)
    A = rng.normal(size=(m, k))
    B = rng.normal(size=(n, k))
    C0 = rng.normal(size=(m, n))
    rs, cs = rng.normal(size=m), rng.normal(size=n)
    Ad = _dev(A if am == 'KC' else A.T.copy())
    Bd = _dev(B if bm == 'KC' else B.T.copy())
    out = _dev(C0.copy())
    vt.ops.gemm(Ad, Bd, am, bm, alpha=-0.5, beta=2.0, out=out, colscale=_dev(cs), rowscale=_dev(rs), tile=tile)
    ref = -0.5 * (rs[:, None] * (A @ B.T) * cs[None, :]) + 2.0 * C0
    assert_close(out, ref, rtol=1e-10, atol_scale=1e-13)


@pytest.mark.parametrize('tile', [0, 64, 128])
@pytest.mark.parametrize('d,k', [(64, 40), (200, 5000), (320, 70000)])
def test_gemm_lower_mirror_splitk(vt, d, k, tile):
    """Symmetric rank-k update: lower tiles only, mirrored, deterministic split-K."""
    rng = np.random.RandomState(d + k)
    Z = rng.normal(size=(k, d))
    ks = rng.uniform(0.5, 1.5, size=k)
    Zd = _dev(Z)
    out = vt.ops.gemm(Zd, Zd, 'KS', 'KS', kscale=_dev(ks), lower=True, mirror=True, tile=tile)
    out2 = vt.ops.gemm(Zd, Zd, 'KS', 'KS', kscale=_dev(ks), lower=True, mirror=True, tile=tile)
    assert torch.equal(out, out2)
    o = out.cpu().numpy()
    assert np.array_equal(o, o.T)
    assert_close(o, (Z * ks[:, None]).T @ Z, rtol=1e-10, atol_scale=1e-13)


def test_cg_solver_matrix_rhs(vt):
    """Extension over scipy/the reference: a (dim, K) right-hand side is solved column by column."""
    rng = np.random.RandomState(11)
    d = 40
    a = rng.normal(size=(d, d + 2))
    h = a @ a.T / d + np.eye(d)
    hd = _dev(h)
    solve = vt.solver_lib.get_cg_solver(lambda v: hd @ v if isinstance(v, torch.Tensor) else h @ v, d,
                                        cg_opts={'tol': 1e-13})
    B = rng.normal(size=(d, 3))
    assert_close(solve(B), np.linalg.solve(h, B), rtol=1e-8, atol_scale=1e-11)
    out = solve(_dev(B))
    assert isinstance(out, torch.Tensor) and out.is_cuda and out.shape == (d, 3)
    with pytest.raises(ValueError):
        solve(rng.normal(size=(d + 1, 3)))


def test_cg_single_column_matrix_keeps_its_shape(vt):
    """(dim, 1) in -> (dim, 1) out (ADVICE r01: the closure used to flatten it, which broke
    LinearResponseCovariances(factorize_hessian=False) with one moment and a scalar hyperparameter)."""
    rng = np.random.RandomState(3)
    d = 24
    a = rng.normal(size=(d, d + 2))
    h = a @ a.T / d + np.eye(d)
    hd = _dev(h)
    solve = vt.solver_lib.get_cg_solver(lambda v: hd @ v if isinstance(v, torch.Tensor) else h @ v, d, {'tol': 1e-13})
    b = rng.normal(size=(d, 1))
    out = solve(b)
    assert out.shape == (d, 1)
    assert_close(out, np.linalg.solve(h, b), rtol=1e-8, atol_scale=1e-11)
    assert solve(b[:, 0]).shape == (d,)
    # the two call sites of the advice
    lr = vt.LinearResponseCovariances(lambda p: 0.5 * p @ (hd @ p), np.zeros(d), factorize_hessian=False)
    J = rng.normal(size=(1, d))
    assert_close(lr.get_lr_covariance_from_jacobians(J, J), J @ np.linalg.solve(h, J.T), rtol=1e-7, atol_scale=1e-10)


def test_cg_columns_stop_where_scipy_stops(vt):
    """K right-hand sides side by side through ONE batched fused Hessian-vector product per iteration
    (GLMObjective.vt_hvp_fn, four columns per pass over X): every column performs exactly the matrix-vector products
    scipy's cg performs on it alone (oracle restatement of the legacy rule) and returns the same iterate."""
    from oracle import models, solver_lib as osl
    n, d, K = 3000, 96, 7
    X, y, _ = models.synth_logistic(17, n, d)
    w = np.ones(n)
    theta = models.glm_newton(X, y, w)
    cf = models.glm_closed_form(X, y, theta, w)
    H = cf['hessian']
    rng = np.random.RandomState(1)
    B = rng.normal(size=(d, K)) * np.logspace(0, 3, K)[None, :]
    B[:, 3] = 0.0                                            # a zero column: scipy returns it at once
    obj = vt.objectives.GLMObjective(X, y, family='logistic')
    hvp = obj.vt_hvp_fn(theta, w)
    assert hvp.batched
    assert_close(hvp(_dev(B)), H @ B, rtol=1e-10, atol_scale=1e-13)          # the batched product itself
    for tol in (1e-5, 1e-11):
        solve = vt.solver_lib.get_cg_solver(hvp, d, cg_opts={'tol': tol})
        out = solve(B)
        for k in range(K):
            xk, info, nmv = osl.cg_reference_iterates(lambda v: H @ v, B[:, k], rtol=tol)
            assert info == 0 and solve.iterations_per_column[k] == nmv, (k, solve.iterations_per_column, nmv)
            assert_close(out[:, k], xk, rtol=1e-7, atol_scale=1e-9 * max(1.0, tol / 1e-11))
        assert solve.last_iterations == max(solve.iterations_per_column)
    # many columns: the two-GEMM form of the batched product
    B2 = rng.normal(size=(d, 40))
    assert_close(hvp(_dev(B2)), H @ B2, rtol=1e-10, atol_scale=1e-13)
    sol = vt.solver_lib.get_cg_solver(hvp, d, cg_opts={'tol': 1e-12})(B2)
    assert_close(sol, np.linalg.solve(H, B2), rtol=1e-8, atol_scale=1e-10)


def test_cg_preconditioner_x0_and_callback(vt):
    """cg_opts are scipy's (``solver_lib.py:70,93`` forwards them verbatim): ``M`` as a Jacobi object, a diagonal
    sparse matrix, a dense matrix and a LinearOperator; ``x0``; ``callback``; non-convergence still warns."""
    import scipy.sparse
    import scipy.sparse.linalg as spla
    rng = np.random.RandomState(5)
    d = 60
    a = rng.normal(size=(d, d + 5))
    scale = np.logspace(0, 2.5, d)
    h = (a @ a.T / d + np.eye(d)) * scale[:, None] * scale[None, :]          # badly scaled: Jacobi helps a lot
    hd = _dev(h)
    mv = lambda v: hd @ v if isinstance(v, torch.Tensor) else h @ v          # noqa: E731
    b = rng.normal(size=d)
    ref = np.linalg.solve(h, b)
    plain = vt.solver_lib.get_cg_solver(mv, d, {'tol': 1e-10})
    x_plain = plain(b)
    minv = 1.0 / np.diag(h)
    variants = {'jacobi object': vt.solver_lib.JacobiPreconditioner(np.diag(h)),
                'sparse diagonal': scipy.sparse.diags(minv),
                'dense diagonal': np.diag(minv),
                'linear operator': spla.LinearOperator((d, d), matvec=lambda r: minv * r)}
    # scipy itself with the same preconditioner (legacy rule == rtol with atol = 0)
    x_sp, info = spla.cg(spla.LinearOperator((d, d), matvec=lambda v: h @ v), b, rtol=1e-10, atol=0.0,
                         M=scipy.sparse.diags(minv))
    assert info == 0
    for name, M in variants.items():
        solve = vt.solver_lib.get_cg_solver(mv, d, {'tol': 1e-10, 'M': M})
        x = solve(b)
        assert_close(x, ref, rtol=1e-6, atol_scale=1e-8, what=name)
        assert_close(x, x_sp, rtol=1e-6, atol_scale=1e-8, what=name + ' vs scipy')
        assert solve.last_iterations < plain.last_iterations, name
    dense_M = np.linalg.inv(h + 0.1 * np.diag(np.diag(h)))                   # a full approximate inverse
    s2 = vt.solver_lib.get_cg_solver(mv, d, {'tol': 1e-10, 'M': dense_M})
    assert_close(s2(np.stack([b, 2 * b], axis=1)), np.stack([ref, 2 * ref], axis=1), rtol=1e-6, atol_scale=1e-8)
    assert s2.last_iterations <= 12
    # x0 = the solution: converged before the first matrix-vector product of the loop
    s3 = vt.solver_lib.get_cg_solver(mv, d, {'tol': 1e-8, 'x0': ref})
    assert_close(s3(b), ref, rtol=1e-8, atol_scale=1e-10)
    assert s3.last_iterations == 0
    seen = []
    s4 = vt.solver_lib.get_cg_solver(mv, d, {'tol': 1e-10, 'callback': lambda xk: seen.append(np.array(xk))})
    s4(b)
    assert len(seen) == s4.last_iterations and np.allclose(seen[-1], x_plain)
    with pytest.warns(UserWarning, match='CG exited with error code 3'):
        vt.solver_lib.get_cg_solver(mv, d, {'maxiter': 3})(b)
    assert_close(x_plain, ref, rtol=1e-6, atol_scale=1e-8)


def test_linear_approximation_with_one_hyperparameter_and_a_cg_solver(vt):
    """ADVICE r01: a scalar hyperparameter gives a (D, 1) cross-Hessian; with a CG ``hess_solver`` the sensitivity
    matrix must stay (D, 1) (it used to collapse to 1-d and break the prediction)."""
    from vittles_b200.sensitivity_lib import EstimatingEquationLinearApproximation
    rng = np.random.RandomState(2)
    d = 12
    a = rng.normal(size=(d, d + 3))
    A = a @ a.T / d + np.eye(d)
    c = rng.normal(size=d)
    Ad, cd = _dev(A), _dev(c)

    def estimating_equation(theta, lam):          # root: theta = -A^{-1} c lam
        return Ad.to(theta.device) @ theta + cd.to(theta.device) * lam[0]
    lam0 = np.array([0.7])
    theta0 = -np.linalg.solve(A, c) * lam0[0]
    solver = vt.solver_lib.get_cg_solver(lambda v: Ad @ v if isinstance(v, torch.Tensor) else A @ v, d, {'tol': 1e-13})
    lin = EstimatingEquationLinearApproximation(estimating_equation, theta0, lam0, solver, validate_solution=True,
                                                solution_tol=1e-9)
    S = lin.get_dinput_dhyper()
    assert S.shape == (d, 1)
    assert_close(S[:, 0], -np.linalg.solve(A, c), rtol=1e-8, atol_scale=1e-11)
    assert_close(lin.predict_input_par_from_hyper_par(np.array([1.1])), -np.linalg.solve(A, c) * 1.1, rtol=1e-8,
                 atol_scale=1e-11)
