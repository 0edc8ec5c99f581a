"""GPU tests of the per-observation influence pass (``vt_glm_influence``) and the ``ObservationInfluence`` API.

The kernel is held bit for bit to torch on integer data (``oracle/exact.py``: every partial sum an integer below
2^53), at every width where its dispatch changes, for K up to two passes beyond the per-pass limit and for N from one
row to more row blocks than the grid; padded and offset inputs and outputs inside sentinel-filled buffers must give
the contiguous result.  The API is held to the rtol 1e-8 parity bar against the numpy closed form
(``oracle/influence.py``) and against ``A @ get_dopt_dhyper()`` of the existing IJ class; the AMIP selection must
equal the numpy greedy run on the same psi, and the refit Newton on the data without the selected rows."""
import math

import numpy as np
import pytest
import torch

from conftest import assert_close
from oracle import exact, influence as oinf, models
from test_gpu_dispatch_edges import _launches, _sentinel_block, _sentinels_intact, _views

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _ref(X, c, V, alpha=-1.0):
    return alpha * ((X @ V.T) * c[:, None]).T


DIMS = [1, 7, 511, 512, 513, 1024, 1025, 2048, 2049, 4096, 8192]
KS = [1, 2, 3, 4, 5, 6, 7, 8, 9, 17]


@pytest.mark.parametrize('D', DIMS)
def test_influence_pass_is_exact_on_integer_data(vt, D):
    """N = 1, a ragged last row block (37 rows), and more row blocks than the grid (two CTAs per SM, 8 / CPT rows per
    block); every K: bit for bit against torch.  K <= max_directions(D) is one launch, larger K ceil(K / max)."""
    sms = vt.ops.device_info()['sm_count']
    qmax = vt.ops.glm_influence_max_directions(D)
    assert qmax == (8 if D <= 2048 else 2 if D <= 4096 else 1)
    cpt = max(1, -(-D // 512))
    rows = max(1, 8 // cpt)
    n_many = 2 * sms * 2 * rows + 3
    for N in (1, 37, n_many):
        X = _dev(exact.integer_design(D + N, N, D))
        c = _dev(exact.integer_vector(D + N + 1, N))
        for K in KS:
            V = _dev(exact.integer_design(K * D + N, K, D, vmax=exact.HMAX))
            out, nl = _launches(vt, lambda: vt.ops.glm_influence(X, c, V, alpha=-1.0))
            assert nl == math.ceil(K / qmax), (D, N, K, nl)
            ref = _ref(X, c, V)
            assert torch.equal(out, ref), 'D={} N={} K={}: {} entries differ'.format(D, N, K, int((out != ref).sum()))


def test_width_beyond_8192_is_refused(vt):
    from vittles_b200._cabi import check, ptr, require_cuda, stream
    X = torch.zeros((4, 8193), dtype=torch.float64, device='cuda')
    c = torch.ones(4, dtype=torch.float64, device='cuda')
    V = torch.ones((1, 8193), dtype=torch.float64, device='cuda')
    assert vt.ops.glm_influence_max_directions(8193) == 0
    with pytest.raises(ValueError):
        vt.ops.glm_influence(X, c, V)
    out = torch.empty((1, 4), dtype=torch.float64, device='cuda')
    with pytest.raises(ValueError):
        check(require_cuda().vt_glm_influence(ptr(X), 8193, 4, 8193, ptr(c), ptr(V), 1, 1.0, ptr(out), 4, stream()))
    with pytest.raises(ValueError):                                     # more directions than one pass takes
        check(require_cuda().vt_glm_influence(ptr(X), 8193, 4, 4096, ptr(c), ptr(V), 3, 1.0, ptr(out), 4, stream()))


@pytest.mark.parametrize('D', [77, 1000, 2500])
def test_padded_and_offset_layouts_are_bit_identical(vt, D):
    """Padded rows (ld = D + 1, D + 2), a base 8 bytes off alignment, a contiguous copy; the output as a block of a
    sentinel-filled wider buffer.  Random data: the results must equal the contiguous run bit for bit, twice."""
    N, K = 3001, 5
    g = torch.Generator(device='cuda').manual_seed(D)
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g) / math.sqrt(D)
    c = torch.randn(N, device='cuda', dtype=torch.float64, generator=g)
    V = torch.randn(K, D, device='cuda', dtype=torch.float64, generator=g)
    base = vt.ops.glm_influence(X, c, V, alpha=-1.0)
    assert torch.equal(vt.ops.glm_influence(X, c, V, alpha=-1.0), base), 'two calls differ'
    assert_close(base, _ref(X, c, V), rtol=1e-10, atol_scale=1e-13, what='random data')
    for lay, Xv in _views(X).items():
        big, out = _sentinel_block(K, N, 3, 1)
        vt.ops.glm_influence(Xv, c, V, alpha=-1.0, out=out)
        assert _sentinels_intact(big, (1, 1 + N)), '{} D={}: sentinels overwritten'.format(lay, D)
        assert torch.equal(out, base), '{} D={}: {} entries differ'.format(lay, D, int((out != base).sum()))


# ------------------------------------------------------------------------------------------------ the API ----
def _problem(family, n, d, seed, dup=False):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, d)) / math.sqrt(d)
    if dup:
        X[1::2] = X[0::2]
    theta_star = rng.normal(size=d)
    z = X @ theta_star
    if family == 'logistic':
        y = (rng.random(n) < 1.0 / (1.0 + np.exp(-z))).astype(np.float64)
    elif family == 'poisson':
        y = rng.poisson(np.exp(0.5 * z)).astype(np.float64)
    else:
        y = z + rng.normal(size=n)
    w = rng.uniform(0.5, 1.5, size=n)
    if dup:
        y[1::2] = y[0::2]
        w[1::2] = w[0::2]
    return X, y, w


@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
def test_influence_matches_closed_form_and_sensitivity_matrix(vt, family):
    n, d, l2 = 3000, 33, 0.1
    X, y, w = _problem(family, n, d, seed=5)
    theta = models.glm_newton(X, y, w, family, l2)
    A = np.random.default_rng(6).normal(size=(3, d))
    obj = vt.objectives.GLMObjective(X, y, family=family, l2=l2)
    inf = vt.ObservationInfluence(obj, theta, w, validate_optimum=True)
    psi = inf.influence(A)
    assert isinstance(psi, np.ndarray) and psi.shape == (3, n)
    assert_close(psi, oinf.psi(X, y, w, theta, A, family, l2), what='closed form')
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    assert_close(psi, A @ sens.get_dopt_dhyper(), what='A @ S')
    assert_close(inf.influence(A[1]), psi[1], what='one QoI')
    drop = [3, 17, 2500, 999]
    w0 = w.copy()
    w0[drop] = 0.0
    assert_close(inf.predict_opt_par_without(drop), sens.predict_opt_par_from_hyper_par(w0), what='prediction')
    with pytest.raises(ValueError):
        vt.ObservationInfluence(obj, theta + 0.1, w, validate_optimum=True)


def _newton(vt, obj, w, d):
    theta = torch.zeros(d, dtype=torch.float64, device='cuda')
    for _ in range(25):
        st = obj.vt_stats(theta, w)
        step = vt.ops.potrf(obj.vt_hessian(theta, w, st), overwrite=True).solve(st['grad'])
        theta = theta - step
        if float(torch.linalg.vector_norm(step)) < 1e-11:
            break
    return theta


@pytest.mark.parametrize('precision', ['auto', 'f64'])
def test_influence_at_1024_features(vt, precision):
    """D = 1024, N = 2e5 (the INT8 Hessian under 'auto'): parity with the closed form evaluated by torch on the
    device and with A @ S; during amip the peak device memory stays below a quarter of the 8 D N bytes of S."""
    n, d = 200_000, 1024
    X = vt.ops.synth_design(77, 0, n, d, 'cuda')
    theta_star = vt.ops.synth_theta(77, d, 'cuda')
    z = vt.ops.glm_stats(X, theta_star, torch.zeros(n, dtype=torch.float64, device='cuda'), None,
                         want_grad=False)[0]
    y = vt.ops.synth_bernoulli(77, 0, z)
    w = 0.5 + torch.rand(n, dtype=torch.float64, device='cuda', generator=torch.Generator('cuda').manual_seed(1))
    obj = vt.objectives.GLMObjective(X, y, l2=0.1, precision=precision)
    assert vt.ops.resolve_precision(precision, n, d, w) == ('f64_ozaki' if precision == 'auto' else 'f64')
    theta = _newton(vt, obj, w, d)
    A = torch.randn(4, d, dtype=torch.float64, device='cuda', generator=torch.Generator('cuda').manual_seed(2))
    inf = vt.ObservationInfluence(obj, theta, w)
    psi = inf.influence(A)
    assert psi.is_cuda and psi.shape == (4, n)
    zz = X @ theta
    p = torch.sigmoid(zz)
    H = X.T @ ((w * p * (1 - p))[:, None] * X) + 0.1 * torch.eye(d, dtype=torch.float64, device='cuda')
    ref = -(X @ torch.linalg.solve(H, A.T)).T * (p - y)[None, :]
    assert_close(psi, ref, what='closed form ({})'.format(precision))
    del H, ref, zz, p
    S = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w).get_dopt_dhyper()
    assert_close(psi, A @ S, what='A @ S ({})'.format(precision))
    del S
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    res = inf.amip((A[0], float(A[0] @ theta)), max_drop=0.01)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - base < 0.25 * 8 * d * n
    assert res.indices.size <= 2000


def _fit(vt, family, n, d, seed, l2=0.0, dup=False):
    X, y, w = _problem(family, n, d, seed, dup=dup)
    theta = models.glm_newton(X, y, w, family, l2)
    obj = vt.objectives.GLMObjective(X, y, family=family, l2=l2)
    return X, y, w, theta, obj


def _check_amip(res, psi, w, value, target, m):
    ref = oinf.amip_greedy(w * psi, value, target, m)
    assert res.n_drop == ref['n_drop']
    assert res.indices.tolist() == ref['indices'].tolist()
    assert res.predicted_value == ref['predicted_value']
    assert res.max_change == ref['max_change']
    assert res.direction == ref['direction']
    return ref


def test_amip_sign_flip_and_refit(vt):
    n, d = 2000, 6
    X, y, w, theta, obj = _fit(vt, 'logistic', n, d, seed=21)
    inf = vt.ObservationInfluence(obj, theta, w)
    j = int(np.argmin(np.abs(theta)))                     # the least certain coefficient: its sign is the QoI
    a = np.eye(d)[j]
    psi = inf.influence(a)
    for sgn in (1.0, -1.0):                               # both directions
        res = inf.amip((sgn * a, sgn * theta[j]), target=0.0, max_drop=0.2)
        ref = _check_amip(res, sgn * psi, w, sgn * theta[j], 0.0, 400)
        assert res.n_drop is not None, 'sign flip out of reach'
        assert ref['direction'] == ('decrease' if sgn * theta[j] > 0 else 'increase')
    res_c = inf.amip(lambda t: t[j], max_drop=0.2)       # the gradient by torch.func.grad
    res_p = inf.amip((a, theta[j]), max_drop=0.2)
    assert res_c.indices.tolist() == res_p.indices.tolist() and res_c.predicted_value == res_p.predicted_value
    # refit without the selected rows against Newton on the reduced data
    assert_close(inf.refit(res_p.indices), oinf.refit(X, y, w, res_p.indices), what='refit')
    # a finite target and an unreachable one
    tgt = theta[j] - 0.5 * np.sign(theta[j]) * abs(res_p.max_change)
    _check_amip(inf.amip((a, theta[j]), target=tgt, max_drop=400), psi, w, theta[j], tgt, 400)
    far = inf.amip((a, theta[j]), target=-np.sign(theta[j]) * 1e3, max_drop=3)
    _check_amip(far, psi, w, theta[j], -np.sign(theta[j]) * 1e3, 3)
    assert far.n_drop is None and far.indices.size == 3


def test_amip_exact_ties_and_zero_weights(vt):
    """Duplicated rows (same x, y, w) get bitwise equal psi: ties go to the lower index.  Zero-weight rows are never
    chosen."""
    n, d = 1000, 5
    X, y, w = _problem('logistic', n, d, seed=31, dup=True)
    w[::10] = 0.0
    w[1::10] = 0.0
    theta = models.glm_newton(X, y, w)
    obj = vt.objectives.GLMObjective(X, y)
    inf = vt.ObservationInfluence(obj, theta, w)
    a = np.eye(d)[0]
    psi = inf.influence(a)
    assert np.array_equal(psi[0::2], psi[1::2])
    tied = 0
    for target in (0.0, theta[0] + 5.0 * np.sign(theta[0])):
        res = inf.amip((a, theta[0]), target=target, max_drop=300)
        _check_amip(res, psi, w, theta[0], target, 300)
        assert not np.any(w[res.indices] == 0.0)
        pos = {int(i): k for k, i in enumerate(res.indices)}
        for i in pos:
            if i % 2 == 0 and i + 1 in pos:
                assert pos[i + 1] == pos[i] + 1
                tied += 1
    assert tied > 0
    with pytest.warns(UserWarning):
        inf.refit([0, 2], maxiter=1)
