"""GPU tests of leave-one-group-out cross-validation: ``ops.group_loo`` on both engines (exact on integer data at
every block edge, group size and chunk boundary, padded and offset layouts, bitwise repeatable), and
``ObservationInfluence.approximate_cv(groups=...)`` / ``loo_linear_predictor(groups=...)`` against the closed forms
and refits of ``lgo_reference.py``, against leave-one-out at groups of one row, on a singular group, and in memory."""
import warnings

import numpy as np
import pytest
import torch

import lgo_reference as lgo
from conftest import assert_close
from oracle import exact, loo as oloo, models
from test_gpu_dispatch_edges import _launches, apply_chunk_rows

pytestmark = pytest.mark.gpu

ENGINES = ['f64', 'f64_ozaki']
OVERLAP = 32                                  # rows by which consecutive chunks overlap (GROUP_LOO_OVERLAP)
DMMA_CHUNK_BYTES = 256 << 20                  # U of one DMMA chunk (quad_forms_chunk_rows, dgemm.cu)


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
    return torch.tril(_dev(exact.integer_design(seed, D, D, vmax=exact.HMAX)))


def _int_rows(N, D, seed):
    return _dev(exact.integer_design(seed, N, D, vmax=16))


def _starts(N, sizes):
    """Group starts cycling through ``sizes`` (the last group cut at N)."""
    out, a, i = [0], 0, 0
    while a < N:
        a = min(N, a + sizes[i % len(sizes)])
        out.append(a)
        i += 1
    return torch.tensor(out, dtype=torch.int64, device='cuda')


def _groups(starts):
    """(G, 32) row indices of every group, padded with N (a zero row appended by the caller)."""
    s = starts.cpu().numpy()
    N, G = int(s[-1]), s.size - 1
    idx = np.full((G, 32), N, dtype=np.int64)
    for g in range(G):
        idx[g, :s[g + 1] - s[g]] = np.arange(s[g], s[g + 1])
    return torch.as_tensor(idx, device='cuda')


def _ref(Linv, X, starts, u, z):
    """(h, z + Q u) by batched products: exact on the integer data of these tests (every partial sum < 2^53)."""
    U = X @ Linv.T
    N = X.shape[0]
    idx = _groups(starts)
    Up = torch.cat([U, torch.zeros(1, U.shape[1], dtype=U.dtype, device=U.device)])
    up = torch.cat([u, torch.zeros(1, dtype=u.dtype, device=u.device)])
    Ug = Up[idx]                                                     # (G, 32, D)
    Q = Ug @ Ug.transpose(1, 2)
    t = (Q @ up[idx].unsqueeze(-1)).squeeze(-1)
    bound = (Q.abs() @ up[idx].abs().unsqueeze(-1)).squeeze(-1)
    assert float(bound.max()) + float(z.abs().max()) < 2.0 ** 52, 'test data outside the exact range'
    keep = idx < N
    h = torch.empty(N, dtype=torch.float64, device='cuda')
    zp = torch.empty(N, dtype=torch.float64, device='cuda')
    h[idx[keep]] = torch.diagonal(Q, dim1=1, dim2=2)[keep]
    zp[idx[keep]] = z[idx[keep]] + t[keep]
    return h, zp


def _int_vectors(N, seed):
    g = torch.Generator(device='cuda').manual_seed(seed)
    u = torch.randint(-2, 3, (N,), device='cuda', generator=g).double()
    z = torch.randint(-50, 51, (N,), device='cuda', generator=g).double()
    s = torch.rand(N, device='cuda', generator=g, dtype=torch.float64)
    return s, u, z


SIZES = {'1': [1], '2': [2], '31': [31], '32': [32], 'mixed': [1, 32, 5, 2, 31, 17, 3, 32, 8, 1, 1, 29]}


# ------------------------------------------------------------------ exactness ----
@pytest.mark.parametrize('engine', ENGINES)
@pytest.mark.parametrize('D', [1, 127, 128, 129, 1024, 1025, 2048])
@pytest.mark.parametrize('sizes', sorted(SIZES))
def test_group_loo_exact_on_integers(vt, engine, D, sizes):
    """N = 700 covers several blocks of the group kernel (224 group starts each) with groups across their edges."""
    N = 700
    Linv = _int_lower(D, 10 + D)
    X = _int_rows(N, D, 20 + D)
    starts = _starts(N, SIZES[sizes])
    s, u, z = _int_vectors(N, D)
    zp, h = vt.ops.group_loo(Linv, X, starts, s, u, z, 'ij', precision=engine)
    h_ref, zp_ref = _ref(Linv, X, starts, u, z)
    assert torch.equal(h, h_ref), (engine, D, sizes)
    assert torch.equal(zp, zp_ref), (engine, D, sizes)
    assert torch.equal(h, vt.ops.quad_forms(Linv, X, precision=engine))
    zn, hn = vt.ops.group_loo(Linv, X, starts, s, u, z, 'ns', precision=engine)
    assert torch.equal(hn, h)


def _chunks(N, ch):
    """Chunks of rows [c p, c p + ch), p = ch - 32, up to the first that reaches N."""
    p = ch - OVERLAP
    return 1 if ch >= N else 1 + -(-(N - ch) // p)


@pytest.mark.parametrize('D', [1024, 1025])
def test_int8_chunk_edges(vt, sms, D):
    """Three INT8 chunks and a ragged fourth.  A group of 17 rows, then groups of 32: every chunk start c (ch - 32)
    and every chunk end is a multiple of 32, so a 32-row group crosses each.  D <= 1024: one slicing launch for
    Linv, one for chunk 0, then GEMM + group kernel per chunk; wider rows: a slicing launch per chunk as well."""
    ch = apply_chunk_rows(10 ** 9, D, sms)
    N = 3 * ch + ch // 3 + 5
    nch = _chunks(N, ch)
    assert nch == 4
    Linv = _int_lower(D, 30 + D)
    X = _int_rows(N, D, 31 + D)
    starts = _starts(N, [17] + [32] * (N // 32 + 1))
    s, u, z = _int_vectors(N, 7)
    vt.ops.group_loo(Linv, X[:64], _starts(64, [32]), s[:64], u[:64], z[:64], 'ij', precision='f64_ozaki')
    (zp, h), launches = _launches(vt, lambda: vt.ops.group_loo(Linv, X, starts, s, u, z, 'ij', precision='f64_ozaki'))
    assert launches == (2 + 2 * nch if D <= 1024 else 1 + 3 * nch), launches
    h_ref, zp_ref = _ref(Linv, X, starts, u, z)
    assert torch.equal(h, h_ref)
    assert torch.equal(zp, zp_ref)
    zp2, h2 = vt.ops.group_loo(Linv, X, starts, s, u, z, 'ij', precision='f64')
    assert torch.equal(h2, h) and torch.equal(zp2, zp)


def test_dmma_chunk_edges(vt):
    """The DMMA engine's chunks (256 MB of U each) with mixed group sizes across their edges."""
    D = 1024
    ch = DMMA_CHUNK_BYTES // (8 * D)
    N = 3 * ch + ch // 3 + 5
    assert _chunks(N, ch) == 4
    Linv = _int_lower(D, 40)
    X = _int_rows(N, D, 41)
    starts = _starts(N, [17, 32, 32, 9, 32, 1, 32, 30])
    s, u, z = _int_vectors(N, 8)
    zp, h = vt.ops.group_loo(Linv, X, starts, s, u, z, 'ij', precision='f64')
    h_ref, zp_ref = _ref(Linv, X, starts, u, z)
    assert torch.equal(h, h_ref)
    assert torch.equal(zp, zp_ref)


# -------------------------------------------------------------------- layouts ----
@pytest.mark.parametrize('engine', ENGINES)
@pytest.mark.parametrize('D', [129, 1024])
def test_layouts_and_repeatability(vt, engine, D):
    N = 3000
    g = torch.Generator(device='cuda').manual_seed(D)
    Linv = torch.tril(torch.randn(D, D, device='cuda', dtype=torch.float64, generator=g)) / D ** 0.5
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g) / D ** 0.5
    s = 0.1 * torch.rand(N, device='cuda', dtype=torch.float64, generator=g)
    u = torch.randn(N, device='cuda', dtype=torch.float64, generator=g)
    z = torch.randn(N, device='cuda', dtype=torch.float64, generator=g)
    starts = _starts(N, SIZES['mixed'])
    for method in ('ns', 'ij'):
        base = vt.ops.group_loo(Linv, X, starts, s, u, z, method, precision=engine)
        assert bool(torch.isfinite(base[0]).all())
        again = vt.ops.group_loo(Linv, X, starts, s, u, z, method, precision=engine)
        assert torch.equal(again[0], base[0]) and torch.equal(again[1], base[1]), 'two calls'
        for pad in (1, 2):
            Xp = torch.zeros(N, D + pad, device='cuda', dtype=torch.float64)
            Xp[:, :D] = X
            got = vt.ops.group_loo(Linv, Xp[:, :D], starts, s, u, z, method, precision=engine)
            assert torch.equal(got[0], base[0]) and torch.equal(got[1], base[1]), ('pad', pad)
        Xo = torch.zeros(N, D + 1, device='cuda', dtype=torch.float64)
        Xo[:, 1:] = X
        got = vt.ops.group_loo(Linv, Xo[:, 1:], starts, s, u, z, method, precision=engine)
        assert torch.equal(got[0], base[0]) and torch.equal(got[1], base[1]), 'offset base'
    # the Newton-step form against its closed form in torch
    zn, h = vt.ops.group_loo(Linv, X, starts, s, u, z, 'ns', precision=engine)
    U = X @ Linv.T
    st = starts.tolist()
    for a, b in list(zip(st[:-1], st[1:]))[:40]:
        Q = U[a:b] @ U[a:b].T
        t = Q @ u[a:b]
        sq = s[a:b].sqrt()
        M = torch.eye(b - a, dtype=torch.float64, device='cuda') - sq[:, None] * Q * sq[None, :]
        want = z[a:b] + t + Q @ (sq * torch.linalg.solve(M, sq * t))
        assert_close(zn[a:b], want, rtol=1e-10, what='ns rows {}..{}'.format(a, b))


def test_argument_checks(vt):
    D, N = 8, 10
    g = torch.Generator(device='cuda').manual_seed(1)
    Linv = torch.tril(torch.randn(D, D, device='cuda', dtype=torch.float64, generator=g))
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g)
    v = torch.ones(N, dtype=torch.float64, device='cuda')
    good = _starts(N, [3])
    n0 = vt.ops.launch_count()
    for p in ('tf32', 'tf32x3'):
        with pytest.raises(ValueError):
            vt.ops.group_loo(Linv, X, good, v, v, v, 'ns', precision=p)
    with pytest.raises(ValueError):
        vt.ops.group_loo(Linv, X, good, v, v, v, 'exact')
    up = Linv.clone()
    up[2, 5] = 1e-300
    with pytest.raises(ValueError):
        vt.ops.group_loo(up, X, good, v, v, v, 'ns')
    for bad in ([0, 3, 3, 10], [0, 5, 4, 10], [1, 5, 10], [0, 5, 9], [0, 5, 11]):
        with pytest.raises(ValueError):
            vt.ops.group_loo(Linv, X, torch.tensor(bad, device='cuda'), v, v, v, 'ns')
    Xl = torch.randn(40, D, device='cuda', dtype=torch.float64, generator=g)
    vl = torch.ones(40, dtype=torch.float64, device='cuda')
    with pytest.raises(ValueError):
        vt.ops.group_loo(Linv, Xl, torch.tensor([0, 33, 40], device='cuda'), vl, vl, vl, 'ij')
    with pytest.raises(TypeError):
        vt.ops.group_loo(Linv, X, good.double(), v, v, v, 'ns')
    with pytest.raises(ValueError):
        vt.ops.group_loo(Linv, X, good, v[:9], v, v, 'ns')
    assert vt.ops.launch_count() == n0


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


def _labels(n, seed):
    rng = np.random.default_rng(seed)
    sizes = rng.integers(1, 33, size=n)
    return np.repeat(np.arange(sizes.size) * 2 + 5, sizes)[:n]


def _influence(vt, X, y, w, family, l2, precision):
    theta = models.glm_newton(X, y, w, family, l2)
    obj = vt.objectives.GLMObjective(_dev(X), _dev(y), family=family, l2=l2, precision=precision)
    return vt.ObservationInfluence(obj, _dev(theta), weights=_dev(w)), theta


@pytest.mark.parametrize('precision', ENGINES)
@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
@pytest.mark.parametrize('l2', [0.0, 0.1])
def test_api_against_the_oracle_and_refits(vt, precision, family, l2):
    X, y, w = _problem(family, 400, 6, seed=len(family) + int(10 * l2))
    labels = _labels(400, seed=3)
    oi, theta = _influence(vt, X, y, w, family, l2, precision)
    starts = np.concatenate([[0], np.nonzero(np.diff(labels))[0] + 1, [400]])
    ref = lgo.group_loo(X, y, w, theta, starts, family, l2)
    for method, zr in (('ns', ref['z_ns']), ('ij', ref['z_ij'])):
        res = oi.approximate_cv(method, groups=labels)
        loss = oloo.glm_loss(zr, y, family)
        ml, nbad = oloo.mean_loss(loss, w, np.isnan(zr))
        assert res.method == method and res.n_invalid == nbad == 0
        assert_close(res.z_loo, zr, what='z_loo ' + method)
        assert_close(res.loss, loss, what='loss ' + method)
        assert_close(res.leverage, ref['leverage'], what='leverage ' + method)
        assert_close(np.array([res.mean_loss]), np.array([ml]), what='mean_loss ' + method)
        assert_close(oi.loo_linear_predictor(method, groups=torch.as_tensor(labels)), zr, what='predictor ' + method)
    z_ns = oi.loo_linear_predictor('ns', groups=list(labels)).cpu().numpy()
    z_ij = oi.loo_linear_predictor('ij', groups=labels).cpu().numpy()
    for a, b in list(zip(starts[:-1], starts[1:]))[::5]:
        rows = np.arange(a, b)
        assert_close(z_ns[rows], lgo.newton_step_without_rows(X, y, w, theta, rows, family, l2), rtol=1e-9,
                     what='one Newton step without rows {}..{}'.format(a, b))
        if family == 'gaussian':
            assert_close(z_ns[rows], lgo.exact_lgo(X, y, w, rows, family, l2), rtol=1e-9,
                         what='exact refit without rows {}..{}'.format(a, b))
        pred = oi.predict_opt_par_without(rows).cpu().numpy()
        assert_close(z_ij[rows], X[rows] @ pred, what='IJ rows {}..{}'.format(a, b))


@pytest.mark.parametrize('precision', ENGINES)
@pytest.mark.parametrize('family', ['logistic', 'gaussian'])
def test_singletons_reproduce_leave_one_out(vt, precision, family):
    X, y, w = _problem(family, 500, 7, seed=8)
    oi, _ = _influence(vt, X, y, w, family, 0.1, precision)
    for method in ('ns', 'ij'):
        one = oi.approximate_cv(method)
        grp = oi.approximate_cv(method, groups=np.arange(500) * 3)
        assert_close(grp.z_loo, one.z_loo, rtol=1e-12, what='z_loo ' + method)
        assert_close(grp.leverage, one.leverage, rtol=1e-12, what='leverage ' + method)
        assert abs(grp.mean_loss - one.mean_loss) <= 1e-12 * abs(one.mean_loss)
        assert grp.n_invalid == one.n_invalid == 0


def test_singular_group(vt):
    """Feature 5 is nonzero on the rows 5 .. 9 (group 1) only and l2 = 0: without the group the Hessian is
    singular."""
    X, y, w = _problem('gaussian', 200, 6, seed=5)
    labels = np.repeat(np.arange(40), 5)
    X[:, 5] = 0.0
    X[5:10, 5] = [1.5, -0.5, 2.0, 1.0, 0.25]
    w[5:10] = 1.0
    oi, theta = _influence(vt, X, y, w, 'gaussian', 0.0, 'f64')
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter('always')
        res = oi.approximate_cv('ns', groups=labels)
    msgs = [str(r.message) for r in rec if issubclass(r.category, UserWarning)]
    assert len(msgs) == 1 and 'Groups on this rank: 1' in msgs[0], msgs
    z = res.z_loo.cpu().numpy()
    bad = np.zeros(200, dtype=bool)
    bad[5:10] = True
    assert np.isnan(z[bad]).all() and np.isnan(res.loss.cpu().numpy()[bad]).all() and res.n_invalid == 5
    assert np.isfinite(z[~bad]).all()
    starts = np.arange(0, 201, 5)
    ref = lgo.group_loo(X, y, w, theta, starts, 'gaussian', 0.0)
    assert np.isnan(ref['z_ns'][bad]).all()
    assert_close(z[~bad], ref['z_ns'][~bad], what='other groups')
    ml, nbad = oloo.mean_loss(oloo.glm_loss(ref['z_ns'], y, 'gaussian'), w, np.isnan(ref['z_ns']))
    assert nbad == 5
    assert_close(np.array([res.mean_loss]), np.array([ml]), what='mean_loss')
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter('always')
        z_ij = oi.loo_linear_predictor('ij', groups=labels)
    assert not [r for r in rec if issubclass(r.category, UserWarning)] and bool(torch.isfinite(z_ij).all())


def test_groups_none_is_unchanged(vt):
    X, y, w = _problem('logistic', 300, 5, seed=6)
    oi, _ = _influence(vt, X, y, w, 'logistic', 0.1, 'auto')
    a = oi.approximate_cv('ns')
    b = oi.approximate_cv('ns', groups=None)
    assert torch.equal(a.z_loo, b.z_loo) and torch.equal(a.leverage, b.leverage) and a.mean_loss == b.mean_loss
    assert torch.equal(oi.loo_linear_predictor('ij'), oi.loo_linear_predictor('ij', groups=None))


# --------------------------------------------------------------- bench width ----
def test_bench_width_memory(vt):
    """D = 1024, N = 2e5 ('auto': the INT8 engine), groups of 8: the engines' workspaces do not grow with N (the INT8
    one holds two chunks of digits and one D x chunk block of U); beyond them, approximate_cv allocates O(N) vectors
    and L^{-1}, nothing of size D x N.  Both engines agree."""
    N, D = 200000, 1024
    assert vt.ops.resolve_precision('auto', N, D) == 'f64_ozaki'
    lib = vt._cabi.load()
    assert lib.vt_group_loo_ozaki_workspace_bytes(N, D, 7) == lib.vt_group_loo_ozaki_workspace_bytes(10 ** 7, D, 7)
    assert lib.vt_group_loo_workspace_bytes(N, D) == lib.vt_group_loo_workspace_bytes(10 ** 7, D)
    g = torch.Generator(device='cuda').manual_seed(9)
    X = torch.randn(N, D, device='cuda', dtype=torch.float64, generator=g) / D ** 0.5
    theta = torch.randn(D, device='cuda', dtype=torch.float64, generator=g) * 0.3
    y = (torch.rand(N, device='cuda', dtype=torch.float64, generator=g) < torch.sigmoid(X @ theta)).double()
    w = torch.rand(N, device='cuda', dtype=torch.float64, generator=g) + 0.5
    labels = torch.arange(N, device='cuda') // 8
    results = {}
    for precision in ('auto', 'f64'):
        vt.ops.free_workspaces()
        obj = vt.objectives.GLMObjective(X, y, family='logistic', l2=1.0, precision=precision)
        oi = vt.ObservationInfluence(obj, theta, weights=w)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        res = oi.approximate_cv('ns', groups=labels)
        torch.cuda.synchronize()
        grown = torch.cuda.max_memory_allocated() - base
        ws = sum(b.numel() * 8 for (k, _), b in vt.ops._workspaces.items() if k in ('glo', 'glo_ozaki'))
        assert grown - ws < 8 * D * N / 4, (precision, grown, ws)
        results[precision] = res
    ra, rf = results['auto'], results['f64']
    assert ra.n_invalid == rf.n_invalid == 0
    assert bool(torch.isfinite(ra.z_loo).all())
    assert_close(ra.z_loo, rf.z_loo, what='z_loo engines')
    assert_close(ra.leverage, rf.leverage, what='leverage engines')
    assert abs(ra.mean_loss - rf.mean_loss) <= 1e-8 * abs(rf.mean_loss)
