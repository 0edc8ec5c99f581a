"""GPU tests of the block-arrow path (``csrc/blockchol.cu``, ``block_solver.py``, ``GMMVBObjective``) at the shapes
where its kernels select different code: every template instance of the batched block kernels with M at the top and
bottom of its range, block and row counts past each kernel's grid cap (so the grid-stride loops run), every thread
count of ``tall_colsum``, every softmax width of ``gmm_blocks``, and the Schur complement at the shapes where 'auto'
would choose the INT8 engine.

Each test checks that it reached its branch: the grid caps restate ``grid_for`` from the SM count, the block sizes
are checked against the instance ranges, and the Schur route against ``resolve_precision``.  References: longdouble
factors and substitutions (``oracle/highprec.py``), with every block's error held to 10x that of numpy / LAPACK
float64 on the same block; integer data on which float64 is exact (``torch.equal``); the GMM closed form restated in
longdouble and autodiff of ``models.gmm_vb_objective``; and for solves, a longdouble residual through the block
structure with one step of iterative refinement."""
import re

import numpy as np
import pytest
import scipy.linalg
import torch

from conftest import assert_close
from oracle import highprec, models

pytestmark = pytest.mark.gpu

EPS = float(np.finfo(np.float64).eps)
LD = np.longdouble
POTRF_MT = (8, 16, 24, 32)                 # template instances of block_potrf_kernel
TRSM_MT = (8, 16, 20, 24, 32)              # ... of block_trsm_kernel (both directions)
BLOCK_MS = (1, 8, 9, 16, 17, 20, 21, 24, 25, 32)
FLOOR = 50 * EPS                           # errors below this are rounding of the data itself


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    import vittles_b200.block_solver      # noqa: F401  (the solver's kernel set, for the f64-route subclass)
    return vittles_b200


@pytest.fixture(scope='module')
def caps(vt):
    """Work items one launch covers before its grid-stride loop wraps: grid_for(work, per_cta, k) caps the grid at
    k * SMs CTAs (csrc/blockchol.cu)."""
    sms = vt.ops.device_info()['sm_count']
    return dict(sms=sms, potrf=4 * 4 * sms, trsm=4 * 3 * sms, solve=4 * 6 * sms, gmm=1 * 8 * sms,
                gemv=32 * 8 * sms)


def _colsum_cap(sms, Dg):
    threads = 1024 if Dg >= 1024 else (Dg + 31) // 32 * 32
    return 64 * sms * (2 if threads > 512 else (4 if threads > 256 else 8)), threads


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _spd_blocks(rng, G, M, kmax, scale=True):
    """G blocks Q diag(lam) Q^T with a spectrum from 1 to kappa_g (log-uniform up to kmax), times a random scale."""
    q = np.linalg.qr(rng.normal(size=(G, M, M)))[0]
    kap = 10.0 ** rng.uniform(0, np.log10(kmax), size=(G, 1))
    lam = kap ** np.linspace(0.0, 1.0, M)[None, :]
    if scale:
        lam = lam * 10.0 ** rng.uniform(-2, 2, size=(G, 1))
    B = (q * lam[:, None, :]) @ q.transpose(0, 2, 1)
    return 0.5 * (B + B.transpose(0, 2, 1))


def _block_err(X, ref):
    """max |X_g - ref_g| / max |ref_g| per block g."""
    ref = np.asarray(ref, dtype=LD)
    G = ref.shape[0]
    num = np.abs(np.asarray(X, dtype=LD) - ref).reshape(G, -1).max(1)
    return (num / np.abs(ref).reshape(G, -1).max(1)).astype(np.float64)


def _no_worse(err, err_np, what):
    bar = 10 * np.maximum(err_np, FLOOR)
    g = int(np.argmax(err / bar))
    assert np.all(err <= bar), '{}: block {} error {:.3e}, numpy {:.3e}'.format(what, g, err[g], err_np[g])


# ------------------------------------------------------------------------------------------------------------------
# 1. Batched block kernels at every instance and past the caps
# ------------------------------------------------------------------------------------------------------------------
def test_block_sizes_cover_every_instance_edge():
    for widths in (POTRF_MT, TRSM_MT):
        for lo, hi in zip((0,) + widths[:-1], widths):
            assert lo + 1 in BLOCK_MS and hi in BLOCK_MS, (widths, lo, hi)


def _g_sizes(caps):
    g_mid = 999                                         # below every cap, not a multiple of the 4 blocks per CTA
    g_big = 2 * max(caps['potrf'], caps['trsm'], caps['solve']) + 5
    assert g_mid % 4 and g_mid < min(caps['potrf'], caps['trsm'], caps['solve'])
    assert g_big % 4 and g_big >= 2 * max(caps['potrf'], caps['trsm'], caps['solve'])
    return g_mid, g_big


@pytest.mark.parametrize('M', BLOCK_MS)
def test_block_potrf_and_solve(vt, caps, M):
    """block_potrf and block_solve (both modes) at G = 1, below the cap and past twice the cap.  The factor is held
    to a longdouble factor of the same block; the substitutions to a longdouble substitution with the kernel's own
    factor, so that the factor's error (amplified by kappa_g, up to 1e6 here) does not hide theirs."""
    rng = np.random.default_rng(M)
    for G in (1,) + _g_sizes(caps):
        B = _spd_blocks(rng, G, M, 1e6)
        L = vt.ops.block_potrf(_dev(B))
        Lh = L.cpu().numpy()
        what = 'M {} G {}'.format(M, G)
        assert bool((torch.triu(L, 1) == 0).all()), what
        Lq = Lh.astype(LD)
        bwd = np.abs(Lq @ Lq.transpose(0, 2, 1) - B).reshape(G, -1).max(1) / np.abs(B).reshape(G, -1).max(1)
        assert np.all(bwd <= 4 * (M + 1) * EPS), (what, float(bwd.max()))
        L_ld = highprec.cholesky_ld_batched(B)
        L_np = np.linalg.cholesky(B)
        _no_worse(_block_err(Lh, L_ld), _block_err(L_np, L_ld), 'potrf ' + what)
        b = rng.normal(size=(G, M))
        for tr in (False, True):                        # the substitution on the kernel's own factor
            y = vt.ops.block_solve(L, _dev(b), transpose=tr).cpu().numpy()
            ref = highprec.solve_lower_ld_batched(Lh, b[:, :, None], transpose=tr)[:, :, 0]
            y_np = np.stack([scipy.linalg.solve_triangular(Lh[g], b[g], lower=True, trans=1 if tr else 0)
                             for g in range(G)])
            _no_worse(_block_err(y, ref), _block_err(y_np, ref), 'solve tr={} {}'.format(tr, what))


@pytest.mark.parametrize('M', BLOCK_MS)
def test_block_trsm(vt, caps, M):
    """block_trsm in both directions: Dg in {1, 31, 257} (one column per item, fewer items than threads, several
    items per thread), G = 1, below the cap and past twice the cap; against a longdouble substitution with the same
    factor."""
    g_mid, g_big = _g_sizes(caps)
    assert g_big >= 2 * caps['trsm']
    rng = np.random.default_rng(100 + M)
    for G, Dg in ((1, 257), (g_mid, 31), (g_mid, 257), (g_big, 1), (g_big, 31)):
        B = _spd_blocks(rng, G, M, 1e6)
        L = vt.ops.block_potrf(_dev(B))
        Lh = L.cpu().numpy()
        C = rng.normal(size=(G, M, Dg))
        for tr in (False, True):
            Z = vt.ops.block_trsm(L, _dev(C), transpose=tr).cpu().numpy()
            ref = highprec.solve_lower_ld_batched(Lh, C, transpose=tr)
            Z_np = np.stack([scipy.linalg.solve_triangular(Lh[g], C[g], lower=True, trans=1 if tr else 0)
                             for g in range(G)])
            _no_worse(_block_err(Z, ref), _block_err(Z_np, ref), 'trsm tr={} M {} G {} Dg {}'.format(tr, M, G, Dg))


@pytest.mark.parametrize('M', [1, 17, 32])
def test_block_potrf_reports_a_non_pd_block(vt, caps, M):
    """One indefinite block at the last position, one that only the grid-stride loop reaches, and several at once
    (the first block to fail reports itself, so any of them may be named)."""
    G = 2 * caps['potrf'] + 3
    late = caps['potrf'] + 6                     # past the first sweep of the grid
    assert late >= caps['potrf'] and late < G - 1
    rng = np.random.default_rng(7 + M)
    good = _spd_blocks(rng, G, M, 1e3)
    q = np.linalg.qr(rng.normal(size=(M, M)))[0]
    bad = (q * np.linspace(-1.0, 2.0, M)) @ q.T                # one eigenvalue -1 (for M = 1, the block -1)
    for where in ([G - 1], [late], [5, late, G - 1]):
        B = good.copy()
        B[where] = 0.5 * (bad + bad.T)
        with pytest.raises(np.linalg.LinAlgError) as e:
            vt.ops.block_potrf(_dev(B))
        g = int(re.search(r'block (\d+) of', str(e.value)).group(1))
        assert g in where, (where, g)


GEMV_DGS = [1, 31, 32, 255, 256, 257, 512, 513, 1023, 1024, 1025, 6000]


@pytest.mark.parametrize('Dg', GEMV_DGS)
def test_tall_gemv_and_colsum(vt, caps, Dg):
    """Every thread count of tall_colsum and the 48 KB shared-x limit of tall_gemv, with R past twice both caps.
    Integer data: float64 is exact, so the kernels must equal torch bit for bit."""
    colsum_cap, threads = _colsum_cap(caps['sms'], Dg)
    R = 2 * max(caps['gemv'], colsum_cap) + 37
    assert R > 2 * caps['gemv'] and R > 2 * colsum_cap
    gen = torch.Generator(device='cuda').manual_seed(Dg)
    Z = torch.randint(-128, 129, (R, Dg), generator=gen, device='cuda').double()
    x = torch.randint(-8, 9, (Dg,), generator=gen, device='cuda').double()
    u = torch.randint(-8, 9, (R,), generator=gen, device='cuda').double()
    y0 = 2.0 * torch.randint(-8, 9, (R,), generator=gen, device='cuda').double()
    c0 = 2.0 * torch.randint(-8, 9, (Dg,), generator=gen, device='cuda').double()
    zx, ztu = Z @ x, Z.T @ u
    assert torch.equal(vt.ops.tall_gemv(Z, x), zx)
    assert torch.equal(vt.ops.tall_gemv(Z, x, alpha=-3.0, y=y0.clone(), beta=0.5), 0.5 * y0 - 3.0 * zx)
    y_nan = torch.full((R,), float('nan'), dtype=torch.float64, device='cuda')
    assert torch.equal(vt.ops.tall_gemv(Z, x, alpha=2.0, y=y_nan, beta=0.0), 2.0 * zx)      # beta = 0 ignores y
    assert torch.equal(vt.ops.tall_colsum(Z, u), ztu)
    assert torch.equal(vt.ops.tall_colsum(Z, u, alpha=-2.0, y0=c0, beta=0.5), 0.5 * c0 - 2.0 * ztu)
    assert torch.equal(vt.ops.tall_colsum(Z, u, alpha=3.0, y0=None, beta=7.0), 3.0 * ztu)
    del Z
    Zr = torch.randn(R, Dg, generator=gen, device='cuda', dtype=torch.float64)
    xr = torch.randn(Dg, generator=gen, device='cuda', dtype=torch.float64)
    ur = torch.randn(R, generator=gen, device='cuda', dtype=torch.float64)
    assert_close(vt.ops.tall_gemv(Zr, xr), Zr @ xr, what='gemv Dg {}'.format(Dg))
    s1 = vt.ops.tall_colsum(Zr, ur)
    assert_close(s1, Zr.T @ ur, what='colsum Dg {} ({} threads)'.format(Dg, threads))
    assert torch.equal(vt.ops.tall_colsum(Zr, ur), s1)                 # a fixed-order reduction
    if Dg == GEMV_DGS[-1]:
        with pytest.raises(ValueError):
            vt.ops.tall_gemv(torch.zeros(8, Dg + 1, dtype=torch.float64, device='cuda'),
                             torch.zeros(Dg + 1, dtype=torch.float64, device='cuda'))


# ------------------------------------------------------------------------------------------------------------------
# 2. gmm_blocks at its edges
# ------------------------------------------------------------------------------------------------------------------
def _gmm_data(seed, N, K, d):
    """Overlapping clusters; logits in [-1.5, 1.5] keep every responsibility in [1e-3, 1 - 1e-3]."""
    rng = np.random.default_rng(seed)
    centers = 0.35 * rng.normal(size=(K, d))
    X = centers[rng.integers(K, size=N)] + rng.normal(size=(N, d))
    m = centers + 0.05 * rng.normal(size=(K, d))
    rho = rng.uniform(-1.5, 1.5, size=(N, K - 1))
    lp = 0.3 * rng.normal(size=K)
    return X, m, rho, lp - np.log(np.sum(np.exp(lp)))


def _gmm_closed_form_ld(X, m, rho, log_pi):
    """r, grad_rho, obj_terms, blocks and the cross-block coefficients r_j (delta_jk - r_k) in longdouble."""
    N, K = X.shape[0], m.shape[0]
    M = K - 1
    logits = np.concatenate([rho, np.zeros((N, 1))], axis=1).astype(LD)
    mx = logits.max(1, keepdims=True)
    logr = logits - mx - np.log(np.exp(logits - mx).sum(1, keepdims=True))
    r = np.exp(logr)
    sq = np.zeros((N, K), dtype=LD)
    for k in range(K):
        sq[:, k] = ((X.astype(LD) - m[k].astype(LD)) ** 2).sum(1)
    a = 0.5 * sq - np.asarray(log_pi, dtype=LD)[None] + logr
    abar = (r * a).sum(1)
    dev = a - abar[:, None]
    rj, dj = r[:, :M], dev[:, :M]
    blocks = -(rj[:, :, None] * rj[:, None, :]) * (dj[:, :, None] + dj[:, None, :] + 1)
    idx = np.arange(M)
    blocks[:, idx, idx] += rj * (dj + 1)
    coef = rj[:, :, None] * (np.eye(M, K, dtype=LD)[None] - r[:, None, :])
    return dict(r=r, grad_rho=rj * dj, obj_terms=abar, blocks=blocks, coef=coef)


def _gmm_autodiff(X, m, rho, log_pi, n):
    """r, grad_rho, objective, local block and cross block of observation n from autodiff of the model's term."""
    K, d = m.shape
    f = models.gmm_vb_objective(X[n:n + 1], K, log_pi=log_pi, prior_prec=0.0)
    p = torch.as_tensor(np.concatenate([m.reshape(-1), rho[n]]))
    J = torch.func.jacrev(lambda q: torch.func.grad(f)(q)[K * d:])(p)
    r = torch.softmax(torch.cat([torch.as_tensor(rho[n]), torch.zeros(1, dtype=torch.float64)]), 0)
    return dict(r=r, grad_rho=torch.func.grad(f)(p)[K * d:], obj_terms=f(p), blocks=J[:, K * d:], cross=J[:, :K * d])


GMM_KD = [(K, d) for K in (2, 3, 17, 32) for d in (1, 31, 33, 257)]


@pytest.mark.parametrize('K,d', GMM_KD)
def test_gmm_blocks_past_the_cap(vt, caps, K, d):
    """Every observation against the closed form in longdouble, and a sample including the observations where the
    grid-stride loop wraps against autodiff of models.gmm_vb_objective."""
    grid = caps['gmm']
    N = 2 * grid + 3
    assert N > 2 * grid
    X, m, rho, log_pi = _gmm_data(K * 1000 + d, N, K, d)
    ref = _gmm_closed_form_ld(X, m, rho, log_pi)
    assert ref['r'].min() >= 1e-3 and ref['r'].max() <= 1 - 1e-3
    out = vt.ops.gmm_blocks(_dev(X), _dev(m), _dev(rho), _dev(log_pi))
    for key in ('r', 'grad_rho', 'obj_terms', 'blocks'):
        assert_close(out[key], ref[key].astype(np.float64), what='{} K {} d {}'.format(key, K, d))
    # cross blocks r_j (delta_jk - r_k) (m_k - x_n): the longdouble coefficient times m_k - x_n, on the device
    coef = _dev(ref['coef'].astype(np.float64))
    Xd, md = _dev(X), _dev(m)
    step = max(1, (1 << 24) // ((K - 1) * K * d))
    for n0 in range(0, N, step):
        dm = md[None] - Xd[n0:n0 + step, None, :]
        want = (coef[n0:n0 + step, :, :, None] * dm[:, None]).reshape(-1, K - 1, K * d)
        assert_close(out['cross'][n0:n0 + step], want, what='cross K {} d {} n0 {}'.format(K, d, n0))
    wrap = [k * grid + o for k in (1, 2) for o in (-1, 0, 1)]
    rng = np.random.default_rng(d)
    n_sample = 64 if K * d <= 2048 else 16           # (autodiff takes ~0.5 s an observation at K d = 8224)
    sample = sorted(set([0, N - 1] + wrap + list(rng.choice(N, n_sample - len(wrap) - 2, replace=False))))
    for n in sample:
        ad = _gmm_autodiff(X, m, rho, log_pi, n)
        for key in ('r', 'grad_rho', 'obj_terms', 'blocks', 'cross'):
            assert_close(out[key][n], ad[key].numpy(), what='{} n {} K {} d {}'.format(key, n, K, d))


@pytest.mark.parametrize('K,d', [(2, 1), (32, 33)])
def test_gmm_blocks_flags_do_not_change_the_other_outputs(vt, caps, K, d):
    N = caps['gmm'] + 5
    X, m, rho, log_pi = (_dev(a) for a in _gmm_data(5, N, K, d))
    full = vt.ops.gmm_blocks(X, m, rho, log_pi)
    for wb, wc in ((False, False), (True, False), (False, True)):
        part = vt.ops.gmm_blocks(X, m, rho, log_pi, want_blocks=wb, want_cross=wc)
        for key in ('r', 'grad_rho', 'obj_terms') + (('blocks',) if wb else ()) + (('cross',) if wc else ()):
            assert torch.equal(part[key], full[key]), (key, wb, wc)
        assert (part['blocks'] is None) != wb and (part['cross'] is None) != wc


# ------------------------------------------------------------------------------------------------------------------
# 3. The solver across instances, and where 'auto' would put its Schur complement on the INT8 engine
# ------------------------------------------------------------------------------------------------------------------
def _host(h):
    return (h.sparsity_array.cpu().numpy(), h.global_inds.cpu().numpy(), h.blocks.cpu().numpy(),
            h.cross.cpu().numpy(), h.hgg.cpu().numpy())


def _refined_errors(parts, b, solutions, solve_f64):
    """Forward error of each solution against x + solve_f64(b - H x), x the f64 route's solution, with the residual
    in longdouble; and the normwise backward error of each."""
    sa, gi, blocks, cross, hgg = parts
    x0 = solutions['f64']
    r0 = highprec.block_arrow_residual_ld(sa, gi, blocks, cross, hgg, x0, b)
    ref = x0 + np.asarray(solve_f64(np.asarray(r0, dtype=np.float64)), dtype=np.float64).reshape(x0.shape)
    rows = np.zeros(b.shape[0])
    rows[sa] = np.abs(blocks).sum(2) + np.abs(cross).sum(2)
    rows[gi] = np.abs(cross).sum((0, 1)) + np.abs(hgg).sum(1)
    hinf = rows.max()
    fwd, bwd = {}, {}
    for k, x in solutions.items():
        fwd[k] = float(np.abs(x - ref).max() / np.abs(ref).max())
        r = highprec.block_arrow_residual_ld(sa, gi, blocks, cross, hgg, x, b) if k != 'f64' else r0
        bwd[k] = float(np.abs(r).max() / (hinf * np.abs(x).max() + np.abs(b).max()))
    return fwd, bwd


@pytest.mark.parametrize('M', [8, 21, 32])
def test_block_arrow_solver_past_the_caps(vt, caps, M):
    """Scattered indices, G past twice every block kernel's cap, K = 1, 2, 3 right-hand sides (the vector kernels,
    the matrix-vector forms of Z^T Y and Y -= Z X_g, and the GEMM forms)."""
    from vittles_b200.sparse_hessian_lib import BlockArrowHessian
    Dg = 96
    G = max(2 * caps['solve'] + 5, 2 * max(caps['gemv'], _colsum_cap(caps['sms'], Dg)[0]) // M + 5)
    R = G * M
    assert G >= 2 * max(caps['potrf'], caps['trsm'], caps['solve'])
    assert R > 2 * caps['gemv'] and R > 2 * _colsum_cap(caps['sms'], Dg)[0]
    assert vt.ops.resolve_precision('auto', R, Dg) == 'f64'
    rng = np.random.default_rng(M)
    d = R + Dg
    perm = rng.permutation(d)
    sa, gi = perm[:R].reshape(G, M), perm[R:]
    blocks = _spd_blocks(rng, G, M, 1e2, scale=False)
    cross = 1e-3 * rng.normal(size=(G, M, Dg))          # ||Z^T Z|| < 1 <= lambda_min(Hgg): H is SPD
    q = np.linalg.qr(rng.normal(size=(Dg, Dg)))[0]
    hgg = (q * np.logspace(0, 1, Dg)) @ q.T
    hgg = 0.5 * (hgg + hgg.T)
    h = BlockArrowHessian(d, torch.as_tensor(sa, device='cuda'), torch.as_tensor(gi, device='cuda'),
                          blocks=_dev(blocks), cross=_dev(cross), hgg=_dev(hgg))
    solve = vt.block_solver.BlockArrowSolver(h).solve
    for K in (1, 2, 3):
        b = rng.normal(size=(d, K))
        x = solve(b)
        assert x.shape == (d, K)
        fwd, bwd = _refined_errors((sa, gi, blocks, cross, hgg), b, {'f64': x}, solve)
        assert bwd['f64'] <= 1e-14, (K, bwd)
        assert fwd['f64'] <= 1e-12, (K, fwd)


def _bar_ratio(actual, desired, scale=None, rtol=1e-8, atol_scale=1e-12):
    """max |actual - desired| / (rtol |desired| + atol_scale scale), scale = max|desired| by default: at most 1
    within the parity bar."""
    err = (actual - desired).abs()
    scale = float(desired.abs().max()) if scale is None else scale
    return float((err / (rtol * desired.abs() + atol_scale * scale)).max())


def _schur_case(vt, case):
    """Dg = 512, G M = 381 900 rows: 'auto' would send Z^T Z to the INT8 engine."""
    from vittles_b200.sparse_hessian_lib import BlockArrowHessian
    G, M, Dg = 20100, 19, 512
    assert vt.ops.resolve_precision('auto', G * M, Dg) == 'f64_ozaki'
    rng = np.random.default_rng({'a': 1, 'b': 2, 'c': 3}[case])
    gen = torch.Generator(device='cuda').manual_seed(len(case) + ord(case))
    d = G * M + Dg
    perm = rng.permutation(d)
    sa, gi = perm[:G * M].reshape(G, M), perm[G * M:]
    blocks = _spd_blocks(rng, G, M, 10.0, scale=False)
    if case == 'a':
        cross = 1e-2 * torch.randn(G, M, Dg, generator=gen, device='cuda', dtype=torch.float64)
    else:       # heavy-tailed columns: a few blocks of O(1) entries, the rest 1e-4 .. 1e-3
        mag = 10.0 ** (-3.0 - torch.rand(G, M, Dg, generator=gen, device='cuda', dtype=torch.float64))
        sign = torch.randint(0, 2, (G, M, Dg), generator=gen, device='cuda').double() * 2 - 1
        cross = mag * sign
        heavy = torch.randperm(G, generator=gen, device='cuda')[:24]
        cross[heavy] = torch.randn(24, M, Dg, generator=gen, device='cuda', dtype=torch.float64)
    Lb = vt.ops.block_potrf(_dev(blocks))
    Z2 = vt.ops.block_trsm(Lb, cross.clone()).reshape(G * M, Dg)
    grams = dict(int8=vt.ops.syrk_weighted(Z2, precision='f64_ozaki'), f64=vt.ops.syrk_weighted(Z2, precision='f64'))
    assert torch.equal(vt.block_solver.CudaBlockKernels.gram(Z2), grams['f64'])       # the route the solver takes
    gram_ref = Z2.T @ Z2                                   # torch float64 (cuBLAS)
    q = torch.linalg.qr(torch.randn(Dg, Dg, generator=gen, device='cuda', dtype=torch.float64))[0]
    A = (q * torch.logspace(-2, 0, Dg, device='cuda', dtype=torch.float64)) @ q.T
    A = 0.5 * (A + A.T)
    if case == 'c':        # S = A: the Schur complement is a large cancellation
        hgg = grams['f64'] + A
        assert float(gram_ref.diagonal().min() / A.diagonal().max()) > 100
    else:
        hgg = A + grams['f64'].abs().sum(1).max() * torch.eye(Dg, dtype=torch.float64, device='cuda')
    # In (c) S is 1e3 times smaller than the terms it is the difference of, and cuBLAS's own rounding of Z^T Z is
    # about the parity floor of S: there S is also held to the floor of the terms (1e-12 max|Hgg|).
    bars = {k: _bar_ratio(hgg - g, hgg - gram_ref) for k, g in grams.items()}
    bars.update({k + ' (terms)': _bar_ratio(hgg - g, hgg - gram_ref, float(hgg.abs().max())) for k, g in grams.items()})
    del Z2, Lb
    h = BlockArrowHessian(d, torch.as_tensor(sa, device='cuda'), torch.as_tensor(gi, device='cuda'),
                          blocks=_dev(blocks), cross=cross, hgg=hgg)
    return h, bars


def _compare_routes(vt, int8_kernels, h, b, what):
    """Forward and backward errors of the solver (Z^T Z on the f64 engine) and of the same solver with Z^T Z on the
    INT8 engine, against the refined solution; None for a route whose Schur complement is not positive definite."""
    solver = vt.block_solver.BlockArrowSolver(h)
    x = {'f64': solver.solve(b).reshape(-1, 1)}
    try:
        x['int8'] = vt.block_solver.BlockArrowSolver(h, kernels=int8_kernels).solve(b).reshape(-1, 1)
    except np.linalg.LinAlgError as e:
        x['int8'] = None
        print('\n{}: INT8 route: {}'.format(what, e))
    fwd, bwd = _refined_errors(_host(h), np.asarray(b).reshape(-1, 1), {k: v for k, v in x.items() if v is not None},
                               solver.solve)
    print('\n{}: forward error {}; backward error {}'.format(what, fwd, bwd))
    return fwd, bwd


@pytest.fixture(scope='module')
def int8_kernels(vt):
    class Int8Kernels(vt.block_solver.CudaBlockKernels):
        """The solver's kernels with Z^T Z on the INT8 error-free-slicing engine."""
        @staticmethod
        def gram(Z2):
            return vt.ops.syrk_weighted(Z2, precision='f64_ozaki')
    return Int8Kernels


@pytest.mark.parametrize('case', ['a', 'b', 'c'])
def test_schur_complement_where_auto_would_pick_the_int8_engine(vt, int8_kernels, case):
    """(a) Gaussian cross blocks, (b) heavy-tailed columns of Z, (c) (b) with Hgg = Z^T Z (f64 engine) + A, so that
    S = Hgg - Z^T Z is a large cancellation.  The solver's Schur complement must meet the parity bar against cuBLAS
    and its solution a backward error of a few eps.  The INT8 engine is measured beside it: it meets the bar in (a)
    and (b); in (c) its S is about 3x further from cuBLAS than the DMMA engine's and misses the bar of S, which is
    why the solver does not use it."""
    h, bars = _schur_case(vt, case)
    print('\nSchur case {}: worst error / parity bar of S: {}'.format(case, bars))
    assert bars['f64'] <= 1 if case != 'c' else bars['f64 (terms)'] <= 1, bars
    b = np.random.default_rng(9).normal(size=h.shape[0])
    fwd, bwd = _compare_routes(vt, int8_kernels, h, b, 'Schur case ' + case)
    assert bwd['f64'] <= 1e-14, bwd
    if case != 'c':
        assert bars['int8'] <= 1 and fwd['int8'] <= 10 * max(fwd['f64'], FLOOR), (bars, fwd)


# ------------------------------------------------------------------------------------------------------------------
# 4. Argument checks: the block kernels take no leading dimension, so what they cannot address is refused
# ------------------------------------------------------------------------------------------------------------------
def test_block_wrappers_refuse_operands_the_kernels_cannot_address(vt):
    rng = np.random.default_rng(4)
    G, M, R, Dg, N, K, d = 6, 5, 30, 7, 9, 4, 3
    Zbig = _dev(rng.normal(size=(R, Dg + 3)))
    Z, x, u, y = Zbig[:, :Dg].contiguous(), _dev(rng.normal(size=Dg)), _dev(rng.normal(size=R)), _dev(np.zeros(R))
    for bad in (Zbig[:, :Dg], Zbig[:, 1:Dg + 1], Zbig[:, :1]):
        with pytest.raises(ValueError):
            vt.ops.tall_gemv(bad, x[:bad.shape[1]].contiguous())
        with pytest.raises(ValueError):
            vt.ops.tall_colsum(bad, u)
    for call in (lambda: vt.ops.tall_gemv(Z, x[:-1]),
                 lambda: vt.ops.tall_gemv(Z, x, y=y[:-1], beta=1.0),
                 lambda: vt.ops.tall_gemv(Z, x, y=_dev(np.zeros(2 * R))[::2], beta=1.0),
                 lambda: vt.ops.tall_colsum(Z, u[:-1]),
                 lambda: vt.ops.tall_colsum(Z, u, y0=x[:-1])):
        with pytest.raises(ValueError):
            call()
    Lb = vt.ops.block_potrf(_dev(_spd_blocks(rng, G, M, 10.0)))
    C, b = _dev(rng.normal(size=(G, M, Dg))), _dev(rng.normal(size=(G, M)))
    bbig = _dev(rng.normal(size=(G, M + 2)))
    for call in (lambda: vt.ops.block_solve(Lb, bbig[:, :M]),
                 lambda: vt.ops.block_solve(Lb, _dev(rng.normal(size=(M, G))).T),
                 lambda: vt.ops.block_solve(Lb[:, :M - 1, :M - 1].contiguous(), b),
                 lambda: vt.ops.block_solve(Lb[:-1], b),
                 lambda: vt.ops.block_trsm(Lb[:-1], C),
                 lambda: vt.ops.block_trsm(Lb[:, :M - 1, :M - 1].contiguous(), C),
                 lambda: vt.ops.block_trsm(Lb, _dev(rng.normal(size=(G, M, Dg + 1)))[:, :, :Dg])):
        with pytest.raises(ValueError):
            call()
    Xbig = _dev(rng.normal(size=(N, d + 2)))
    X, m = Xbig[:, :d].contiguous(), _dev(rng.normal(size=(K, d)))
    rho, lp = _dev(rng.normal(size=(N, K - 1))), _dev(np.full(K, -np.log(K)))
    for call in (lambda: vt.ops.gmm_blocks(Xbig[:, :d], m, rho, lp),
                 lambda: vt.ops.gmm_blocks(Xbig[:, 1:d + 1], m, rho, lp),
                 lambda: vt.ops.gmm_blocks(X, m, _dev(rng.normal(size=(N, K))), lp),
                 lambda: vt.ops.gmm_blocks(X, m, rho[:-1], lp),
                 lambda: vt.ops.gmm_blocks(X, m, rho, lp[:-1]),
                 lambda: vt.ops.gmm_blocks(X, m[:, :-1], rho, lp)):
        with pytest.raises(ValueError):
            call()


def test_block_wrappers_pass_packed_operands_through_unchanged(vt):
    """For packed operands the wrappers hand the kernels exactly what they did before the checks: the same bits as
    calling the C ABI directly."""
    from vittles_b200._cabi import load, ptr, stream
    lib = load()
    rng = np.random.default_rng(5)
    G, M, R, Dg = 9, 7, 5000, 33
    Z, x, u = _dev(rng.normal(size=(R, Dg))), _dev(rng.normal(size=Dg)), _dev(rng.normal(size=R))
    y = _dev(rng.normal(size=R))
    out = vt.ops.tall_gemv(Z, x, alpha=-1.5, y=y.clone(), beta=0.25)
    raw = y.clone()
    assert lib.vt_tall_gemv(ptr(Z), R, Dg, ptr(x), -1.5, ptr(raw), 0.25, stream()) == 0
    assert torch.equal(out, raw)
    s = vt.ops.tall_colsum(Z, u, alpha=2.0, y0=x, beta=-1.0)
    ws = torch.empty(lib.vt_tall_colsum_workspace_bytes(Dg) // 8, dtype=torch.float64, device='cuda')
    raw = torch.empty(Dg, dtype=torch.float64, device='cuda')
    assert lib.vt_tall_colsum(ptr(Z), R, Dg, ptr(u), 2.0, ptr(x), -1.0, ptr(raw), ptr(ws), ws.numel() * 8,
                              stream()) == 0
    assert torch.equal(s, raw)
    Lb = vt.ops.block_potrf(_dev(_spd_blocks(rng, G, M, 10.0)))
    C, b = _dev(rng.normal(size=(G, M, Dg))), _dev(rng.normal(size=(G, M)))
    for tr in (0, 1):
        raw = C.clone()
        fn = lib.vt_block_trsmt_batched if tr else lib.vt_block_trsm_batched
        assert fn(ptr(Lb), ptr(raw), G, M, Dg, stream()) == 0
        assert torch.equal(vt.ops.block_trsm(Lb, C.clone(), transpose=bool(tr)), raw)
        raw = b.clone()
        assert lib.vt_block_solve_batched(ptr(Lb), ptr(raw), G, M, tr, stream()) == 0
        assert torch.equal(vt.ops.block_solve(Lb, b.clone(), transpose=bool(tr)), raw)
    N, K, d = 300, 5, 4
    X, m, rho, lp = (_dev(a) for a in _gmm_data(6, N, K, d))
    got = vt.ops.gmm_blocks(X, m, rho, lp)
    raw = dict(blocks=torch.empty(N, K - 1, K - 1), cross=torch.empty(N, K - 1, K * d), r=torch.empty(N, K),
               grad_rho=torch.empty(N, K - 1), obj_terms=torch.empty(N))
    raw = {k: v.double().cuda() for k, v in raw.items()}
    assert lib.vt_gmm_blocks(ptr(X), N, d, K, ptr(m), ptr(rho), ptr(lp), ptr(raw['blocks']), ptr(raw['cross']),
                             ptr(raw['r']), ptr(raw['grad_rho']), ptr(raw['obj_terms']), stream()) == 0
    for k in raw:
        assert torch.equal(got[k], raw[k]), k
