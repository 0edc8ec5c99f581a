"""GPU tests of the INT8 error-free-slicing engine (``csrc/ogemm.cu``): FP64-grade
results from tcgen05.mma.kind::i8.  Unlike the TF32 path this engine IS held to
the parity bar of the FP64 path (rtol 1e-8 with the 1e-12 max|ref| floor of
``conftest.assert_close``): the slicing is exact, every digit product is exact in
INT32, and only digit pairs below 2^-54 of the row scales are dropped."""
import numpy as np
import pytest
import torch

from conftest import assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


def _rnd(*shape, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return torch.randn(*shape, device='cuda', dtype=torch.float64, generator=g)


@pytest.mark.parametrize('S', [5, 6, 7])
def test_slicing_is_exact_to_8S_bits(vt, S):
    X = _rnd(300, 102) * torch.exp(3 * _rnd(300, 1, seed=1))        # rows of very different magnitude
    X[7] = 0.0                                                      # an all-zero row
    d, sc = vt.ops.ozaki_slice(X, S)
    assert d.dtype == torch.int8 and d.shape == (S, 300, 112)
    assert int(d[0].abs().max()) <= 65 and bool((d[:, :, 102:] == 0).all())
    assert bool((torch.frexp(sc)[0] == 0.5).all())                  # powers of two
    rowmax = X.abs().max(dim=1).values
    assert bool((sc > rowmax).all())
    rec = torch.zeros_like(X)
    for s in range(S - 1, -1, -1):
        rec += d[s, :, :102].double() * 2.0 ** (-8 * s - 6)
    resid = (X - rec * sc[:, None]).abs().max(dim=1).values
    assert bool((resid <= sc * 2.0 ** (-(8 * S - 1)) * (1 + 2.0 ** -40)).all())   # round to nearest: half a unit
    fold = _rnd(300, seed=2)
    _, sc2 = vt.ops.ozaki_slice(X, S, fold=fold)
    assert torch.equal(sc2, sc * fold)


@pytest.mark.parametrize('S', [5, 6, 7])
def test_digits_and_products_match_the_cpu_model_exactly(vt, S):
    """Integer work: bit-exact against the oracle's model of the engine (oracle/slicing.py) - the digits, the scales
    and the product (same INT32 accumulators, same FP64 Horner recombination, power-of-two scales)."""
    from oracle import slicing
    A = _rnd(150, 333, seed=20) * torch.exp(2 * _rnd(150, 1, seed=21))
    B = _rnd(70, 333, seed=22)
    d, sc = vt.ops.ozaki_slice(A, S)
    d_ref, sc_ref = slicing.slice_rows(A.cpu().numpy(), S)
    assert np.array_equal(d[:, :, :333].cpu().numpy(), d_ref)
    assert np.array_equal(sc.cpu().numpy(), sc_ref)
    out = vt.ops.ozaki_gemm(A, B, nslices=S).cpu().numpy()
    model = slicing.sliced_gemm(A.cpu().numpy(), B.cpu().numpy(), S)
    assert np.array_equal(out, model)


def _awkward_matrix(rows, cols, S, seed):
    """Values that exercise the rounding of the slicers: exact ties at the last digit, subnormals, zeros, the row
    maximum itself (a power of two: the largest fixed-point value), all of mixed sign."""
    X = _rnd(rows, cols, seed=seed) * torch.exp(4 * _rnd(rows, 1, seed=seed + 1))
    ulp = 2.0 ** -(8 * S - 2)                     # one unit of the last digit relative to the row scale
    X[0, :] = 0.0
    X[1, 0] = 1.0 - 2.0 ** -53                    # just below the scale 1: the largest q
    X[1, 1:9] = torch.tensor([0.5, 1.5, 2.5, 3.5, -0.5, -1.5, -2.5, 127.5], device='cuda', dtype=torch.float64) * ulp
    X[1, 9:] = X[1, 9:].clamp(-0.9, 0.9)
    X[2, :] = 5e-324 * torch.arange(cols, device='cuda', dtype=torch.float64)       # subnormal row
    X[3, 0], X[3, 1], X[3, 2] = 1e300, 1e-300, -4.9e-324                            # 600 orders of magnitude apart
    X[4, :] = -2.0 ** -3                          # every entry the negative of a power of two
    return X


@pytest.mark.parametrize('cols', [100, 256, 333, 1024])
@pytest.mark.parametrize('S', [5, 6, 7])
def test_row_slicer_matches_the_cpu_model_at_every_width(vt, S, cols):
    """The row slicer forms digits with integer instructions only, as the converter warps of the GEMM kernel do: digit
    for digit against the oracle's model at widths that reach every register-resident instance (RC = 1, 2, 4 and 8,
    the last at the 1024-element boundary)."""
    from oracle import slicing
    X = _awkward_matrix(200, cols, S, seed=40)
    d, sc = vt.ops.ozaki_slice(X, S)
    d_ref, sc_ref = slicing.slice_rows(X.cpu().numpy(), S)
    assert np.array_equal(d[:, :, :cols].cpu().numpy(), d_ref)
    assert np.array_equal(sc.cpu().numpy(), sc_ref)
    assert bool((d[:, :, cols:] == 0).all())


@pytest.mark.parametrize('S', [5, 7])
@pytest.mark.parametrize('shape', [(1000, 70), (257, 33), (16, 520)])
def test_transposed_slicer_matches_the_cpu_model(vt, S, shape):
    """Digits of sqrt(s_n) x_ni written observation-contiguous with one scale per feature, digit for digit against
    the oracle's row slicer applied to the transposed weighted matrix."""
    from oracle import slicing
    N, D = shape
    X = _rnd(N, D, seed=50) * torch.exp(2 * _rnd(1, D, seed=51))
    X[3, :] = 0.0
    X[:, 2] = 0.0                                                       # a feature that is zero everywhere
    sq = torch.rand(N, device='cuda', dtype=torch.float64, generator=torch.Generator(device='cuda').manual_seed(52)).sqrt()
    d, sc = vt.ops.ozaki_slice_t(X, sq, S)
    W = (X * sq[:, None]).T.contiguous().cpu().numpy()                  # the same FP64 products
    d_ref, sc_ref = slicing.slice_rows(W, S)
    assert np.array_equal(d[:, :, :N].cpu().numpy(), d_ref)
    assert np.array_equal(sc.cpu().numpy(), sc_ref)
    assert bool((d[:, :, N:] == 0).all())
    # unweighted (the Schur complement Z^T Z of the block-arrow solver): no multiplication at all
    d, sc = vt.ops.ozaki_slice_t(X, None, S)
    d_ref, sc_ref = slicing.slice_rows(X.T.contiguous().cpu().numpy(), S)
    assert np.array_equal(d[:, :, :N].cpu().numpy(), d_ref) and np.array_equal(sc.cpu().numpy(), sc_ref)


def test_extreme_digits_do_not_overflow_int32(vt):
    """All digits -128 over the longest K one accumulation may see (16384): the INT32 accumulators hold
    7 K 2^14 < 2^31 (checked through the raw digit GEMM entry point against the integer model)."""
    from oracle import slicing
    from vittles_b200._cabi import check, ptr, require_cuda, stream
    lib = require_cuda()
    S, M, N, K = 7, 128, 64, 16384
    dA = torch.full((S, M, K), -128, dtype=torch.int8, device='cuda')
    dB = torch.full((S, N, K), -128, dtype=torch.int8, device='cuda')
    one_m = torch.ones(M, dtype=torch.float64, device='cuda')
    one_n = torch.ones(N, dtype=torch.float64, device='cuda')
    out = torch.empty((M, N), dtype=torch.float64, device='cuda')
    check(lib.vt_ozaki_gemm(M, N, K, ptr(dA), K, M * K, ptr(dB), K, N * K, S, 1.0, ptr(one_m), ptr(one_n), ptr(out), N,
                            stream()))
    model = slicing.digits_gemm(dA[:, :2].cpu().numpy(), np.ones(2), dB[:, :2].cpu().numpy(), np.ones(2))
    assert bool((out == float(model[0, 0])).all())


@pytest.mark.parametrize('shape', [(128, 64, 128), (1024, 1024, 1024), (200, 300, 100), (130, 515, 1000), (1, 1, 1),
                                   (257, 65, 36)])
def test_ozaki_gemm_is_fp64_grade(vt, shape):
    M, N, K = shape
    A, B = _rnd(M, K, seed=3), _rnd(N, K, seed=4)
    out = vt.ops.ozaki_gemm(A, B, alpha=-2.0, nslices=6)
    assert_close(out, -2.0 * (A @ B.T), rtol=1e-8, atol_scale=1e-12, what='ozaki_gemm {}'.format(shape))
    out7 = vt.ops.ozaki_gemm(A, B, alpha=-2.0, nslices=7)
    assert float((out7 + 2.0 * (A @ B.T)).abs().max() / (A @ B.T).abs().max()) < 1e-13


def test_ozaki_gemm_badly_scaled_rows(vt):
    """Row scales spanning 12 orders of magnitude: the per-row power-of-two scaling keeps every row at 54 bits."""
    A = _rnd(256, 512, seed=5) * torch.exp(6 * _rnd(256, 1, seed=6))
    B = _rnd(192, 512, seed=7) * torch.exp(6 * _rnd(192, 1, seed=8))
    out = vt.ops.ozaki_gemm(A, B, nslices=7)
    ref = A @ B.T
    rowcol = A.abs().max(dim=1).values[:, None] * B.abs().max(dim=1).values[None, :]
    assert float(((out - ref).abs() / rowcol).max()) < 1e-12


def test_six_slices_stay_inside_the_parity_bar(vt, monkeypatch):
    """The engine's default is 7 balanced digits (54 bits); 6 digits (46 bits, 21 instead of 28 products) still meet
    rtol 1e-8 on well-scaled data but sit close to the 1e-12 max|ref| floor, which is why they are not the default."""
    monkeypatch.setattr(vt.ops, 'OZAKI_SLICES', 6)
    N, D = 20000, 512
    X = vt.ops.synth_design(21, 0, N, D, 'cuda')
    Hm = _rnd(D, D, seed=13)
    Hinv = torch.linalg.inv(Hm @ Hm.T / D + 0.05 * torch.eye(D, device='cuda', dtype=torch.float64)).contiguous()
    resid = _rnd(N, seed=14)
    S64 = vt.ops.ij_apply(Hinv, X, resid)
    S6 = vt.ops.ij_apply(Hinv, X, resid, precision='f64_ozaki')
    assert float((S6 - S64).abs().max() / S64.abs().max()) < 5e-12
    s = torch.rand(N, device='cuda', dtype=torch.float64)
    H64 = vt.ops.syrk_weighted(X, s)
    H6 = vt.ops.syrk_weighted(X, s, precision='f64_ozaki')
    assert float((H6 - H64).abs().max() / H64.abs().max()) < 5e-12


def test_ij_apply_on_the_int8_engine(vt):
    N, D = 40000, 1024
    X = vt.ops.synth_design(11, 0, N, D, 'cuda')
    Hm = _rnd(D, D, seed=9)
    Hinv = torch.linalg.inv(Hm @ Hm.T / D + 0.05 * torch.eye(D, device='cuda', dtype=torch.float64)).contiguous()
    resid = _rnd(N, seed=10)
    S64 = vt.ops.ij_apply(Hinv, X, resid)
    S = vt.ops.ij_apply(Hinv, X, resid, precision='f64_ozaki')
    assert_close(S, S64, rtol=1e-8, atol_scale=1e-12, what='ij_apply f64_ozaki')
    # ragged sizes
    N2, D2 = 3001, 77
    X2 = vt.ops.synth_design(12, 0, N2, D2, 'cuda')
    Hinv2 = torch.eye(D2, device='cuda', dtype=torch.float64) + 0.1 * _rnd(D2, D2, seed=11)
    r2 = _rnd(N2, seed=12)
    assert_close(vt.ops.ij_apply(Hinv2, X2, r2, precision='f64_ozaki'), vt.ops.ij_apply(Hinv2, X2, r2), rtol=1e-8,
                 atol_scale=1e-12)


@pytest.mark.parametrize('shape', [(50000, 1024), (777, 200), (3001, 77), (40000, 10), (1, 5)])
def test_hessian_assembly_on_the_int8_engine(vt, shape):
    """H = X^T diag(s) X: transposed slicing with per-feature, per-chunk scales; chunks of more than
    16384 observations per split-K part exercise the FP64 accumulation across INT32 segments."""
    N, D = shape
    X = vt.ops.synth_design(13, 0, N, D, 'cuda')
    s = torch.rand(N, device='cuda', dtype=torch.float64) * 0.25
    s[::17] = 0.0
    H64 = vt.ops.syrk_weighted(X, s, l2=0.5)
    H = vt.ops.syrk_weighted(X, s, l2=0.5, precision='f64_ozaki')
    assert torch.equal(H, H.T)
    assert_close(H, H64, rtol=1e-8, atol_scale=1e-12, what='syrk f64_ozaki {}'.format(shape))
    assert_close(vt.ops.syrk_weighted(X, precision='f64_ozaki'), vt.ops.syrk_weighted(X), rtol=1e-8, atol_scale=1e-12)
    with pytest.raises(ValueError):
        vt.ops.syrk_weighted(X, -s - 1.0, precision='f64_ozaki')


@pytest.mark.parametrize('shape', [(50000, 1024), (3001, 77), (40000, 2048)])
def test_statistics_pass_hands_the_hessian_its_column_scales(vt, shape):
    """vt_glm_stats_colmax: sqrt(s) and the binades of the per-feature maxima of sqrt(s_n) |x_ni| from the
    statistics pass equal what the INT8 Hessian assembly computes in its own sweep, so the scales, the digits and the
    Hessian are bit-identical; a NaN in X poisons exactly what it poisons there."""
    N, D = shape
    X = vt.ops.synth_design(23, 0, N, D, 'cuda')
    theta = 0.3 * vt.ops.synth_theta(23, D, 'cuda')
    y = (torch.rand(N, device='cuda', dtype=torch.float64) < 0.5).double()
    w = torch.rand(N, device='cuda', dtype=torch.float64) + 0.5
    z, resid, s, grad = vt.ops.glm_stats(X, theta, y, w)
    z2, resid2, s2, grad2, (sq, cmax) = vt.ops.glm_stats(X, theta, y, w, want_colmax=True)
    assert torch.equal(z, z2) and torch.equal(resid, resid2) and torch.equal(s, s2) and torch.equal(grad, grad2)
    assert torch.equal(sq, torch.sqrt(s))
    ref = (X.abs() * torch.sqrt(s)[:, None]).max(dim=0).values
    # the maxima are kept to their high words (sign, exponent, 20 bits): the same binade, hence the same scales
    assert torch.equal(cmax >> 32, ref.view(torch.int64) >> 32) and bool(((cmax & 0xFFFFFFFF) == 0).all())
    H_own = vt.ops.syrk_weighted(X, s, precision='f64_ozaki')
    H_fused = vt.ops.syrk_weighted(X, s, precision='f64_ozaki', colmax=(sq, cmax))
    assert torch.equal(H_own, H_fused)
    X[5, 3] = float('nan')
    _, _, s3, _, (sq3, cmax3) = vt.ops.glm_stats(X, theta, y, w, want_colmax=True)
    bad = torch.isnan(cmax3.view(torch.float64))
    # row 5's z is NaN, so its s and sqrt(s) are NaN: every column with a non-zero entry in that row is poisoned -
    # as in the engine's own sweep
    H3 = vt.ops.syrk_weighted(X, s3, precision='f64_ozaki', colmax=(sq3, cmax3))
    H3_own = vt.ops.syrk_weighted(X, s3, precision='f64_ozaki')
    assert bool(bad.any()) and torch.equal(torch.isnan(H3), torch.isnan(H3_own))


def test_ij_sensitivities_through_the_api_match_the_oracle(vt):
    """precision='f64_ozaki' through HyperparameterSensitivityLinearApproximation: the
    same rtol 1e-8 bar against the oracle as the default FP64 path."""
    from oracle import models, sensitivity as osens
    n, d = 4000, 64
    X, y, _ = models.synth_logistic(31, n, d)
    w = np.ones(n)
    theta = models.glm_newton(X, y, w)
    ref = osens.linear_sensitivity(models.glm_objective(X, y), theta, w)
    obj = vt.objectives.GLMObjective(X, y, family='logistic', precision='f64_ozaki')
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    assert_close(sens.get_dopt_dhyper(), ref['sens'], rtol=1e-8, atol_scale=1e-12, what='dopt_dhyper (f64_ozaki)')
    assert_close(sens.get_hessian_at_opt(), ref['hessian'], rtol=1e-9)


def test_non_finite_inputs_propagate_like_fp64(vt):
    """An Inf / NaN in an operand row poisons exactly the results FP64 arithmetic would poison (the digits of a
    non-finite value are meaningless, so its row gets a NaN scale)."""
    N, D = 3000, 96
    X = vt.ops.synth_design(17, 0, N, D, 'cuda')
    Hinv = torch.eye(D, device='cuda', dtype=torch.float64) + 0.05 * _rnd(D, D, seed=30)
    resid = _rnd(N, seed=31)
    X[5, 7] = float('nan')
    X[11, 3] = float('inf')
    S = vt.ops.ij_apply(Hinv, X, resid, precision='f64_ozaki')
    bad = torch.isnan(S).any(dim=0)
    assert bool(bad[5]) and bool(bad[11]) and int(bad.sum()) == 2
    assert bool(torch.isnan(S[:, 5]).all()) and bool(torch.isnan(S[:, 11]).all())
    ok = ~bad
    assert_close(S[:, ok], vt.ops.ij_apply(Hinv, X, resid)[:, ok], rtol=1e-8, atol_scale=1e-12)
    H = vt.ops.syrk_weighted(X, torch.ones(N, device='cuda', dtype=torch.float64), precision='f64_ozaki')
    nan_rows = torch.isnan(H).all(dim=1)
    assert sorted(torch.nonzero(nan_rows).flatten().tolist()) == [3, 7]
    keep = [i for i in range(D) if i not in (3, 7)]
    Xc = X[:, keep].contiguous()
    assert_close(H[keep][:, keep], vt.ops.syrk_weighted(Xc), rtol=1e-8, atol_scale=1e-12)


def test_bad_arguments(vt):
    A = _rnd(8, 20000)
    with pytest.raises(ValueError):
        vt.ops.ozaki_gemm(A, A)                       # K beyond the INT32 accumulation bound
    with pytest.raises(ValueError):
        vt.ops.ozaki_gemm(_rnd(8, 16), _rnd(8, 32))
    with pytest.raises(ValueError):
        vt.ops.ozaki_gemm(_rnd(8, 16), _rnd(8, 16), nslices=8)
