"""GPU tests of the FP64-grade kernels at the shapes where their drivers switch code paths: rows of more than 1024
elements (separate slicing launches), three or more chunks with a ragged last one, the wide instances of the fused
passes over X (D > 2048), every regime of the dense triangular solve, non-PD pivots in late blocks, and padded or
offset views (every way rows are staged).

Each test checks that it reached its branch: the chunk counts of the INT8 engine through launch-count deltas, the
solve regime from the SM count, the engine 'auto' picks through ``resolve_precision``.  Three kinds of reference:
integer designs on which every engine must be exact (``oracle/exact.py``: ``torch.equal``), random data at the
parity bar against torch float64 on the device (cuBLAS / cuSOLVER, no code shared with this project) and against
the other engine, and the INT8 engine's arithmetic model (``oracle/slicing.py``) bit for bit."""
import math
import re

import numpy as np
import pytest
import scipy.linalg
import torch

from conftest import assert_close
from oracle import exact, slicing

pytestmark = pytest.mark.gpu

S7 = 7                                   # the engine's default number of digits (ops.OZAKI_SLICES)
OBM, OBN, OBK, MAXK = 128, 64, 128, 16384  # INT8 GEMM tile (M, N, K) and the INT32 accumulation bound (ogemm.cuh)
APPLY_CHUNK_BYTES = 288 << 20            # digits of one apply chunk
SYRK_CHUNK_BYTES = 320 << 20             # digits of one Hessian chunk
SENTINEL = 0x7FF8DEADBEEF0001            # a NaN with a payload no kernel writes


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    assert vittles_b200.ops.OZAKI_SLICES == S7
    return vittles_b200


@pytest.fixture(scope='module')
def sms(vt):
    return vt.ops.device_info()['sm_count']


def _rnd(*shape, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return torch.randn(*shape, device='cuda', dtype=torch.float64, generator=g)


def _uni(*shape, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return torch.rand(*shape, device='cuda', dtype=torch.float64, generator=g)


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _parity(actual, desired, rtol=1e-8, atol_scale=1e-12, what=''):
    """conftest.assert_close's bar (rtol with a floor of atol_scale * max|desired|), evaluated on the device."""
    assert actual.shape == desired.shape, what
    assert bool(torch.isfinite(actual).all()), '{}: non-finite entries'.format(what)
    scale = float(desired.abs().max())
    err = (actual - desired).abs()
    bad = err > atol_scale * scale + rtol * desired.abs()
    nbad = int(bad.sum())
    assert nbad == 0, '{}: {} entries outside the bar, worst |err| {:.3e} (max|ref| {:.3e})'.format(
        what, nbad, float(err.max()), scale)


def _pow2_above(m):
    """The slicers' scale: the power of two 2^e with m = f 2^e, f in [0.5, 1) (1 for m = 0)."""
    e = torch.frexp(m)[1]
    return torch.where(m > 0, torch.ldexp(torch.ones_like(m), e), torch.ones_like(m))


def _launches(vt, fn):
    n0 = vt.ops.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, vt.ops.launch_count() - n0


# --------------------------------------------------------- plans of the drivers ----
def apply_chunk_rows(N, D, G):
    """ozaki_chunk_rows (ogemm.cu): rows of X per apply chunk on G SMs."""
    ld = (D + 15) // 16 * 16
    nb = max(1, APPLY_CHUNK_BYTES // (ld * S7) // OBN)
    tiles_m = (D + OBM - 1) // OBM
    best, best_eff = nb, 0.0
    b = nb
    while b >= 1 and b > nb // 2:
        T = b * tiles_m
        eff = T / (G * ((T + G - 1) // G))
        if eff > best_eff + 1e-9:
            best, best_eff = b, eff
        b -= 1
    return min(best * OBN, N)


def apply_chunk_max(D):
    """The largest apply chunk at any SM count."""
    ld = (D + 15) // 16 * 16
    return max(1, APPLY_CHUNK_BYTES // (ld * S7) // OBN) * OBN


def syrk_chunk_rows(N, D, G):
    """syrk_plan (ogemm.cu): observations per Hessian chunk on G SMs."""
    tiles_m, tiles_n = (D + OBM - 1) // OBM, (D + OBN - 1) // OBN
    ntiles = sum(min((tm * OBM + OBM - 1) // OBN + 1, tiles_n) for tm in range(tiles_m))
    parts = max(1, min(16, G // ntiles))
    chunk = parts * MAXK
    by_mem = SYRK_CHUNK_BYTES // (S7 * D) // (parts * OBK) * (parts * OBK)
    if parts * OBK <= by_mem < chunk:
        chunk = by_mem
    return min(chunk, N)


def solve_scratch_cols(D):
    """Columns of one pass of the 512-row out-of-place solve (chol.cu)."""
    return max(512, (D // 2 + 63) // 64 * 64)


def solve_regime(D, K, G):
    """The branch chol_potrs takes: 'chain' (K <= 8), 'oop512' or 'inplace256'."""
    if K <= 8:
        return 'chain'
    if D >= 1024 and (K + 127) // 128 < 2 * G:
        return 'oop512'
    return 'inplace256'


# ------------------------------------------------------------ INT8 row slicer ----
def _awkward_wide(rows, cols, seed):
    """oracle-level rounding hazards spread over a row of more than 1024 elements: exact ties at the last digit in
    the first and in the last 128-column stretch, subnormals, zeros, the largest fixed-point value, 600 orders of
    magnitude within one row and rows of very different magnitude."""
    X = _rnd(rows, cols, seed=seed) * torch.exp(4 * _rnd(rows, 1, seed=seed + 1))
    ulp = 2.0 ** -(8 * S7 - 2)
    ties = torch.tensor([0.5, 1.5, 2.5, 3.5, -0.5, -1.5, -2.5, 127.5], device='cuda', dtype=torch.float64) * ulp
    X[0, :] = 0.0
    X[1, :] = X[1, :].clamp(-0.9, 0.9)
    X[1, 0] = 1.0 - 2.0 ** -53
    X[1, 1:9] = ties
    X[1, cols - 8:] = ties
    X[1, 1024] = -(1.0 - 2.0 ** -53)                      # the row maximum beyond column 1024
    X[2, :] = 5e-324 * torch.arange(cols, device='cuda', dtype=torch.float64)
    X[3, 0], X[3, cols // 2], X[3, cols - 1] = 1e-300, -4.9e-324, 1e300
    X[4, :] = -2.0 ** -3
    X[5, :-1] = 0.0                                       # a single non-zero in the last column
    X[5, -1] = 3.0
    return X


@pytest.mark.parametrize('cols', [1025, 2048, 3001])
def test_row_slicer_beyond_1024_columns(vt, cols):
    """Rows longer than 1024 elements are sliced by the RC = 0 instance, which re-reads the row from global memory:
    digits and scales bit-identical to the CPU model (the integer variant, which keeps rows in registers, refuses
    such rows, so this is the only path for them)."""
    X = _awkward_wide(203, cols, seed=60)
    d, sc = vt.ops.ozaki_slice(X, S7)
    d_ref, sc_ref = slicing.slice_rows(X.cpu().numpy(), S7)
    assert np.array_equal(d[:, :, :cols].cpu().numpy(), d_ref)
    assert np.array_equal(sc.cpu().numpy(), sc_ref)
    assert bool((d[:, :, cols:] == 0).all())
    fold = _rnd(203, seed=61)
    d2, sc2 = vt.ops.ozaki_slice(X, S7, fold=fold)
    assert torch.equal(d2, d) and torch.equal(sc2, sc * fold)
    with pytest.raises(ValueError):
        vt.ops.ozaki_slice(X, S7, integer_variant=True)


# ------------------------------------------------------- INT8 apply, many chunks ----
def _apply_model_check(Hinv, X, r, S, ch, seed):
    """Sampled entries of S against -digits_gemm of the CPU model bit for bit: first, second, middle and last
    column of EVERY chunk (the ragged last one included), 50 rows of H^{-1}."""
    N, D = X.shape
    cols = set()
    for c0 in range(0, N, ch):
        c1 = min(c0 + ch, N)
        cols.update([c0, c0 + 1, (c0 + c1) // 2, c1 - 1])
    cols = sorted(c for c in cols if c < N)
    rng = np.random.default_rng(seed)
    rows = sorted(set(rng.choice(D, size=min(D, 48), replace=False).tolist()) | {0, D - 1})
    dA, sA = slicing.slice_rows(Hinv[rows].cpu().numpy(), S7)
    dB, sB = slicing.slice_rows(X[cols].cpu().numpy(), S7)
    model = -slicing.digits_gemm(dA, sA, dB, sB * r[cols].cpu().numpy())
    got = S[rows][:, cols].cpu().numpy()
    mism = np.argwhere(got != model)
    assert mism.size == 0, 'apply differs from the CPU model at (row, col) {} of {}'.format(
        [(rows[i], cols[j]) for i, j in mism[:5]], len(mism))


@pytest.mark.parametrize('D', [1024, 1025, 2048, 2049, 4096])
def test_int8_apply_over_many_chunks(vt, sms, D):
    """ij_apply(precision='f64_ozaki') with at least three chunks at any SM count and a ragged last chunk.  D <= 1024:
    the GEMM of chunk c slices chunk c + 1 (fused converters, here on a third and later chunk); D > 1024: one
    slicing launch per chunk."""
    N = 3 * apply_chunk_max(D) + 777
    ch = apply_chunk_rows(N, D, sms)
    nchunks = -(-N // ch)
    assert nchunks >= 3 and N % ch != 0
    expected_launches = (2 + nchunks) if D <= 1024 else (1 + 2 * nchunks)
    assert vt.ops.resolve_precision('auto', N, D) == 'f64_ozaki'
    # exact design: every engine and torch agree to the last bit
    Hi = _dev(exact.integer_design(70 + D, D, D, vmax=exact.HMAX))
    Xi = _dev(exact.integer_design(71 + D, N, D))
    ri = _dev(exact.integer_vector(72 + D, N))
    S, nl = _launches(vt, lambda: vt.ops.ij_apply(Hi, Xi, ri, precision='f64_ozaki'))
    assert nl == expected_launches, (nl, expected_launches, ch)
    ref = -(Hi @ (Xi * ri[:, None]).T)
    assert torch.equal(S, ref), 'exact design: {} entries differ'.format(int((S != ref).sum()))
    del ref
    assert torch.equal(vt.ops.ij_apply(Hi, Xi, ri, precision='f64'), S)
    del S, Hi, Xi, ri
    # random full-precision data: rows of X on scales 12 orders of magnitude apart
    Hinv = torch.eye(D, device='cuda', dtype=torch.float64) + _rnd(D, D, seed=73) / math.sqrt(D)
    X = _rnd(N, D, seed=74) * torch.exp(3 * _rnd(N, 1, seed=75))
    r = _rnd(N, seed=76)
    S = vt.ops.ij_apply(Hinv, X, r, precision='f64_ozaki')
    _apply_model_check(Hinv, X, r, S, ch, seed=D)
    ref = -(Hinv @ (X * r[:, None]).T)
    _parity(S, ref, what='f64_ozaki vs torch D={}'.format(D))
    # the model bound: digits dropped and rounded, relative to the power-of-two scales, plus the reference's own error
    sig = _pow2_above(Hinv.abs().amax(dim=1))
    tau = _pow2_above(X.abs().amax(dim=1)) * r.abs()
    Ha = Hinv.abs()
    for c0 in range(0, N, 16384):                            # (in column blocks: the whole would need 3 more copies)
        c1 = min(c0 + 16384, N)
        acc = Ha @ (X[c0:c1].abs() * r[c0:c1].abs()[:, None]).T
        bound = slicing.error_bound(D, S7) * sig[:, None] * tau[None, c0:c1] + 2 * D * 2.0 ** -53 * acc
        assert bool(((S[:, c0:c1] - ref[:, c0:c1]).abs() <= bound).all()), 'model bound, columns {}..{}'.format(c0, c1)
    del ref, acc, bound
    _parity(S, vt.ops.ij_apply(Hinv, X, r, precision='f64'), what='f64_ozaki vs DMMA D={}'.format(D))


# ------------------------------------------------------ INT8 Hessian, many chunks ----
@pytest.mark.parametrize('D', [1536, 2048, 2049, 4096])
def test_int8_hessian_over_many_chunks(vt, sms, D):
    """syrk_weighted(precision='f64_ozaki') over at least three chunks with a ragged tail; the per-feature scales from
    the engine's own sweep (D > 2048: the only way) and, for D <= 2048, from the statistics pass."""
    ch = syrk_chunk_rows(1 << 40, D, sms)
    N = 3 * ch + 1001
    nchunks = -(-N // ch)
    assert nchunks == 4 and N <= exact.MAX_N
    # exact design
    Xi = _dev(exact.integer_design(80 + D, N, D))
    si = _dev(exact.square_weights(81 + D, N))
    H, nl = _launches(vt, lambda: vt.ops.syrk_weighted(Xi, si, precision='f64_ozaki'))
    assert nl == nchunks + 3, (nl, nchunks)          # column sweep, first slicing, one GEMM per chunk, finish
    ref = Xi.T @ (Xi * si[:, None])
    assert torch.equal(H, ref), 'exact design: {} entries differ'.format(int((H != ref).sum()))
    assert torch.equal(vt.ops.syrk_weighted(Xi, si, precision='f64'), ref)
    assert torch.equal(vt.ops.syrk_weighted(Xi, si, l2=3.0, precision='f64_ozaki'),
                       ref + 3.0 * torch.eye(D, device='cuda', dtype=torch.float64))
    del Xi, si, H, ref
    # random data, feature scales 6 orders of magnitude apart
    X = _rnd(N, D, seed=82) * torch.exp(2 * _rnd(1, D, seed=83))
    s = 0.25 * _uni(N, seed=84)
    s[::13] = 0.0
    H = vt.ops.syrk_weighted(X, s, precision='f64_ozaki')
    ref = X.T @ (X * s[:, None])
    _parity(H, ref, what='f64_ozaki vs torch D={}'.format(D))
    _parity(H, vt.ops.syrk_weighted(X, s, precision='f64'), what='f64_ozaki vs DMMA D={}'.format(D))
    assert torch.equal(H, H.T)
    sig = _pow2_above((X.abs() * s.sqrt()[:, None]).amax(dim=0))
    acc = X.abs().T @ (X.abs() * s[:, None])
    bound = slicing.error_bound(N, S7) * sig[:, None] * sig[None, :] + 2 * N * 2.0 ** -53 * acc
    assert bool(((H - ref).abs() <= bound).all())
    del acc, bound, ref
    theta = _rnd(D, seed=85) / math.sqrt(D)
    y = (_uni(N, seed=86) < 0.5).double()
    w = _uni(N, seed=87) + 0.5
    if D <= vt.ops.COLMAX_MAX_DIM:
        _, _, s2, _, cm = vt.ops.glm_stats(X, theta, y, w, want_colmax=True)
        Hf, nl = _launches(vt, lambda: vt.ops.syrk_weighted(X, s2, precision='f64_ozaki', colmax=cm))
        assert nl == nchunks + 2, (nl, nchunks)      # no sweep of its own
        assert torch.equal(Hf, vt.ops.syrk_weighted(X, s2, precision='f64_ozaki'))
        _parity(Hf, X.T @ (X * s2[:, None]), what='f64_ozaki with colmax vs torch D={}'.format(D))
    else:
        with pytest.raises(ValueError):
            vt.ops.glm_stats(X, theta, y, w, want_colmax=True)


def test_default_precision_end_to_end_beyond_the_colmax_width(vt, sms):
    """HyperparameterSensitivityLinearApproximation(GLMObjective(X, y)) with the default precision at D = 2560: 'auto'
    takes the INT8 engine, the statistics pass cannot carry the column maxima (D > 2048), the apply slices in
    separate launches (D > 1024).  The whole (D, N) result against torch float64 (cuSOLVER's Cholesky)."""
    N, D = 40001, 2560
    X = _rnd(N, D, seed=90) / math.sqrt(D)
    theta = 0.5 * _rnd(D, seed=91)
    p = torch.sigmoid(X @ (2 * _rnd(D, seed=92)))
    y = (_uni(N, seed=93) < p).double()
    w = torch.ones(N, device='cuda', dtype=torch.float64)
    obj = vt.objectives.GLMObjective(X, y)
    assert obj.precision == 'auto' and vt.ops.resolve_precision('auto', N, D, w) == 'f64_ozaki'
    assert D > vt.ops.COLMAX_MAX_DIM and 'colmax' not in obj.vt_stats(theta, w, for_hessian=True)
    sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
    S = torch.as_tensor(sens.get_dopt_dhyper(), device='cuda')
    assert sens.used_explicit_inverse
    mu = torch.sigmoid(X @ theta)
    H_ref = X.T @ (X * (mu * (1 - mu))[:, None])
    _parity(torch.as_tensor(sens.get_hessian_at_opt(), device='cuda'), H_ref, what='Hessian (auto, D=2560)')
    S_ref = -torch.cholesky_solve((X * (mu - y)[:, None]).T.contiguous(), torch.linalg.cholesky(H_ref))
    _parity(S, S_ref, what='dopt_dhyper (auto, D=2560)')
    del S, S_ref
    # the apply of that run: unfused, one slicing launch and one GEMM per chunk
    ch = apply_chunk_rows(N, D, sms)
    nchunks = -(-N // ch)
    stats = obj.vt_stats(theta, w, want_grad=False)
    _, nl = _launches(vt, lambda: obj.vt_ij_sensitivity(sens._hinv, stats))
    assert nchunks >= 2 and nl == 1 + 2 * nchunks, (nl, nchunks)


# ------------------------------------------------- fused GLM passes beyond 2048 ----
def _glm_refs(X, theta, y, w, l2):
    z = X @ theta
    mu = torch.sigmoid(z)
    resid = mu - y
    s = w * mu * (1 - mu)
    grad = X.T @ (w * resid) + l2 * theta
    return z, resid, s, grad, mu


@pytest.mark.parametrize('D', [2049, 4096, 8192])
def test_fused_glm_passes_beyond_2048(vt, D):
    """glm_stats / glm_hvp / glm_dirderiv (one direction) on the CPT = 8 (D <= 4096) and CPT = 16 (D <= 8192)
    instances, one row per staged block, against torch float64."""
    N = 3001
    X = _rnd(N, D, seed=100) / math.sqrt(D)
    theta = _rnd(D, seed=101)
    y = (_uni(N, seed=102) < 0.5).double()
    w = _uni(N, seed=103) + 0.5
    z, resid, s, grad, mu = _glm_refs(X, theta, y, w, 0.3)
    z1, r1, s1, g1 = vt.ops.glm_stats(X, theta, y, w, l2=0.3)
    for a, b, name in ((z1, z, 'z'), (r1, resid, 'resid'), (s1, s, 's'), (g1, grad, 'grad')):
        _parity(a, b, what='glm_stats {} D={}'.format(name, D))
    v = _rnd(D, seed=104)
    _parity(vt.ops.glm_hvp(X, s, v, ridge=0.7), X.T @ (s * (X @ v)) + 0.7 * v, what='glm_hvp D={}'.format(D))
    d2 = w * mu * (1 - mu)                                    # b''(z) for the logistic family
    _parity(vt.ops.glm_dirderiv(X, z, v[None, :], w), X.T @ (d2 * (X @ v)), what='glm_dirderiv D={}'.format(D))


def test_fused_glm_passes_refuse_d_above_8192(vt):
    N, D = 17, 8193
    X = _rnd(N, D, seed=110)
    theta, v = _rnd(D, seed=111), _rnd(D, seed=112)
    y, s = torch.zeros(N, device='cuda', dtype=torch.float64), torch.ones(N, device='cuda', dtype=torch.float64)
    with pytest.raises(ValueError, match='8192'):
        vt.ops.glm_stats(X, theta, y)
    with pytest.raises(ValueError, match='8192'):
        vt.ops.glm_hvp(X, s, v)
    with pytest.raises(ValueError, match='8192'):
        vt.ops.glm_dirderiv(X, X @ theta, v[None, :])
    torch.cuda.synchronize()


def test_hvp_multi_beyond_2048_takes_the_gemm_route(vt):
    """K > 1 directions at D = 2049: the fused multi-direction kernel refuses (checked through the C entry point),
    glm_hvp_multi takes the two-GEMM route (fewer launches than K single passes) and matches K single products."""
    from vittles_b200._cabi import ptr, require_cuda, stream
    N, D, K = 3001, 2049, 5
    X = _rnd(N, D, seed=120) / math.sqrt(D)
    s = _uni(N, seed=121)
    V = _rnd(K, D, seed=122)
    out, nl = _launches(vt, lambda: vt.ops.glm_hvp_multi(X, s, V, ridge=0.25))
    assert nl <= 4 < 2 * K
    single = torch.stack([vt.ops.glm_hvp(X, s, V[k], ridge=0.25) for k in range(K)])
    _parity(out, single, what='hvp_multi vs single products')
    _parity(out, (V @ X.T * s[None, :]) @ X + 0.25 * V, what='hvp_multi vs torch')
    lib = require_cuda()
    ws = torch.empty(lib.vt_glm_hvp_multi_workspace_bytes(D, 3) // 8 + 1, dtype=torch.float64, device='cuda')
    o = torch.empty((3, D), dtype=torch.float64, device='cuda')
    st = lib.vt_glm_hvp_multi(ptr(X), D, N, D, ptr(s), ptr(V), 3, 0.0, ptr(o), ptr(ws), ws.numel() * 8, stream())
    assert st == 2                                      # VT_ERR_INVALID, no launch


# ---------------------------------------------------------------- dense Cholesky ----
def _spd(D, seed):
    A = _rnd(D, D + 5, seed=seed)
    return A @ A.T / D + torch.eye(D, device='cuda', dtype=torch.float64)


def _backward_error(H, Xs, B):
    return float(torch.linalg.matrix_norm(H @ Xs - B) / (torch.linalg.matrix_norm(H) * torch.linalg.matrix_norm(Xs)))


def _sentinel_block(rows, cols, pad, off):
    """A (rows, cols + pad) buffer of sentinel NaNs and its (rows, cols) column block at column `off`."""
    big = torch.full((rows, cols + pad), SENTINEL, dtype=torch.int64, device='cuda').view(torch.float64)
    return big, big[:, off:off + cols]


def _sentinels_intact(big, view_cols):
    """Every entry of `big` outside the given column range still holds the sentinel bit pattern."""
    bits = big.view(torch.int64)
    mask = torch.ones_like(bits, dtype=torch.bool)
    mask[:, view_cols[0]:view_cols[1]] = False
    return bool((bits[mask] == SENTINEL).all())


@pytest.mark.parametrize('D', [1023, 1024, 1025, 2049])
def test_potrf_and_solve_at_block_edges(vt, sms, D):
    """D = 2049: the last 128-, 256- and 512-blocks hold one row (the n1 <= 0 branches of the inverted-block
    builds).  scipy's cho_solve and the backward error, which does not depend on scipy."""
    H = _spd(D, seed=130 + D)
    B = _rnd(D, 300, seed=131)
    f = vt.ops.potrf(H)
    Xs = f.solve(B)
    Hn, Bn = H.cpu().numpy(), B.cpu().numpy()
    ref = scipy.linalg.cho_solve(scipy.linalg.cho_factor(Hn, lower=True), Bn)
    assert_close(Xs, ref, rtol=1e-8, atol_scale=1e-11, what='solve D={}'.format(D))
    assert _backward_error(H, Xs, B) <= D * 2.0 ** -53
    assert_close(torch.tril(f.L), np.linalg.cholesky(Hn), rtol=1e-9, atol_scale=1e-12)
    assert solve_regime(D, 300, sms) == ('oop512' if D >= 1024 else 'inplace256')


def _regime_K(kind, D, G):
    if kind == 'chain':
        return 8
    if kind == 'chain+1':
        return 9
    if kind == 'ragged':
        return {1024: 1300, 2049: 1100}[D]
    return 2 * 128 * G + 77                       # in place


@pytest.mark.parametrize('D', [1024, 2049])
@pytest.mark.parametrize('kind', ['chain', 'chain+1', 'ragged', 'inplace'])
def test_solve_regimes_and_padded_right_hand_sides(vt, sms, D, kind):
    """chol_potrs in each regime, K computed from the SM count: the chain (K = 8) and its first excluded width (K =
    9, the 512-row form), the 512-row out-of-place form over several passes with a ragged last one, and the 256-row
    in-place form at D >= 1024 (K >= 2 x 128 x #SM - 127).  Then vt_potrs on a (D, K) column block of a (D, K + 24)
    buffer at an even and an odd column offset: bit-identical to the contiguous solve, padding untouched."""
    from vittles_b200._cabi import check, ptr, require_cuda, stream
    K = _regime_K(kind, D, sms)
    regime = solve_regime(D, K, sms)
    assert regime == {'chain': 'chain', 'chain+1': 'oop512', 'ragged': 'oop512', 'inplace': 'inplace256'}[kind]
    if kind == 'ragged':
        cap = solve_scratch_cols(D)
        assert K > cap and K % cap != 0
    H = _spd(D, seed=140 + D)
    f = vt.ops.potrf(H)
    B = _rnd(D, K, seed=141)
    Xs, nl = _launches(vt, lambda: f.solve(B))
    if regime == 'chain':
        assert nl == 2                          # one cooperative launch per direction
    if K <= 2000:
        ref = _dev(scipy.linalg.cho_solve(scipy.linalg.cho_factor(H.cpu().numpy(), lower=True), B.cpu().numpy()))
    else:
        ref = torch.cholesky_solve(B, torch.linalg.cholesky(H))
    _parity(Xs, ref, atol_scale=1e-11, what='{} D={} K={}'.format(kind, D, K))
    del ref
    assert _backward_error(H, Xs, B) <= D * 2.0 ** -53
    lib = require_cuda()
    for off in (2, 7):
        big, view = _sentinel_block(D, K, 24, off)
        view.copy_(B)
        check(lib.vt_potrs(ptr(f.L), f.L.stride(0), D, ptr(f.dinv), ptr(view), big.stride(0), K, stream()))
        assert torch.equal(view, Xs), 'column offset {}: {} entries differ'.format(off, int((view != Xs).sum()))
        assert _sentinels_intact(big, (off, off + K)), 'column offset {}: padding overwritten'.format(off)
        del big, view


def test_cholesky_inverse_at_2049(vt, sms):
    """CholeskyFactor.inverse(): 2049 right-hand sides, three passes of the 512-row form (the last of one column)."""
    D = 2049
    H = _spd(D, seed=150)
    assert solve_regime(D, D, sms) == 'oop512' and D % solve_scratch_cols(D) != 0
    inv = vt.ops.potrf(H).inverse()
    _parity(inv, torch.cholesky_inverse(torch.linalg.cholesky(H)), atol_scale=1e-11, what='inverse D=2049')


def test_substitution_in_place_regime_matches_the_explicit_inverse(vt, sms):
    """vt_ij_sensitivity_by_substitution solves the (D, N) matrix -G^T in place; with N above the in-place threshold
    and D = 1024 that is the 256-row in-place regime (one CTA per block row of each column tile)."""
    D = 1024
    N = 2 * 128 * sms + 77
    assert solve_regime(D, N, sms) == 'inplace256'
    X = _rnd(N, D, seed=160) / math.sqrt(D)
    theta = _rnd(D, seed=161)
    y = (_uni(N, seed=162) < 0.5).double()
    obj = vt.objectives.GLMObjective(X, y, precision='f64')
    stats = obj.vt_stats(theta, None)
    f = vt.ops.potrf(obj.vt_hessian(theta, None, stats))
    assert f.cond_lower_bound() < 1e3
    S_sub = obj.vt_ij_sensitivity_by_substitution(f, stats)
    S_inv = obj.vt_ij_sensitivity(f.inverse(), stats)
    _parity(S_sub, S_inv, what='substitution vs explicit inverse')


def _minor(err):
    """The index of the failing leading minor in a LinAlgError: ours and older scipy say 'k-th leading minor',
    newer scipy 'potrf return info = [k]' (LAPACK's info)."""
    m = re.search(r'(\d+)-th leading minor|info = \[?(\d+)', str(err))
    return int(m.group(1) or m.group(2))


@pytest.mark.parametrize('k', [1, 128, 129, 300, 1500])
def test_first_non_pd_minor_is_reported(vt, k):
    """H = L diag(d) L^T with d_{k-1} = -1: the leading minors 1 .. k-1 are PD, minor k is not.  potrf raises
    LinAlgError naming minor k - the index scipy reports - also when k lies in a late block while the look-ahead
    updates run on the helper stream."""
    D = 1500
    L = torch.eye(D, device='cuda', dtype=torch.float64) + torch.tril(_rnd(D, D, seed=170), -1) / math.sqrt(D)
    d = torch.ones(D, device='cuda', dtype=torch.float64)
    d[k - 1] = -1.0
    H = (L * d[None, :]) @ L.T
    H = 0.5 * (H + H.T)
    with pytest.raises(np.linalg.LinAlgError) as ours:
        vt.ops.potrf(H)
    with pytest.raises(np.linalg.LinAlgError) as theirs:
        scipy.linalg.cho_factor(H.cpu().numpy(), lower=True)
    assert _minor(ours.value) == k, str(ours.value)
    assert _minor(theirs.value) == k, str(theirs.value)


# ------------------------------------------------------- padded and offset views ----
def _views(X):
    """{name: a view with the values of X}: padded rows (ld = D + 1, D + 2), a base one row into a buffer (8 bytes
    off the 16-byte alignment when D is odd) and a contiguous copy."""
    N, D = X.shape
    out = {'contiguous': X.clone()}
    for pad in (1, 2):
        big = torch.full((N, D + pad), float('nan'), dtype=torch.float64, device='cuda')
        big[:, :D] = X
        out['ld+{}'.format(pad)] = big[:, :D]
    big = torch.full((N + 1, D), float('nan'), dtype=torch.float64, device='cuda')
    big[1:] = X
    out['offset'] = big[1:]
    return out


def _run_layout(vt, name, Xv, ops_in):
    """One kernel on the view Xv; matrix outputs go to a column block of a wider sentinel buffer."""
    N, D = Xv.shape
    theta, y, w, s, V, Hinv, r, z = ops_in
    if name == 'gemm':
        big, out = _sentinel_block(N, 5, 3, 1)
        vt.ops.gemm(Xv, V[:5], out=out)
        return out.clone(), _sentinels_intact(big, (1, 6))
    if name in ('syrk_f64', 'syrk_f64_ozaki'):
        big, out = _sentinel_block(D, D, 3, 1)
        vt.ops.syrk_weighted(Xv, s, out=out, precision=name[5:])
        return out.clone(), _sentinels_intact(big, (1, 1 + D))
    if name in ('apply_f64', 'apply_f64_ozaki'):
        big, out = _sentinel_block(D, N, 3, 1)
        vt.ops.ij_apply(Hinv, Xv, r, out=out, precision=name[6:])
        return out.clone(), _sentinels_intact(big, (1, 1 + N))
    if name == 'glm_stats':
        big = torch.full((3, N + 2), SENTINEL, dtype=torch.int64, device='cuda').view(torch.float64)
        z, res, sv, g = vt.ops.glm_stats(Xv, theta, y, w, l2=0.1, out=(big[0, 1:1 + N], big[1, 1:1 + N], big[2, 1:1 + N]))
        return torch.cat([z, res, sv, g]), _sentinels_intact(big, (1, 1 + N))
    if name == 'glm_hvp':
        return vt.ops.glm_hvp(Xv, s, V[0], ridge=0.5), True
    if name == 'glm_hvp_multi':
        return vt.ops.glm_hvp_multi(Xv, s, V[:3], ridge=0.5), True
    if name == 'glm_dirderiv':
        return vt.ops.glm_dirderiv(Xv, z, V[:2] if D <= 2048 else V[:1], w), True     # (one direction beyond 2048)
    raise AssertionError(name)


KERNELS = ['gemm', 'syrk_f64', 'syrk_f64_ozaki', 'apply_f64', 'apply_f64_ozaki', 'glm_stats', 'glm_hvp',
           'glm_hvp_multi', 'glm_dirderiv']


@pytest.mark.parametrize('D', [77, 1000, 2500])
def test_padded_and_offset_views_are_bit_identical(vt, D):
    """Every row-staging branch (one bulk copy, a bulk copy per row, plain loads; vector or scalar loads in the GEMM
    and slicing kernels) with the same arithmetic order: results bit-identical to the contiguous input, and the
    sentinels around every output block untouched."""
    N = 3001
    X = _rnd(N, D, seed=180) / math.sqrt(D)
    theta = _rnd(D, seed=181)
    y = (_uni(N, seed=182) < 0.5).double()
    w = _uni(N, seed=183) + 0.5
    s = _uni(N, seed=184)
    V = _rnd(5, D, seed=185)
    Hinv = torch.eye(D, device='cuda', dtype=torch.float64) + _rnd(D, D, seed=186) / math.sqrt(D)
    r = _rnd(N, seed=187)
    z = X @ theta
    ops_in = (theta, y, w, s, V, Hinv, r, z)
    views = _views(X)
    for name in KERNELS:
        base, ok = _run_layout(vt, name, views['contiguous'], ops_in)
        assert ok, '{}: sentinels overwritten (contiguous)'.format(name)
        for lay, Xv in views.items():
            got, ok = _run_layout(vt, name, Xv, ops_in)
            assert ok, '{} {} D={}: sentinels overwritten'.format(name, lay, D)
            assert torch.equal(got, base), '{} {} D={}: {} entries differ from the contiguous run'.format(
                name, lay, D, int((got != base).sum()))
