"""GPU tests of the TF32 engine (``csrc/tgemm.cu``, precision 'tf32' | 'tf32x3') at the points where its plan
changes: the 128-row and 256 / 128-column tile edges, the 32-k block edges, the 4096-k FP32 accumulation segments
(flushed to FP64), split-K parts, several conversion chunks with a ragged last one, D > 4096 in the apply, padded and
offset views, the scalar epilogue and non-finite inputs.

The drivers' plans are restated below from the SM count (``chunk_rows``, ``pick_parts``, ``count_tiles``, the
segment rule), and every test checks that it reached its branch: through the launch count (one reduction launch
when the GEMM keeps FP64 partial tiles, one conversion and one GEMM per chunk) and through the workspace sizes the
library reports, which are functions of the chunk rows and the number of parts.

Three kinds of reference:

* Integer data on which both splits must equal torch float64 bit for bit.  Operands are integers of magnitude at
  most 16 (for the Hessian sqrt(s) x with s a power of four, so |sqrt(s) x| <= 16 and sqrt(s) is exact), integer
  H^{-1} and residuals, power-of-two alpha / row / column scales.  TF32 (11 significant bits) holds every operand
  exactly, so lo = 0; every product is exact in FP32; a 4096-term segment sums at most 4096 x 256 = 2^20 in
  magnitude on a grid of 1/4 at the finest, which FP32 holds exactly; segments, parts and chunks are summed in FP64,
  exactly.  Any difference is a misplaced tile, block, segment, part or chunk.
* Probes of the low-order operands of 'tf32x3': A with one power of two a per row, at column k (every k mod 32, in
  several k-blocks and segments), gives out[m, n] = a (B_hi + B_lo)[n, k].  For FP32-valued B that sum is a multiple
  of ulp(B) below 2 |B|, so FP32 holds it and the accumulation is exact.  The mirror case (B one-hot) probes A_lo.
* A componentwise bar on random data, |out - A B^T| <= c (|A| |B|^T) entry by entry, from the engine's model:
  - TF32 rounding (to nearest, 11 significant bits) after the FP64 -> FP32 cast: relative u = 2^-11 (1 + 2^-12) per
    operand; after the hi / lo split the operand error is 2^-22 (1 + 2^-11), and the omitted A_lo B_lo term is below
    2^-22 (1 + 2^-9) |A| |B|, so 'tf32' has 2u + u^2 and 'tf32x3' 3 * 2^-22 (1 + 2^-8);
  - products exact in FP32;
  - FP32 accumulation of the n products of one segment (n = L for 'tf32', 3 L for 'tf32x3', L <= 4096 the k of the
    longest segment in the plan), one rounding of unit 2^-24 per product: gamma_n = n 2^-24 / (1 - n 2^-24),
    times the sum of |products| <= (1 + 2^-8) |A| |B|;
  - FP64 beyond: segment, part and chunk sums, the scaling epilogue and the float64 reference itself, 2 (K + 8) 2^-53.
  At K <= 256 the 'tf32x3' bar is below the error of a split that drops either cross term (checked on the host by
  ``test_componentwise_bar_rejects_a_dropped_cross_term``, which needs no GPU).
"""
import math

import numpy as np
import pytest
import torch

from test_gpu_dispatch_edges import _launches, _sentinel_block, _sentinels_intact

TBM, TBK, SEG_KBLOCKS = 128, 32, 128      # tile rows, k per block, k-blocks per FP32 segment (tgemm.cu)
BN = {1: 256, 3: 128}                     # tile columns of the 'tf32' / 'tf32x3' instances
CHUNK_BYTES = 160 << 20                   # converted X of one chunk (chunk_rows in tgemm.cu)
SPLIT = {'tf32': 1, 'tf32x3': 3}
PRECISIONS = ['tf32', 'tf32x3']
U_TF32 = 2.0 ** -11 * (1 + 2.0 ** -12)
gpu = pytest.mark.gpu


@pytest.fixture(scope='module')
def vt():
    import vittles_b200
    return vittles_b200


@pytest.fixture(scope='module')
def sms(vt):
    return vt.ops.device_info()['sm_count']


@pytest.fixture(scope='module')
def lib(vt):
    from vittles_b200._cabi import require_cuda
    return require_cuda()


def _cdiv(a, b):
    return -(-a // b)


def _align(x, a=256):
    return _cdiv(x, a) * a


# --------------------------------------------------------- plans of the drivers ----
def lower_cols(tm, tiles_n, bn):
    return min((tm * TBM + TBM - 1) // bn + 1, tiles_n)


def count_tiles(M, N, bn, lower):
    tm, tn = _cdiv(M, TBM), _cdiv(N, bn)
    return sum(lower_cols(i, tn, bn) for i in range(tm)) if lower else tm * tn


def pick_parts(ntiles, kblocks, G):
    """Split-K parts: the fewest that fill 90 % of a wave of G CTAs, each with at least 16 k-blocks."""
    if ntiles >= 2 * G:
        return 1
    pmax = min(kblocks // 16, 4 * G)
    if pmax < 2:
        return 1
    best, best_eff = 1, 0.0
    for P in range(1, pmax + 1):
        U = ntiles * P
        eff = U / (G * _cdiv(U, G))
        if eff > best_eff + 1e-9:
            best, best_eff = P, eff
        if eff >= 0.9:
            break
    return best


def chunk_rows(N, D, split, tile_n, tiles_m, G):
    """Rows of X converted per pass: 160 MB of TF32 operands, trimmed so that the chunk's tiles fill whole waves."""
    ld = _cdiv(D, 4) * 4
    nb = max(1, CHUNK_BYTES // (ld * 4 * (2 if split == 3 else 1)) // tile_n)
    if tiles_m > 0:
        best, best_eff, b = nb, 0.0, nb
        while b >= 1 and b > nb // 2:
            T = b * tiles_m
            eff = T / (G * _cdiv(T, G))
            if eff > best_eff + 1e-9:
                best, best_eff = b, eff
            b -= 1
        nb = best
    return min(nb * tile_n, N)


def gemm_plan(M, N, K, split, G, parts=0, lower=False):
    """One GEMM launch: tiles, parts, FP32 segments of the longest unit, whether FP64 partial tiles (and the
    reduction launch) are used, and the k of the longest segment."""
    bn = BN[split]
    kblocks = _cdiv(K, TBK)
    ntiles = count_tiles(M, N, bn, lower)
    P = parts or pick_parts(ntiles, kblocks, G)
    unit_kb = _cdiv(kblocks, P)
    use_ws = P > 1 or unit_kb > SEG_KBLOCKS or lower
    return dict(ntiles=ntiles, parts=P, segments=_cdiv(unit_kb, SEG_KBLOCKS), use_ws=use_ws,
                ws_bytes=ntiles * min(P, kblocks) * TBM * bn * 8 if use_ws else 0,
                seg_len=min(K, TBK * min(unit_kb, SEG_KBLOCKS)))


def apply_plan(N, D, split, G):
    """ij_apply_tf32: Hinv converted once, then per chunk of X one conversion and one GEMM (M = D, K = D)."""
    ld, nops = _cdiv(D, 4) * 4, 2 if split == 3 else 1
    ch = chunk_rows(N, D, split, BN[split], _cdiv(D, TBM), G)
    g = gemm_plan(D, ch, D, split, G, parts=1)
    chunks = _cdiv(N, ch)
    return dict(g, chunk=ch, chunks=chunks, launches=1 + chunks * (2 + g['use_ws']),
                ws_bytes=(_align(D * ld * 4) + _align(ch * ld * 4)) * nops + g['ws_bytes'])


def hessian_plan(N, D, split, G):
    """syrk_tf32: per chunk of observations one conversion and one GEMM into the lower-triangle partial tiles,
    then one reduction (mirror)."""
    ld, nops = _cdiv(D, 4) * 4, 2 if split == 3 else 1
    ch = chunk_rows(N, D, split, TBK, 0, G)
    parts = pick_parts(count_tiles(D, D, BN[split], True), _cdiv(ch, TBK), G)
    g = gemm_plan(D, D, ch, split, G, parts=parts, lower=True)
    chunks = _cdiv(N, ch)
    return dict(g, chunk=ch, chunks=chunks, launches=2 * chunks + 1,
                ws_bytes=_align(ch * ld * 4) * nops + g['ws_bytes'])


def _report(what, plan):
    print('{}: {}'.format(what, ', '.join('{}={}'.format(k, plan[k]) for k in
                                          ('chunks', 'parts', 'segments', 'use_ws') if k in plan)))


# ------------------------------------------------------------------ data ----
def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _ints(shape, vmax, seed):
    return torch.randint(-vmax, vmax + 1, shape, generator=_gen(seed), device='cuda').double()


def _pow2(n, seed, emax=4):
    """(n,) powers of two 2^e, |e| <= emax, with random signs."""
    g = _gen(seed)
    e = torch.randint(-emax, emax + 1, (n,), generator=g, device='cuda')
    sign = torch.randint(0, 2, (n,), generator=g, device='cuda').double() * 2 - 1
    return torch.ldexp(sign, e)


def _pow4_weights(n, seed):
    """(n,) weights in {0, 1/4, 1, 4}: sqrt(s) is exact."""
    idx = torch.randint(0, 4, (n,), generator=_gen(seed), device='cuda')
    return torch.tensor([0.0, 0.25, 1.0, 4.0], dtype=torch.float64, device='cuda')[idx]


def _rnd(*shape, seed=0):
    return torch.randn(*shape, generator=_gen(seed), device='cuda', dtype=torch.float64)


def _tf32_round(x32):
    b = x32.view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def _product(A, B, mode):
    return A @ B.T if mode == 'KC' else A.T @ B


def _diff(out, ref):
    return '{} of {} entries differ'.format(int((out != ref).sum()), out.numel())


# ------------------------------------------------------- the componentwise bar ----
def bar(seg_len, split, K):
    """c in |out - A B^T| <= c (|A| |B|^T) (module docstring)."""
    if split == 1:
        e_op, n = 2 * U_TF32 + U_TF32 ** 2, seg_len
    else:
        e_op, n = 3 * 2.0 ** -22 * (1 + 2.0 ** -8), 3 * seg_len
    gamma = n * 2.0 ** -24 / (1 - n * 2.0 ** -24)
    return e_op + gamma * (1 + 2.0 ** -8) + 2 * (K + 8) * 2.0 ** -53


def _np_tf32(x):
    b = x.astype(np.float32).view(np.int32)
    return ((b + 0x1000) & ~0x1FFF).view(np.float32).astype(np.float64)


def _np_split(x):
    h = _np_tf32(x)
    return h, _np_tf32(x - h)


@pytest.mark.parametrize('K', [4, 32, 100, 256])
def test_componentwise_bar_rejects_a_dropped_cross_term(K):
    """Host simulation of the split in float64 (no FP32 accumulation): A_hi B_hi + A_hi B_lo + A_lo B_hi is within
    the 'tf32x3' bar; with either cross term dropped it is not, so a lo operand the engine misreads fails it."""
    rng = np.random.default_rng(K)
    A = rng.standard_normal((200, K)) * np.exp2(rng.integers(-10, 11, size=(200, 1)))
    B = rng.standard_normal((300, K)) * np.exp2(rng.integers(-10, 11, size=(300, 1)))
    exact, acc = A @ B.T, np.abs(A) @ np.abs(B).T
    (Ah, Al), (Bh, Bl) = _np_split(A), _np_split(B)
    c = bar(K, 3, K)
    rel = lambda out: float((np.abs(out - exact) / acc).max())
    assert rel(Ah @ Bh.T + Ah @ Bl.T + Al @ Bh.T) <= c
    assert rel(Ah @ Bh.T + Ah @ Bl.T) > c, 'A_lo B_hi dropped'
    assert rel(Ah @ Bh.T + Al @ Bh.T) > c, 'A_hi B_lo dropped'
    assert rel(Ah @ Bh.T) <= bar(K, 1, K)


# ---------------------------------------------------- coverage of the shapes ----
APPLY_D = [1, 3, 77, 128, 129, 256, 257, 1024, 2049, 4096, 4097, 6000, 8192]
SWEEP_MN = [1, 127, 128, 129, 255, 256, 257]
SWEEP_K = [1, 4, 31, 32, 33, 4095, 4096, 4097, 8193]
LONG_K = 300013                           # few tiles: split-K parts of more than one segment each


def _segment_shape(split, G):
    """(M, N) with at least 2 G tiles (so one part per tile, every unit as long as K) and ragged edges."""
    return 16 * TBM - 3, BN[split] * _cdiv(2 * G, 16) - 5


def _big_chunks(chunk):
    """Three full chunks and a ragged fourth."""
    return 3 * chunk + chunk // 2 + 77


@gpu
def test_the_shapes_reach_every_branch(sms):
    """At this SM count the parametrisations below reach: split-K parts in the tile sweep; parts of several
    segments; a single part of several segments; applies with and without FP64 partial tiles (D > 4096); Hessians
    whose chunks run in parts and in several segments."""
    for split in (1, 3):
        sweep = [gemm_plan(M, N, K, split, sms) for M in SWEEP_MN for N in SWEEP_MN for K in SWEEP_K]
        assert any(p['parts'] > 1 for p in sweep) and any(not p['use_ws'] for p in sweep)
        long_k = gemm_plan(129, 129, LONG_K, split, sms)
        assert long_k['parts'] > 1 and long_k['segments'] > 1, long_k
        seg = gemm_plan(*_segment_shape(split, sms), 8193, split, sms)
        assert seg['parts'] == 1 and seg['segments'] == 3, seg
        applies = [apply_plan(1 << 40, D, split, sms) for D in APPLY_D]
        assert [p['use_ws'] for p in applies] == [D > 4096 for D in APPLY_D]
        hess = [hessian_plan(1 << 40, D, split, sms) for D in APPLY_D]
        assert any(p['parts'] > 1 and p['segments'] > 1 for p in hess)
        assert any(p['parts'] == 1 and p['segments'] > 1 for p in hess)


# ---------------------------------------------------- probes of the lo operands ----
def _one_hot(rows, K):
    """(rows, K) with one power of two per row: row h at k = 32 kb + kk, kk running through every k mod 32 in each
    group of 32 rows (shifted from group to group), kb through early, segment-edge and last k-blocks."""
    kblocks = _cdiv(K, TBK)
    sel = sorted({0, 1, 31, 126, 127, 128, 129, 200, 255, kblocks - 2, kblocks - 1})
    h = torch.arange(rows, device='cuda')
    kb = torch.tensor(sel, device='cuda')[(h // 32) % len(sel)]
    k = torch.clamp(kb * TBK + (h + h // 32) % 32, max=K - 1)
    a = torch.ldexp(torch.where(h % 3 == 0, -1.0, 1.0).double(), (h % 7 - 3))
    hot = torch.zeros((rows, K), dtype=torch.float64, device='cuda')
    hot[h, k] = a
    return hot, k, a


@gpu
@pytest.mark.parametrize('case', ['split-k', 'segments'])
@pytest.mark.parametrize('side', ['A', 'B'])
@pytest.mark.parametrize('mode', ['KC', 'KS'])
def test_lo_operand_probe(vt, sms, mode, side, case):
    """'tf32x3' with one operand one-hot and the other FP32-valued: out = a (hi + lo) of the other operand at the hot
    k, bit for bit.  Side 'A' (A one-hot) reads B_lo, side 'B' reads A_lo; a lo tile from a wrong stage, k offset or
    swizzle row, or a dropped cross term, changes the low bits."""
    K = 8193
    hot_rows, other_rows = (320, 200) if case == 'split-k' else _segment_shape(3, sms)
    M, N = (hot_rows, other_rows) if side == 'A' else (other_rows, hot_rows)
    plan = gemm_plan(M, N, K, 3, sms)
    assert (plan['parts'] > 1) if case == 'split-k' else (plan['parts'] == 1 and plan['segments'] == 3), plan
    hot, k, a = _one_hot(hot_rows, K)
    other = _rnd(other_rows, K, seed=2).float().double()
    if mode == 'KS':
        hot, other = hot.T.contiguous(), other.T.contiguous()
    hi, lo = vt.ops.tf32_convert(other, split=3)
    cols = other.shape[1]
    assert torch.equal(hi[:, :cols], _tf32_round(other.float()))
    assert torch.equal(lo[:, :cols], _tf32_round((other - hi[:, :cols].double()).float()))
    osum = hi[:, :cols].double() + lo[:, :cols].double()
    if mode == 'KS':
        osum = osum.T                                            # (other_rows, K)
    expect = a[:, None] * osum[:, k].T                           # (hot_rows, other_rows)
    if side == 'A':
        out = vt.ops.tf32_gemm(hot, other, mode, mode, precision='tf32x3')
    else:
        out = vt.ops.tf32_gemm(other, hot, mode, mode, precision='tf32x3')
        expect = expect.T
    assert torch.equal(out, expect), '{} side {} {}: {}'.format(mode, side, case, _diff(out, expect))
    _report('probe {} side {} {} M={} N={}'.format(mode, side, case, M, N), plan)


# ----------------------------------------------------------- exact: tf32_gemm ----
def _exact_gemm_case(vt, lib, sms, mode, precision, M, N, K, A, B, seed):
    split = SPLIT[precision]
    rs, cs = _pow2(M, seed), _pow2(N, seed + 1)
    plan = gemm_plan(M, N, K, split, sms)
    out, nl = _launches(vt, lambda: vt.ops.tf32_gemm(A, B, mode, mode, alpha=-0.25, precision=precision,
                                                     rowscale=rs, colscale=cs))
    assert nl == 3 + plan['use_ws'], (M, N, K, nl, plan)          # two conversions, the GEMM [, the reduction]
    assert lib.vt_tf32_gemm_workspace_bytes(M, N, K, split) == plan['ws_bytes'], (M, N, K)
    ref = -0.25 * rs[:, None] * cs[None, :] * _product(A, B, mode)
    assert torch.equal(out, ref), '{} {} M={} N={} K={}: {}'.format(mode, precision, M, N, K, _diff(out, ref))
    return plan


@gpu
@pytest.mark.parametrize('K', SWEEP_K)
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('mode', ['KC', 'KS'])
def test_gemm_exact_at_tile_and_block_edges(vt, lib, sms, mode, precision, K):
    """Every M, N in {1, 127, 128, 129, 255, 256, 257} (the 128-row tile, the 256 / 128-column tiles) at this K;
    integer operands, power-of-two alpha and scales: bit for bit equal to torch float64."""
    Mx = max(SWEEP_MN)
    A = _ints((Mx, K) if mode == 'KC' else (K, Mx), 16, seed=K)
    B = _ints((Mx, K) if mode == 'KC' else (K, Mx), 16, seed=K + 1)
    reached = set()
    for M in SWEEP_MN:
        for N in SWEEP_MN:
            Am = A[:M] if mode == 'KC' else A[:, :M]
            Bn = B[:N] if mode == 'KC' else B[:, :N]
            plan = _exact_gemm_case(vt, lib, sms, mode, precision, M, N, K, Am, Bn, seed=M * 1000 + N)
            reached.add((plan['parts'], plan['segments']))
    print('{} {} K={}: (parts, segments) reached {}'.format(mode, precision, K, sorted(reached)))
    if _cdiv(K, TBK) >= 32:                                       # at least two parts of 16 k-blocks
        assert any(p > 1 for p, _ in reached)


@gpu
@pytest.mark.parametrize('case', ['split-k', 'segments'])
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('mode', ['KC', 'KS'])
def test_gemm_exact_long_k(vt, lib, sms, mode, precision, case):
    """'split-k': a 129 x 129 output over 300013 k, split into parts of several segments each; 'segments': at
    least 2 x #SM tiles, so one part per tile, over 8193 k (three segments, the last of one k)."""
    split = SPLIT[precision]
    M, N, K = (129, 129, LONG_K) if case == 'split-k' else _segment_shape(split, sms) + (8193,)
    plan = gemm_plan(M, N, K, split, sms)
    if case == 'split-k':
        assert plan['parts'] > 1 and plan['segments'] > 1, plan
    else:
        assert plan['parts'] == 1 and plan['segments'] == 3, plan
    A = _ints((M, K) if mode == 'KC' else (K, M), 16, seed=5)
    B = _ints((N, K) if mode == 'KC' else (K, N), 16, seed=6)
    _exact_gemm_case(vt, lib, sms, mode, precision, M, N, K, A, B, seed=7)
    _report('{} {} {} M={} N={} K={}'.format(mode, precision, case, M, N, K), plan)


# ------------------------------------------------------------ exact: ij_apply ----
@gpu
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('D', APPLY_D)
def test_apply_exact_over_chunks(vt, lib, sms, D, precision):
    """ij_apply over three full conversion chunks and a ragged fourth; D > 4096 runs the GEMM over two or more
    FP32 segments into FP64 partial tiles.  Integer data: bit for bit equal to torch float64."""
    split = SPLIT[precision]
    N = _big_chunks(apply_plan(1 << 40, D, split, sms)['chunk'])
    plan = apply_plan(N, D, split, sms)
    assert plan['chunks'] == 4 and N % plan['chunk'] != 0
    assert plan['use_ws'] == (D > 4096) and (plan['segments'] > 1) == (D > 4096)
    Hi = _ints((D, D), 8, seed=D)
    Hi.diagonal().fill_(5.0)
    Xi = _ints((N, D), 16, seed=D + 1)
    ri = _ints((N,), 8, seed=D + 2)
    S, nl = _launches(vt, lambda: vt.ops.ij_apply(Hi, Xi, ri, precision=precision))
    assert nl == plan['launches'], (nl, plan)
    assert lib.vt_ij_apply_tf32_workspace_bytes(N, D, split) == plan['ws_bytes']
    ref = -(Hi @ (Xi * ri[:, None]).T)
    assert torch.equal(S, ref), 'D={} {}: {}'.format(D, precision, _diff(S, ref))
    _report('apply {} D={} N={}'.format(precision, D, N), plan)


# ------------------------------------------------------ exact: syrk_weighted ----
@gpu
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('D', APPLY_D)
def test_hessian_exact_over_chunks(vt, lib, sms, D, precision):
    """syrk_weighted (+ l2) over three full chunks and a ragged fourth: the lower-triangle tile walk, parts and
    segments of every chunk accumulated in the FP64 partial tiles, the mirror.  Integer X (|x| <= 8), weights in
    {0, 1/4, 1, 4}: bit for bit equal to torch float64 and exactly symmetric."""
    split = SPLIT[precision]
    N = _big_chunks(hessian_plan(1 << 40, D, split, sms)['chunk'])
    plan = hessian_plan(N, D, split, sms)
    assert plan['chunks'] == 4 and N % plan['chunk'] != 0
    Xi = _ints((N, D), 8, seed=D + 3)
    si = _pow4_weights(N, seed=D + 4)
    H, nl = _launches(vt, lambda: vt.ops.syrk_weighted(Xi, si, l2=3.0, precision=precision))
    assert nl == plan['launches'] + 1, (nl, plan)                   # + the l2 diagonal
    assert lib.vt_syrk_tf32_workspace_bytes(N, D, split) == plan['ws_bytes']
    ref = Xi.T @ (Xi * si[:, None]) + 3.0 * torch.eye(D, dtype=torch.float64, device='cuda')
    assert torch.equal(H, ref), 'D={} {}: {}'.format(D, precision, _diff(H, ref))
    assert torch.equal(H, H.T)
    _report('hessian {} D={} N={}'.format(precision, D, N), plan)


# ------------------------------------------------- componentwise bar, random data ----
RANDOM_SHAPES = [(200, 300, 100), (128, 256, 32), (257, 129, 256), (1, 257, 4), (129, 255, 4097), (255, 1, 8193),
                 'segments']


@gpu
@pytest.mark.parametrize('shape', RANDOM_SHAPES, ids=str)
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('mode', ['KC', 'KS'])
def test_gemm_componentwise_bound(vt, sms, mode, precision, shape):
    """Rows of A and B and columns of A on scales 2^+-10 apart, random alpha and row / column scales: every entry
    within c |alpha rs cs| (|A| |B|^T) of the float64 product, c from the plan's longest segment."""
    split = SPLIT[precision]
    M, N, K = shape if shape != 'segments' else _segment_shape(split, sms) + (8193,)
    plan = gemm_plan(M, N, K, split, sms)
    g = _gen(11)
    A = _rnd(M, K, seed=12) * torch.exp2(torch.randint(-10, 11, (M, 1), generator=g, device='cuda').double())
    A = A * torch.exp2(torch.randint(-10, 11, (1, K), generator=g, device='cuda').double())
    B = _rnd(N, K, seed=13) * torch.exp2(torch.randint(-10, 11, (N, 1), generator=g, device='cuda').double())
    rs, cs = _rnd(M, seed=14), _rnd(N, seed=15)
    if mode == 'KS':
        A, B = A.T.contiguous(), B.T.contiguous()
    out = vt.ops.tf32_gemm(A, B, mode, mode, alpha=-0.75, precision=precision, rowscale=rs, colscale=cs)
    scale = 0.75 * rs.abs()[:, None] * cs.abs()[None, :]
    err = (out - (-0.75) * rs[:, None] * cs[None, :] * _product(A, B, mode)).abs()
    acc = scale * _product(A.abs(), B.abs(), mode)
    c = bar(plan['seg_len'], split, K)
    worst = float((err / acc).max())
    assert bool((err <= c * acc).all()), '{} {} {}: worst err / (|A||B|) {:.3e} above the bar {:.3e}'.format(
        mode, precision, (M, N, K), worst, c)
    print('{} {} {}: worst err / (|A||B|) {:.3e}, bar {:.3e}'.format(mode, precision, (M, N, K), worst, c))


@gpu
@pytest.mark.parametrize('precision', PRECISIONS)
def test_apply_and_hessian_componentwise_bound(vt, sms, precision):
    """ij_apply and syrk_weighted on random data with features on scales 2^+-8 apart: entry by entry within the bar
    of their GEMMs (K = D for the apply, the observations for the Hessian)."""
    split = SPLIT[precision]
    N, D = 20011, 300
    X = _rnd(N, D, seed=20) * torch.exp2(torch.randint(-8, 9, (1, D), generator=_gen(21), device='cuda').double())
    Hinv = _rnd(D, D, seed=22)
    r = _rnd(N, seed=23)
    s = torch.rand(N, generator=_gen(24), device='cuda', dtype=torch.float64)
    S = vt.ops.ij_apply(Hinv, X, r, precision=precision)
    c = bar(apply_plan(N, D, split, sms)['seg_len'], split, D)
    acc = Hinv.abs() @ (X.abs() * r.abs()[:, None]).T
    assert bool(((S + Hinv @ (X * r[:, None]).T).abs() <= c * acc).all()), 'apply'
    H = vt.ops.syrk_weighted(X, s, precision=precision)
    c = bar(hessian_plan(N, D, split, sms)['seg_len'], split, N)
    acc = X.abs().T @ (X.abs() * s[:, None])
    assert bool(((H - X.T @ (X * s[:, None])).abs() <= c * acc).all()), 'hessian'


# ------------------------------------------------------------------ layouts ----
def _x_layouts(X):
    """{name: a view with the values of X}: padded rows (ld = D + 1, D + 2; NaN padding) and a base 8 bytes off the
    16-byte alignment with an even ld (the converter's scalar path)."""
    N, D = X.shape
    out = {}
    for pad in (1, 2):
        big = torch.full((N, D + pad), float('nan'), dtype=torch.float64, device='cuda')
        big[:, :D] = X
        out['ld+{}'.format(pad)] = big[:, :D]
    ld = D + (1 if D % 2 else 2)
    flat = torch.full((N * ld + 1,), float('nan'), dtype=torch.float64, device='cuda')
    v = flat[1:].view(N, ld)[:, :D]
    v.copy_(X)
    assert v.data_ptr() % 16 == 8 and v.stride(0) % 2 == 0
    out['base+8'] = v
    return out


def _out_blocks(rows, cols):
    """(pad, offset, what) for output blocks of a wider sentinel buffer: ldc not a multiple of 4; ldc a multiple of
    4 with a base 8 bytes off 32-byte alignment (both the scalar epilogue); and an aligned block (vector stores)."""
    p1 = next(p for p in range(1, 5) if (cols + p) % 4 != 0)
    p2 = next(p for p in range(1, 5) if (cols + p) % 4 == 0)
    return [(p1, 0, 'ldc % 4 != 0'), (p2, 1, 'base % 32 == 8'), (p2 + 4, 4, 'aligned')]


@gpu
@pytest.mark.parametrize('D', [77, 256])
@pytest.mark.parametrize('precision', PRECISIONS)
def test_layouts_are_bit_identical(vt, precision, D):
    """ij_apply and syrk_weighted with X and Hinv as padded or offset views and the output as a block of a wider
    sentinel-filled buffer: bit-identical to the contiguous run, sentinels untouched."""
    N = 3001
    X = _rnd(N, D, seed=30)
    Hinv = torch.eye(D, dtype=torch.float64, device='cuda') + _rnd(D, D, seed=31) / math.sqrt(D)
    r, s = _rnd(N, seed=32), torch.rand(N, generator=_gen(33), device='cuda', dtype=torch.float64)
    S0 = vt.ops.ij_apply(Hinv, X, r, precision=precision)
    H0 = vt.ops.syrk_weighted(X, s, l2=0.5, precision=precision)
    for lay, Xv in _x_layouts(X).items():
        S = vt.ops.ij_apply(Hinv, Xv, r, precision=precision)
        assert torch.equal(S, S0), 'apply, X {}: {}'.format(lay, _diff(S, S0))
        H = vt.ops.syrk_weighted(Xv, s, l2=0.5, precision=precision)
        assert torch.equal(H, H0), 'hessian, X {}: {}'.format(lay, _diff(H, H0))
    bigH = torch.full((D, D + 3), float('nan'), dtype=torch.float64, device='cuda')
    bigH[:, 1:1 + D] = Hinv
    S = vt.ops.ij_apply(bigH[:, 1:1 + D], X, r, precision=precision)
    assert torch.equal(S, S0), 'apply, Hinv view: {}'.format(_diff(S, S0))
    for rows, cols, run, ref in ((D, N, lambda o: vt.ops.ij_apply(Hinv, X, r, out=o, precision=precision), S0),
                                 (D, D, lambda o: vt.ops.syrk_weighted(X, s, l2=0.5, out=o, precision=precision), H0)):
        for pad, off, what in _out_blocks(rows, cols):
            big, o = _sentinel_block(rows, cols, pad, off)
            vec = o.stride(0) % 4 == 0 and o.data_ptr() % 32 == 0
            assert vec == (what == 'aligned'), what
            run(o)
            assert torch.equal(o, ref), 'out block ({}), {} x {}: {}'.format(what, rows, cols, _diff(o, ref))
            assert _sentinels_intact(big, (off, off + cols)), 'out block ({}): sentinels overwritten'.format(what)


# ---------------------------------------------------------- non-finite inputs ----
def _same_poison(out, ref, what):
    fo, fr = torch.isfinite(out), torch.isfinite(ref)
    assert bool((~fr).any()), '{}: the FP64 engine shows no non-finite entry'.format(what)
    assert torch.equal(fo, fr), '{}: {} entries finite in one engine only ({} non-finite in FP64, {} here)'.format(
        what, int((fo != fr).sum()), int((~fr).sum()), int((~fo).sum()))


@gpu
@pytest.mark.parametrize('precision', PRECISIONS)
def test_non_finite_inputs_poison_like_fp64(vt, precision):
    """A NaN or +-Inf in X, H^{-1} or the residuals, and a NaN or Inf weight, poison the same entries as in the FP64
    engine (isfinite patterns: Inf - Inf in the lo split gives NaN where FP64 gives +-Inf)."""
    N, D = 5003, 200
    X = _rnd(N, D, seed=40)
    X[17, 5], X[4000, 150], X[2222, 0] = float('nan'), float('inf'), float('-inf')
    Hinv = torch.eye(D, dtype=torch.float64, device='cuda') + _rnd(D, D, seed=41) / math.sqrt(D)
    r = _rnd(N, seed=42)
    s = torch.rand(N, generator=_gen(43), device='cuda', dtype=torch.float64)
    Xf = _rnd(N, D, seed=44)
    Hn = Hinv.clone()
    Hn[33, 7] = float('nan')
    rn = r.clone()
    rn[1234] = float('nan')
    for name, (Hv, Xv, rv) in (('X', (Hinv, X, r)), ('Hinv', (Hn, Xf, r)), ('resid', (Hinv, Xf, rn))):
        _same_poison(vt.ops.ij_apply(Hv, Xv, rv, precision=precision), vt.ops.ij_apply(Hv, Xv, rv, precision='f64'),
                     'apply, non-finite ' + name)
    _same_poison(vt.ops.syrk_weighted(X, s, precision=precision), vt.ops.syrk_weighted(X, s, precision='f64'),
                 'hessian, non-finite X')
    for bad in (float('nan'), float('inf')):
        sb = s.clone()
        sb[99] = bad
        _same_poison(vt.ops.syrk_weighted(Xf, sb, precision=precision),
                     vt.ops.syrk_weighted(Xf, sb, precision='f64'), 'hessian, weight {}'.format(bad))
        hi, _ = vt.ops.tf32_convert(Xf, rowscale=sb, sqrt_scale=True, split=SPLIT[precision])
        assert not bool(torch.isfinite(hi[99, :D]).any()) and bool(torch.isfinite(hi[100, :D]).all())
