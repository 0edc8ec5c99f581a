"""Tensor-level wrappers over the C ABI.

Each function takes float64 CUDA tensors, sizes the workspace the library asks
for, launches on the current stream and returns tensors.  No arithmetic on the
hot path happens in torch: torch is the allocator and the stream provider.
"""
import ctypes
import os

import numpy as np
import torch

from . import _cabi
from ._cabi import check, ptr, stream

_workspaces = {}
# balanced base-256 digits per operand of the 'f64_ozaki' engine: 7 -> 54 bits of the row scale (FP64 DMMA results
# reproduced to ~1e-14 of max|C|, 28 digit products); 6 -> 46 bits (~1e-12: on the edge of the parity floor, 21
# products); 5 -> 38 bits (VT_OZAKI_SLICES=5|6|7 overrides)
OZAKI_SLICES = int(os.environ.get('VT_OZAKI_SLICES', '7'))
if OZAKI_SLICES not in (5, 6, 7):
    raise ValueError('VT_OZAKI_SLICES must be 5, 6 or 7')


def _ws(key, nbytes, device):
    """Grow-only per-device scratch buffer, keyed by purpose."""
    nbytes = int(nbytes)
    if nbytes == 0:
        return None, 0
    k = (key, device.index)
    buf = _workspaces.get(k)
    if buf is None or buf.numel() * 8 < nbytes:
        buf = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=device)
        _workspaces[k] = buf
    return buf, buf.numel() * 8


def free_workspaces():
    _workspaces.clear()


def _f64(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.float64:
        raise TypeError('{} must be a float64 CUDA tensor'.format(name))
    return t


def _mat(t, name):
    _f64(t, name)
    if t.dim() != 2 or (t.stride(1) != 1 and t.shape[1] > 1):       # (the stride of a length-1 dimension is arbitrary)
        raise ValueError('{} must be a row-major 2-d tensor (unit stride in the last dimension)'.format(name))
    return t


def _vec_opt(t, name, n=None):
    """Optional per-row / per-column vector: packed float64 on the device (None stays None)."""
    if t is None:
        return None
    t = _f64(t, name).reshape(-1).contiguous()
    if n is not None and t.numel() < n:
        raise ValueError('{} has {} entries, expected {}'.format(name, t.numel(), n))
    return t


def _ld(t):
    # leading dimension of a row-major matrix (handles single-row views)
    return t.stride(0) if t.shape[0] > 1 else max(t.shape[1], t.stride(0))


def device_info():
    lib = _cabi.require_cuda()
    sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    check(lib.vt_device_info(ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)))
    return dict(sm_count=sm.value, cc=(ma.value, mi.value))


def launch_count():
    return int(_cabi.load().vt_launch_count())


def fp64_peak_probe(seconds=0.3):
    lib = _cabi.require_cuda()
    tf = ctypes.c_double()
    check(lib.vt_fp64_peak_probe(float(seconds), ctypes.byref(tf), stream()))
    return tf.value


def i8_peak_probe(seconds=1.0, n_tile=256):
    """{'tops': dense INT8 TOP/s of a bare tcgen05.mma.kind::i8 loop of 128 x n_tile x 32 instructions run for
    about `seconds`, 'clocks_per_mma': SM clocks per instruction} - the denominator of the slicing engine's roofline."""
    lib = _cabi.require_cuda()
    tops, clk = ctypes.c_double(), ctypes.c_double()
    check(lib.vt_i8_peak_probe(float(seconds), int(n_tile), ctypes.byref(tops), ctypes.byref(clk), stream()))
    return {'tops': tops.value, 'clocks_per_mma': clk.value, 'n_tile': int(n_tile), 'seconds': float(seconds)}


# ------------------------------------------------------------------ GEMM ----
def gemm(A, B, amode='KC', bmode='KC', alpha=1.0, beta=0.0, out=None, M=None, N=None, K=None,
         kscale=None, colscale=None, rowscale=None, lower=False, mirror=False, tile=0):
    """out(m,n) = alpha * rs[m] cs[n] sum_k ks[k] A(m,k) B(n,k) + beta * out.

    ``KC``: the tensor is (rows, K); ``KS``: the tensor is (K, rows).  ``tile``:
    CTA tile edge (128 or 64), 0 = chosen from the shape."""
    lib = _cabi.require_cuda()
    _mat(A, 'A'); _mat(B, 'B')
    am = _cabi.OP_KC if amode == 'KC' else _cabi.OP_KS
    bm = _cabi.OP_KC if bmode == 'KC' else _cabi.OP_KS
    m, ka = (A.shape if am == _cabi.OP_KC else A.shape[::-1])
    n, kb = (B.shape if bm == _cabi.OP_KC else B.shape[::-1])
    if K is None:
        if ka != kb:
            raise ValueError('gemm: inner dimensions differ ({} vs {})'.format(ka, kb))
        K = ka
    M = m if M is None else M
    N = n if N is None else N
    if not (0 <= M <= m and 0 <= N <= n and 0 <= K <= min(ka, kb)):
        raise ValueError('gemm: M, N, K = {}, {}, {} exceed the operands ({} x {} and {} x {})'.format(M, N, K, m, ka, n, kb))
    kscale, colscale, rowscale = (_vec_opt(kscale, 'kscale', K), _vec_opt(colscale, 'colscale', N),
                                  _vec_opt(rowscale, 'rowscale', M))
    if out is None:
        if beta != 0.0:
            raise ValueError('gemm: beta != 0 needs `out`')
        out = torch.empty((M, N), dtype=torch.float64, device=A.device)
    _mat(out, 'out')
    wsb = lib.vt_dgemm_workspace_bytes(M, N, K, int(lower), int(tile))
    ws, wsb = _ws('gemm', wsb, A.device)
    check(lib.vt_dgemm(M, N, K, float(alpha), ptr(A), _ld(A), am, ptr(B), _ld(B), bm, float(beta), ptr(out),
                       _ld(out), ptr(kscale), ptr(colscale), ptr(rowscale), int(lower), int(mirror), int(tile), ptr(ws), wsb,
                       stream()))
    return out


# ------------------------------------------------- TF32 engine (optional) ----
def tf32_convert(X, rowscale=None, sqrt_scale=False, split=1):
    """(hi, lo | None): TF32-rounded FP32 copies of a float64 matrix, leading
    dimension padded to a multiple of 4 (zero filled)."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    rows, cols = X.shape
    ld = (cols + 3) // 4 * 4
    hi = torch.empty((rows, ld), dtype=torch.float32, device=X.device)
    lo = torch.empty_like(hi) if split == 3 else None
    check(lib.vt_tf32_convert(ptr(X), _ld(X), rows, cols, ptr(rowscale), int(bool(sqrt_scale)), ptr(hi), ptr(lo), ld,
                              stream()))
    return hi, lo


def tf32_gemm(A, B, amode='KC', bmode='KC', alpha=1.0, precision='tf32', colscale=None, rowscale=None, out=None):
    """out (FP64) = alpha * rs[m] cs[n] sum_k A(m,k) B(n,k) on tcgen05.mma.kind::tf32
    (FP32 accumulation in TMEM).  A and B are float64 CUDA matrices (KC: (rows, K);
    KS: (K, rows)) that are rounded to TF32 (hi [+ lo]) here."""
    lib = _cabi.require_cuda()
    split = _split(precision)
    if not split:
        raise ValueError("tf32_gemm: precision must be 'tf32' or 'tf32x3'")
    if amode != bmode:
        raise ValueError('tf32_gemm: both operands must use the same mode')
    mode = _cabi.OP_KC if amode == 'KC' else _cabi.OP_KS
    Ah, Al = tf32_convert(A, split=split)
    Bh, Bl = tf32_convert(B, split=split)
    (M, K) = A.shape if mode == _cabi.OP_KC else A.shape[::-1]
    (N, Kb) = B.shape if mode == _cabi.OP_KC else B.shape[::-1]
    if K != Kb:
        raise ValueError('tf32_gemm: inner dimensions differ ({} vs {})'.format(K, Kb))
    if out is None:
        out = torch.empty((M, N), dtype=torch.float64, device=A.device)
    ws, wsb = _ws('tf32_gemm', lib.vt_tf32_gemm_workspace_bytes(M, N, K, split), A.device)
    check(lib.vt_tf32_gemm(M, N, K, float(alpha), ptr(Ah), ptr(Al), Ah.stride(0), mode, ptr(Bh), ptr(Bl), Bh.stride(0),
                           mode, ptr(out), _ld(out), ptr(colscale), ptr(rowscale), ptr(ws), wsb, stream()))
    return out


# ------------------------------------- INT8 error-free slicing (optional) ----
def ozaki_slice(X, nslices=OZAKI_SLICES, fold=None, integer_variant=False):
    """(digits (nslices, rows, ld) int8, scale (rows,) float64) of a float64 matrix:
    X[r, k] = scale[r] * 2^-6 sum_s digits[s, r, k] 2^{-8 s} up to scale[r] 2^{-(8 nslices - 1)}
    (``fold`` multiplies the returned scale row by row).  ``integer_variant``: the
    integer-only instruction sequence that the GEMM kernel's converter warps run
    (same digits; rows of at most 1024 elements)."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    rows, cols = X.shape
    ld = (cols + 15) // 16 * 16
    out = torch.empty((nslices, rows, ld), dtype=torch.int8, device=X.device)
    scale = torch.empty(rows, dtype=torch.float64, device=X.device)
    fn = lib.vt_ozaki_slice_int if integer_variant else lib.vt_ozaki_slice
    check(fn(ptr(X), _ld(X), rows, cols, ptr(out), ld, rows * ld, nslices, ptr(scale), ptr(fold), stream()))
    return out, scale


def ozaki_slice_t(X, sq, nslices=OZAKI_SLICES, integer_variant=False):
    """The Hessian's operand: (digits (nslices, cols, ld) int8, scale (cols,) float64) of
    sq[n] * X[n, i] (sq None: of X[n, i]), transposed (observations contiguous), one power-of-two scale per feature."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    rows, cols = X.shape
    if sq is not None:
        _f64(sq, 'sq')
        if sq.numel() != rows:
            raise ValueError('sq must have one entry per row of X')
    W = X if sq is None else X * sq[:, None]
    cmax = W.abs().amax(dim=0).contiguous().view(torch.int64)                    # bit patterns of the maxima
    ld = (rows + 15) // 16 * 16
    out = torch.zeros((nslices, cols, ld), dtype=torch.int8, device=X.device)
    scale = torch.empty(cols, dtype=torch.float64, device=X.device)
    check(lib.vt_ozaki_slice_t(ptr(X), _ld(X), rows, cols, ptr(sq), ptr(cmax), ptr(out), ld, cols * ld, nslices,
                               ptr(scale), 1 if integer_variant else 0, stream()))
    return out, scale


def ozaki_gemm(A, B, alpha=1.0, nslices=OZAKI_SLICES, out=None):
    """out = alpha * A @ B.T for float64 A (M, K), B (N, K) on the INT8 tensor
    cores (tcgen05.mma.kind::i8) with FP64-grade accuracy."""
    lib = _cabi.require_cuda()
    (M, K), (N, Kb) = A.shape, B.shape
    if K != Kb:
        raise ValueError('ozaki_gemm: inner dimensions differ ({} vs {})'.format(K, Kb))
    As, sa = ozaki_slice(A, nslices)
    Bs, sb = ozaki_slice(B, nslices)
    if out is None:
        out = torch.empty((M, N), dtype=torch.float64, device=A.device)
    check(lib.vt_ozaki_gemm(M, N, K, ptr(As), As.stride(1), As.stride(0), ptr(Bs), Bs.stride(1), Bs.stride(0), nslices,
                            float(alpha), ptr(sa), ptr(sb), ptr(out), _ld(out), stream()))
    return out


# ------------------------------------------------------- Hessian assembly ----
PRECISIONS = {'auto': 0, 'f64': 0, 'tf32': 1, 'tf32x3': 3, 'f64_ozaki': 0}
# 'auto' (the default of the objective classes) picks between the two FP64-grade engines, which are held to the
# same parity bar: the INT8 error-free-slicing engine once the contraction is large enough to amortise its slicing
# passes and fill its 128 x 64 tiles (N D^2 >= 1e11, e.g. N >= 1e5 at D = 1024), the FP64 DMMA engine otherwise
# (and whenever the weights of the Hessian are not all non-negative: the slicing engine factors out sqrt(s)).
AUTO_OZAKI_MIN_WORK = 1e11
AUTO_OZAKI_MIN_DIM = 512          # narrower outputs cover too few 128 x 64 tiles (measured at D = 320: no faster than DMMA)


def _split(precision):
    """0 for the FP64-grade engines, else the TF32 split (1 | 3) of the tcgen05 engine."""
    if precision not in PRECISIONS:
        raise ValueError("precision must be 'auto', 'f64', 'f64_ozaki', 'tf32' or 'tf32x3', not {!r}".format(precision))
    return PRECISIONS[precision]


def resolve_precision(precision, N, D, weights=None):
    """The engine 'auto' stands for at this shape ('f64_ozaki' | 'f64'); any other value is returned as is."""
    _split(precision)
    if precision != 'auto':
        return precision
    if D < AUTO_OZAKI_MIN_DIM or float(N) * D * D < AUTO_OZAKI_MIN_WORK:
        return 'f64'
    if weights is not None and bool((weights < 0).any()):
        return 'f64'
    return 'f64_ozaki'


def syrk_weighted(X, s=None, l2=0.0, out=None, precision='f64', colmax=None):
    """H = X^T diag(s) X + l2 I  (FP64 DMMA, deterministic split-K; or, for
    s >= 0, the INT8 error-free-slicing engine 'f64_ozaki' (FP64-grade) or the
    optional reduced-precision TF32 / TF32x3 tcgen05 path).  ``colmax=(sq, cmax)``
    from ``glm_stats(..., want_colmax=True)`` spares the INT8 engine its own sweep
    over X for the per-feature scales."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, D = X.shape
    precision = resolve_precision(precision, N, D, s)
    split = _split(precision)
    if s is None and not split and precision != 'f64_ozaki':      # (the INT8 engine takes "unweighted" as such)
        s = torch.ones(N, dtype=torch.float64, device=X.device)
    if s is not None:
        _f64(s, 's')
        if s.numel() != N:
            raise ValueError('s must have one entry per row of X')
    if out is None:
        out = torch.empty((D, D), dtype=torch.float64, device=X.device)
    if (split or precision == 'f64_ozaki') and s is not None and bool((s < 0).any()):
        raise ValueError("syrk_weighted: precision {!r} needs non-negative weights (it factors out sqrt(s)); "
                         "use precision='f64'".format(precision))
    if precision == 'f64_ozaki':
        ws, wsb = _ws('syrk_ozaki', lib.vt_syrk_ozaki_workspace_bytes(N, D, OZAKI_SLICES), X.device)
        sq, cmax = colmax if (colmax is not None and s is not None) else (None, None)
        if sq is not None and (sq.numel() != N or cmax.numel() != D or cmax.dtype != torch.int64):
            raise ValueError('colmax must be (sq (N,) float64, cmax (D,) int64) from glm_stats(want_colmax=True)')
        check(lib.vt_syrk_ozaki(ptr(X), _ld(X), N, D, ptr(s), float(l2), ptr(out), _ld(out), OZAKI_SLICES, ptr(sq),
                                ptr(cmax), ptr(ws), wsb, stream()))
        return out
    if split:
        ws, wsb = _ws('syrk_tf32', lib.vt_syrk_tf32_workspace_bytes(N, D, split), X.device)
        check(lib.vt_syrk_tf32(ptr(X), _ld(X), N, D, ptr(s), float(l2), ptr(out), _ld(out), split, ptr(ws), wsb,
                               stream()))
        return out
    wsb = lib.vt_syrk_workspace_bytes(N, D)
    ws, wsb = _ws('syrk', wsb, X.device)
    check(lib.vt_syrk_weighted(ptr(X), _ld(X), N, D, ptr(s), float(l2), ptr(out), _ld(out), ptr(ws), wsb, stream()))
    return out


# ------------------------------------------------------------- GLM passes ----
COLMAX_MAX_DIM = 2048         # the statistics pass can carry the column maxima up to this width


def glm_stats(X, theta, y, w=None, family='logistic', l2=0.0, want_grad=True, want_z=True, out=None, want_colmax=False):
    """One pass over X: z = X theta, resid = b'(z) - y, s = w b''(z) and
    (optionally) grad = X^T (w resid) + l2 theta.  ``out=(z, resid, s)`` writes the
    per-observation outputs into existing (slices of) tensors.  ``want_colmax`` (D <= 2048):
    the same pass also yields ``(sq, cmax)`` = sqrt(s) and the bit patterns of
    max_n sqrt(s_n) |x_nc| - the per-feature scales ``syrk_weighted(precision='f64_ozaki')``
    otherwise sweeps X for - returned as a fifth value."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, D = X.shape
    dev = X.device
    if out is not None:
        z, resid, s = out
    else:
        z = torch.empty(N, dtype=torch.float64, device=dev) if want_z else None
        resid = torch.empty(N, dtype=torch.float64, device=dev)
        s = torch.empty(N, dtype=torch.float64, device=dev)
    grad = torch.empty(D, dtype=torch.float64, device=dev) if want_grad else None
    if want_colmax:
        if D > COLMAX_MAX_DIM:
            raise ValueError('glm_stats: want_colmax needs D <= {}'.format(COLMAX_MAX_DIM))
        sq = torch.empty(N, dtype=torch.float64, device=dev)
        cmax = torch.empty(D, dtype=torch.int64, device=dev)
        ws, wsb = _ws('glm', 2 * lib.vt_glm_workspace_bytes(D), dev)
        check(lib.vt_glm_stats_colmax(ptr(X), _ld(X), N, D, ptr(_f64(theta, 'theta').contiguous()), ptr(_f64(y, 'y')),
                                      ptr(_vec_opt(w, 'w', N)), _cabi.GLM_FAMILIES[family], ptr(z), ptr(resid), ptr(s),
                                      ptr(grad), float(l2), ptr(sq), ptr(cmax), ptr(ws), wsb, stream()))
        return z, resid, s, grad, (sq, cmax)
    ws, wsb = _ws('glm', lib.vt_glm_workspace_bytes(D), dev)
    check(lib.vt_glm_stats(ptr(X), _ld(X), N, D, ptr(_f64(theta, 'theta').contiguous()), ptr(_f64(y, 'y')),
                           ptr(_vec_opt(w, 'w', N)), _cabi.GLM_FAMILIES[family], ptr(z), ptr(resid), ptr(s), ptr(grad), float(l2),
                           ptr(ws), wsb, stream()))
    return z, resid, s, grad


def glm_hvp(X, s, v, ridge=0.0, out=None):
    """out = X^T (s .* (X v)) + ridge v  - one fused pass over X."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, D = X.shape
    if out is None:
        out = torch.empty(D, dtype=torch.float64, device=X.device)
    ws, wsb = _ws('glm', lib.vt_glm_workspace_bytes(D), X.device)
    check(lib.vt_glm_hvp(ptr(X), _ld(X), N, D, ptr(_f64(s, 's')), ptr(_f64(v, 'v').contiguous()), float(ridge),
                         ptr(out), ptr(ws), wsb, stream()))
    return out


HVP_MULTI_MAX = 4            # directions per pass of the fused kernel (XT_MAXQ)
HVP_GEMM_MIN = 24            # from this many directions on, two GEMMs (X read twice) beat ceil(K / 4) fused passes


def glm_hvp_multi(X, s, V, ridge=0.0):
    """out (K, D) = V X^T diag(s) X + ridge V for the K rows of V.  Up to four directions share ONE fused pass over X
    (vt_glm_hvp_multi); many directions go through the FP64 GEMM engine: T = diag(s) X V^T (N, K) and out = T^T X,
    two reads of X whatever K is."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    V = _mat(_f64(V, 'V').contiguous(), 'V')
    N, D = X.shape
    K = V.shape[0]
    if V.shape[1] != D:
        raise ValueError('V must have shape (K, D)')
    s = _f64(s, 's').contiguous()
    if K >= HVP_GEMM_MIN or (K > 1 and D > 2048):
        T = gemm(X, V, 'KC', 'KC', rowscale=s)                  # (N, K) = diag(s) X V^T
        out = gemm(T, X, 'KS', 'KS')                            # (K, D) = T^T X
        if ridge != 0.0:
            out.add_(V, alpha=float(ridge))
        return out
    out = torch.empty((K, D), dtype=torch.float64, device=X.device)
    ws, wsb = _ws('glm_multi', lib.vt_glm_hvp_multi_workspace_bytes(D, min(K, HVP_MULTI_MAX)), X.device)
    for k0 in range(0, K, HVP_MULTI_MAX):
        q = min(HVP_MULTI_MAX, K - k0)
        check(lib.vt_glm_hvp_multi(ptr(X), _ld(X), N, D, ptr(s), ptr(V[k0:k0 + q]), q, float(ridge), ptr(out[k0:k0 + q]),
                                   ptr(ws), wsb, stream()))
    return out


def glm_dirderiv(X, z, dirs, w=None, family='logistic', out=None):
    """out = X^T ( w .* b^{(q+1)}(z) .* prod_j X dirs[j] ) for dirs of shape (q, D)."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, D = X.shape
    dirs = _f64(dirs, 'dirs').contiguous()
    if dirs.dim() != 2 or dirs.shape[1] != D:
        raise ValueError('dirs must have shape (q, D)')
    if out is None:
        out = torch.empty(D, dtype=torch.float64, device=X.device)
    ws, wsb = _ws('glm', lib.vt_glm_dirderiv_workspace_bytes(N, D), X.device)
    check(lib.vt_glm_dirderiv(ptr(X), _ld(X), N, D, ptr(_f64(z, 'z')), ptr(_vec_opt(w, 'w', N)), _cabi.GLM_FAMILIES[family],
                              ptr(dirs), dirs.shape[0], ptr(out), ptr(ws), wsb, stream()))
    return out


def glm_influence_max_directions(D):
    """Directions one pass of ``glm_influence`` takes at width D: 8 up to 2048, 2 up to 4096, 1 up to 8192, else 0."""
    return int(_cabi.load().vt_glm_influence_max_directions(int(D)))


def glm_influence(X, c, V, alpha=1.0, out=None):
    """out (K, N) = alpha * c[None, :] * (V @ X.T): row k holds alpha c_n (x_n . V[k]) for every row n of X.  One pass
    over X (vt_glm_influence) per glm_influence_max_directions(D) rows of V; nothing of size N x D is formed.  ``out``
    may be a row-major view with a leading dimension >= N."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, D = X.shape
    V = _f64(V, 'V')
    if V.dim() != 2 or V.shape[1] != D or V.shape[0] < 1:
        raise ValueError('V must have shape (K, D) with K >= 1 and D = {}, got {}'.format(D, tuple(V.shape)))
    K = V.shape[0]
    qmax = glm_influence_max_directions(D)
    if qmax == 0:
        raise ValueError('glm_influence: D = {} is not supported (D <= 8192)'.format(D))
    c = _f64(c, 'c').reshape(-1).contiguous()
    if c.numel() != N:
        raise ValueError('c must have one entry per row of X ({}), got {}'.format(N, c.numel()))
    V = V.contiguous()
    if out is None:
        out = torch.empty((K, N), dtype=torch.float64, device=X.device)
    _mat(out, 'out')
    if tuple(out.shape) != (K, N):
        raise ValueError('out must have shape ({}, {}), got {}'.format(K, N, tuple(out.shape)))
    for k0 in range(0, K, qmax):
        q = min(qmax, K - k0)
        check(lib.vt_glm_influence(ptr(X), _ld(X), N, D, ptr(c), ptr(V[k0:k0 + q]), q, float(alpha), ptr(out[k0:k0 + q]),
                                   _ld(out), stream()))
    return out


# --------------------------------------------------------------- Cholesky ----
class CholeskyFactor:
    """Lower Cholesky factor of a dense SPD matrix, resident on the GPU.

    The analogue of the ``(c, lower)`` tuple of ``scipy.linalg.cho_factor``
    that the reference stores (``solver_lib.py:26-27``)."""

    def __init__(self, L, dinv):
        self.L = L
        self.dinv = dinv
        self.dim = L.shape[0]

    def solve(self, B, overwrite=False):
        """(L L^T)^{-1} B for B of shape (D,) or (D, K); float64 CUDA tensor."""
        lib = _cabi.require_cuda()
        _f64(B, 'B')
        vec = B.dim() == 1
        if B.shape[0] != self.dim or B.dim() > 2:
            raise ValueError('right-hand side has shape {}, expected ({},) or ({}, K)'.format(
                tuple(B.shape), self.dim, self.dim))
        X = B.reshape(self.dim, -1)
        if not (overwrite and X.is_contiguous()):
            X = X.contiguous()
            if X.data_ptr() == B.data_ptr():
                X = X.clone()
        check(lib.vt_potrs(ptr(self.L), _ld(self.L), self.dim, ptr(self.dinv), ptr(X), _ld(X), X.shape[1], stream()))
        return X.reshape(-1) if vec else X

    def inverse(self):
        eye = torch.eye(self.dim, dtype=torch.float64, device=self.L.device)
        return self.solve(eye, overwrite=True)

    def cond_lower_bound(self):
        """(max_i L_ii / min_i L_ii)^2 <= kappa_2(L L^T): a free lower bound on the condition number of the
        factorised matrix (one D-element reduction), used to decide whether the explicit inverse is safe."""
        d = torch.diagonal(self.L)
        return float((d.max() / d.min()) ** 2)


def potrf(H, overwrite=False, check_pd=True):
    """Cholesky-factor a dense symmetric positive-definite matrix on the GPU.
    Raises ``numpy.linalg.LinAlgError`` like ``cho_factor`` if H is not PD."""
    lib = _cabi.require_cuda()
    _f64(H, 'H')
    if H.dim() != 2 or H.shape[0] != H.shape[1]:
        raise ValueError('expected a square matrix')
    D = H.shape[0]
    if overwrite and H.is_contiguous():
        L = H
    else:
        L = H.contiguous()
        if L.data_ptr() == H.data_ptr():
            L = L.clone()
    dinv = torch.empty(lib.vt_potrf_dinv_doubles(D), dtype=torch.float64, device=H.device)
    info = torch.zeros(1, dtype=torch.int32, device=H.device)
    check(lib.vt_potrf(ptr(L), _ld(L), D, ptr(dinv), ctypes.c_void_p(info.data_ptr()), stream()))
    if check_pd:
        i = int(info.item())
        if i != 0:
            raise np.linalg.LinAlgError(
                '{}-th leading minor of the array is not positive definite'.format(i))
    return CholeskyFactor(L, dinv)


# ------------------------------------------------------------- IJ apply ----
def ij_apply(Hinv, X, resid, out=None, precision='f64'):
    """S (D, N) = -Hinv @ (resid[:, None] * X).T without materialising the
    cross-Hessian.  ``precision``: 'f64' (DMMA engine), 'f64_ozaki' (FP64-grade on the
    INT8 tensor cores), 'auto' (one of those two by size) or the optional
    reduced-precision 'tf32' / 'tf32x3' tcgen05 path."""
    lib = _cabi.require_cuda()
    _mat(Hinv, 'Hinv'); _mat(X, 'X')
    N, D = X.shape
    if out is None:
        out = torch.empty((D, N), dtype=torch.float64, device=X.device)
    precision = resolve_precision(precision, N, D)
    split = _split(precision)
    if precision == 'f64_ozaki':
        ws, wsb = _ws('ij_ozaki', lib.vt_ij_apply_ozaki_workspace_bytes(N, D, OZAKI_SLICES), X.device)
        check(lib.vt_ij_apply_ozaki(ptr(Hinv), _ld(Hinv), ptr(X), _ld(X), N, D, ptr(_f64(resid, 'resid')), ptr(out),
                                    _ld(out), OZAKI_SLICES, ptr(ws), wsb, stream()))
        return out
    if split:
        ws, wsb = _ws('ij_tf32', lib.vt_ij_apply_tf32_workspace_bytes(N, D, split), X.device)
        check(lib.vt_ij_apply_tf32(ptr(Hinv), _ld(Hinv), ptr(X), _ld(X), N, D, ptr(_f64(resid, 'resid')), ptr(out),
                                   _ld(out), split, ptr(ws), wsb, stream()))
        return out
    check(lib.vt_ij_apply(ptr(Hinv), _ld(Hinv), ptr(X), _ld(X), N, D, ptr(_f64(resid, 'resid')), ptr(out), _ld(out),
                          stream()))
    return out


def gemv(A, x, alpha=1.0, y0=None, beta=1.0):
    """alpha * A @ x + beta * y0 for a row-major (M, N) matrix with N long."""
    lib = _cabi.require_cuda()
    _mat(A, 'A')
    M, N = A.shape
    y = torch.empty(M, dtype=torch.float64, device=A.device)
    ws, wsb = _ws('gemv', lib.vt_gemv_workspace_bytes(M, N), A.device)
    check(lib.vt_gemv(ptr(A), _ld(A), M, N, ptr(_f64(x, 'x').contiguous()), float(alpha), ptr(y0), float(beta),
                      ptr(y), ptr(ws), wsb, stream()))
    return y


# -------------------------------------------------------------------- CG ----
def cg_batch_init(B, X, R, state, rtol, atol, keep_xr=False):
    """B, X, R: (K, D) rows; state (K, 8).  See include/vittles_b200.h."""
    K, D = B.shape
    check(_cabi.require_cuda().vt_cg_batch_init(D, K, ptr(B), ptr(X), ptr(R), ptr(state), float(rtol), float(atol),
                                                int(bool(keep_xr)), stream()))


def cg_batch_update_p(R, P, state, maxiter, Z=None, minv=None):
    K, D = R.shape
    check(_cabi.require_cuda().vt_cg_batch_update_p(D, K, ptr(R), ptr(Z), ptr(minv), ptr(P), ptr(state), int(maxiter),
                                                    stream()))


def cg_batch_update_xr(P, Q, X, R, state):
    K, D = P.shape
    check(_cabi.require_cuda().vt_cg_batch_update_xr(D, K, ptr(P), ptr(Q), ptr(X), ptr(R), ptr(state), stream()))


# ------------------------------------------------------------- synthetic ----
_IH_STD = float(np.sqrt((65536.0 ** 2 - 1.0) / 3.0))


def synth_design(seed, row0, nrows, ncols, device, scale=None, out=None):
    lib = _cabi.require_cuda()
    if scale is None:
        scale = 1.0 / (_IH_STD * np.sqrt(float(ncols)))
    if out is None:
        out = torch.empty((nrows, ncols), dtype=torch.float64, device=device)
    check(lib.vt_synth_design(ptr(out), _ld(out), int(row0), int(nrows), int(ncols), int(seed), float(scale), stream()))
    return out


def synth_theta(seed, ncols, device):
    return synth_design(seed ^ 0x5EED, 1 << 40, 1, ncols, device, scale=1.0 / _IH_STD)[0]


def synth_bernoulli(seed, row0, z):
    lib = _cabi.require_cuda()
    y = torch.empty_like(z)
    check(lib.vt_synth_bernoulli(ptr(y), ptr(z), int(row0), z.numel(), int(seed), stream()))
    return y


# ------------------------------------------------------- block-arrow path ----
def block_potrf(blocks, check_pd=True):
    """In-place lower Cholesky of (G, M, M) blocks; returns the same tensor."""
    lib = _cabi.require_cuda()
    _f64(blocks, 'blocks')
    if blocks.dim() != 3 or blocks.shape[1] != blocks.shape[2] or not blocks.is_contiguous():
        raise ValueError('blocks must be a contiguous (G, M, M) tensor')
    G, M, _ = blocks.shape
    info = torch.zeros(1, dtype=torch.int32, device=blocks.device)
    check(lib.vt_block_potrf_batched(ptr(blocks), G, M, ctypes.c_void_p(info.data_ptr()), stream()))
    if check_pd:
        i = int(info.item())
        if i != 0:
            raise np.linalg.LinAlgError('block {} of the block-diagonal part is not positive definite'.format(i - 1))
    return blocks


def block_trsm(Lb, C, transpose=False):
    """C[g] <- L[g]^{-1} C[g] (or L[g]^{-T} C[g]) in place, C of shape (G, M, Dg)."""
    lib = _cabi.require_cuda()
    G, M, Dg = C.shape
    if not C.is_contiguous():
        raise ValueError('C must be contiguous')
    fn = lib.vt_block_trsmt_batched if transpose else lib.vt_block_trsm_batched
    check(fn(ptr(_f64(Lb, 'Lb')), ptr(_f64(C, 'C')), G, M, Dg, stream()))
    return C


def block_solve(Lb, b, transpose=False):
    """b[g] <- L[g]^{-1} b[g] (or L[g]^{-T} b[g]) in place, b of shape (G, M)."""
    lib = _cabi.require_cuda()
    G, M = b.shape
    check(lib.vt_block_solve_batched(ptr(_f64(Lb, 'Lb')), ptr(_f64(b, 'b')), G, M, 1 if transpose else 0, stream()))
    return b


def tall_gemv(Z, x, alpha=1.0, y=None, beta=0.0):
    """y = beta*y + alpha * Z @ x for a (R, Dg) matrix with R very long."""
    lib = _cabi.require_cuda()
    _mat(Z, 'Z')
    R, Dg = Z.shape
    if y is None:
        y = torch.empty(R, dtype=torch.float64, device=Z.device)
        beta = 0.0
    check(lib.vt_tall_gemv(ptr(Z), R, Dg, ptr(_f64(x, 'x').contiguous()), float(alpha), ptr(y), float(beta), stream()))
    return y


def tall_colsum(Z, u, alpha=1.0, y0=None, beta=1.0):
    """alpha * Z.T @ u + beta * y0 for a (R, Dg) matrix with R very long."""
    lib = _cabi.require_cuda()
    _mat(Z, 'Z')
    R, Dg = Z.shape
    out = torch.empty(Dg, dtype=torch.float64, device=Z.device)
    ws, wsb = _ws('colsum', lib.vt_tall_colsum_workspace_bytes(Dg), Z.device)
    check(lib.vt_tall_colsum(ptr(Z), R, Dg, ptr(_f64(u, 'u').contiguous()), float(alpha), ptr(y0), float(beta),
                             ptr(out), ptr(ws), wsb, stream()))
    return out


def gmm_blocks(X, m, rho, log_pi, want_blocks=True, want_cross=True):
    """Closed-form pieces of the GMM-VB objective: local Hessian blocks
    (N, K-1, K-1), cross blocks (N, K-1, K*d), responsibilities (N, K), local
    gradient (N, K-1) and per-observation objective terms (N,)."""
    lib = _cabi.require_cuda()
    _mat(X, 'X')
    N, d = X.shape
    K = m.shape[0]
    dev = X.device
    blocks = torch.empty((N, K - 1, K - 1), dtype=torch.float64, device=dev) if want_blocks else None
    cross = torch.empty((N, K - 1, K * d), dtype=torch.float64, device=dev) if want_cross else None
    rmat = torch.empty((N, K), dtype=torch.float64, device=dev)
    grad_rho = torch.empty((N, K - 1), dtype=torch.float64, device=dev)
    obj = torch.empty(N, dtype=torch.float64, device=dev)
    check(lib.vt_gmm_blocks(ptr(X), N, d, K, ptr(_f64(m, 'm').contiguous()), ptr(_f64(rho, 'rho').contiguous()),
                            ptr(_f64(log_pi, 'log_pi').contiguous()), ptr(blocks), ptr(cross), ptr(rmat),
                            ptr(grad_rho), ptr(obj), stream()))
    return dict(blocks=blocks, cross=cross, r=rmat, grad_rho=grad_rho, obj_terms=obj)


# ---------------------------------------------------------- device scoping ----
# The library launches on the CURRENT device's current stream (its workspace queries and SM count use
# cudaGetDevice).  Every wrapper above therefore runs with the device of its first CUDA tensor argument
# (or its `device` argument) made current, so tensors on a non-current GPU are handled on their own device
# and stream instead of faulting or racing.
def _device_of(args, kwargs):
    for a in list(args) + list(kwargs.values()):
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device
        if isinstance(a, CholeskyFactor):
            return a.L.device
        if isinstance(a, torch.device) and a.type == 'cuda':
            return a
        if isinstance(a, (tuple, list)):
            for b in a:
                if isinstance(b, torch.Tensor) and b.is_cuda:
                    return b.device
    return None


def _device_scoped(fn):
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = _device_of(args, kwargs)
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


for _name in ('gemm', 'tf32_convert', 'tf32_gemm', 'ozaki_slice', 'ozaki_gemm', 'syrk_weighted', 'glm_stats', 'glm_hvp',
              'glm_hvp_multi', 'glm_dirderiv', 'glm_influence', 'potrf', 'ij_apply', 'gemv', 'cg_batch_init', 'cg_batch_update_p', 'cg_batch_update_xr',
              'synth_design',
              'synth_theta', 'synth_bernoulli', 'block_potrf', 'block_trsm', 'block_solve', 'tall_gemv', 'tall_colsum',
              'gmm_blocks'):
    globals()[_name] = _device_scoped(globals()[_name])
CholeskyFactor.solve = _device_scoped(CholeskyFactor.solve)
del _name
