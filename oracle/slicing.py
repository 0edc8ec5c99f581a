"""CPU model of the INT8 error-free-slicing engine (``vittles_b200/csrc/ogemm.cu``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).  This is not a restatement of reference code - the
reference computes ``cho_solve(h_chol, cross_hess)`` (``solver_lib.py:29``, ``sensitivity_lib.py:226``) and
``X^T diag(s) X`` through autograd (``sensitivity_lib.py:381-383``) in float64 - but the arithmetic model of the
engine that replaces those two contractions on the INT8 tensor cores, in exact integer arithmetic, so that its error
bound can be checked without a GPU and the CUDA kernels can be checked digit for digit.

    x_rk = sigma_r 2^-6 sum_{s=0..S-1} d_s[r,k] 2^{-8 s} + sigma_r 2^{-(8S-2)} * (|rounding| <= 1/2)
    sum_k a_mk b_nk ~= sigma_m tau_n 2^-12 sum_{s+t < S} 2^{-8 (s+t)} (A_s B_t^T)[m,n]

with BALANCED base-256 digits d_s in [-128, 127] (an int8 digit then carries 8 bits, a sign-magnitude digit 7).
"""
import numpy as np


def _bias(nslices):
    return sum(128 << (8 * p) for p in range(nslices))


def slice_rows(x, nslices):
    """(digits (S, rows, cols) int8, scale (rows,) float64): per-row power-of-two scale 2^e > max_k |x_rk| and the
    balanced base-256 digits of the fixed-point value q = rint(x 2^(8S-2) / scale): with B = sum_p 128 256^p the
    bytes of (q + B) ^ B - the computation of ``fixed4_set_bits`` / ``fixed4_digits`` in ``ogemm.cu``."""
    assert 1 <= nslices <= 7
    x = np.asarray(x, dtype=np.float64)
    m = np.max(np.abs(x), axis=1)
    e = np.where(m > 0, np.frexp(np.where(m > 0, m, 1.0))[1], 0)          # m = f 2^e, f in [0.5, 1)
    scale = np.ldexp(1.0, e)
    t = np.ldexp(x, (8 * nslices - 2 - e)[:, None])                       # exact; |t| <= 2^(8S-2) <= 2^54
    q = np.rint(t).astype(np.int64)                                       # one rounding (ties to even)
    B = _bias(nslices)
    u = (q + B) ^ B
    digits = np.empty((nslices,) + x.shape, dtype=np.int8)
    for s in range(nslices):
        digits[s] = ((u >> (8 * (nslices - 1 - s))) & 255).astype(np.uint8).view(np.int8)
    return digits, scale


def reconstruct(digits, scale):
    """scale_r 2^-6 sum_s d_s 2^{-8 s} in float64 (exact: the value has at most 8S - 1 <= 55 bits only when the top
    digit is small; summed from the least significant digit, at most one rounding for S = 7)."""
    S = digits.shape[0]
    acc = np.zeros(digits.shape[1:], dtype=np.float64)
    for s in range(S - 1, -1, -1):
        acc += digits[s].astype(np.float64) * 2.0 ** (-8 * s - 6)
    return acc * scale[:, None]


def sliced_gemm(a, b, nslices):
    """A @ B.T the way the engine evaluates it: exact INT64 digit products, products with the same s + t share an
    accumulator, the accumulators are combined by Horner's rule in FP64 (``ogemm_kernel`` epilogue), then the
    row / column scales."""
    da, sa = slice_rows(a, nslices)
    db, sb = slice_rows(b, nslices)
    return digits_gemm(da, sa, db, sb)


def digits_gemm(da, sa, db, sb):
    """The engine's product from the digits (S, rows, K) and scales of both operands."""
    nslices = da.shape[0]
    groups = [np.zeros((da.shape[1], db.shape[1]), dtype=np.int64) for _ in range(nslices)]
    for s in range(nslices):
        for t in range(nslices - s):
            groups[s + t] += da[s].astype(np.int64) @ db[t].astype(np.int64).T
    for g in groups:
        assert np.max(np.abs(g)) < 2 ** 31, 'INT32 accumulator bound violated (K too large)'
    # Horner's rule in float64 from the least significant accumulator over PAIRS of accumulators (P_l 256 + P_{l+1}
    # is an exact integer below 2^41), as the epilogue of ``ogemm_kernel`` does it (t * 2^-k is exact, so numpy's
    # multiply-add equals the kernel's fused multiply-add bit for bit)
    def pair(g):
        return (groups[g] * 256 + groups[g + 1]).astype(np.float64)
    if nslices % 2 == 1:
        g = nslices - 3
        val = groups[nslices - 1].astype(np.float64) * (1.0 / 256.0) + pair(g)
    else:
        g = nslices - 2
        val = pair(g)
    for g in range(g - 2, -1, -2):
        val = val * (1.0 / 65536.0) + pair(g)
    return (sa[:, None] * 2.0 ** -20) * sb[None, :] * val


def error_bound(k, nslices):
    """|sliced - exact| <= bound * sigma_m * tau_n: each operand is rounded by <= 2^{-(8S-1)} of its scale (at most
    2 K 2^{-(8S-1)} for the two first-order terms) and the dropped digit pairs s + t >= S contribute less than
    sum_{l >= S} (2S - 1 - l) K 2^14 2^{-8l - 12} < S K 2^{2 - 8S}."""
    return (1.0 + 4.0 * nslices) * k * 2.0 ** (-8 * nslices)
