"""ctypes binding of ``libvittles_b200.so`` (the C ABI of ``include/vittles_b200.h``).

PyTorch supplies device memory (``tensor.data_ptr()``) and the current CUDA
stream; every numerical operation on the hot path is a kernel of the library.
There is NO CPU fallback: if the library is missing, or no CUDA device is
visible, the first compute call raises ``RuntimeError``.
"""
import ctypes
import os

import numpy as np
import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('VT_LIB_PATH') or os.path.join(_PKG, 'lib', 'libvittles_b200.so')   # (override: A/B builds)

VT_OK, VT_ERR_CUDA, VT_ERR_INVALID, VT_ERR_NOT_PD, VT_ERR_NO_CONVERGENCE = 0, 1, 2, 3, 4
GLM_FAMILIES = {'logistic': 0, 'poisson': 1, 'gaussian': 2}
OP_KC, OP_KS = 0, 1

_c = ctypes
_P, _I, _I64, _D, _SZ, _U64 = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_double, _c.c_size_t, _c.c_uint64

# name -> (restype, argtypes); must list every symbol declared in include/vittles_b200.h
SIGNATURES = {
    'vt_last_error': (_c.c_char_p, []),
    'vt_abi_version': (_I, []),
    'vt_launch_count': (_I64, []),
    'vt_device_info': (_I, [_c.POINTER(_I)] * 3),
    'vt_fp64_peak_probe': (_I, [_D, _c.POINTER(_D), _P]),
    'vt_i8_peak_probe': (_I, [_D, _I, _c.POINTER(_D), _c.POINTER(_D), _P]),
    'vt_dgemm_workspace_bytes': (_SZ, [_I, _I, _I, _I, _I]),
    'vt_dgemm': (_I, [_I, _I, _I, _D, _P, _I64, _I, _P, _I64, _I, _D, _P, _I64, _P, _P, _P, _I, _I, _I, _P, _SZ, _P]),
    'vt_syrk_workspace_bytes': (_SZ, [_I64, _I]),
    'vt_syrk_weighted': (_I, [_P, _I64, _I64, _I, _P, _D, _P, _I64, _P, _SZ, _P]),
    'vt_glm_workspace_bytes': (_SZ, [_I]),
    'vt_glm_stats': (_I, [_P, _I64, _I64, _I, _P, _P, _P, _I, _P, _P, _P, _P, _D, _P, _SZ, _P]),
    'vt_glm_stats_colmax': (_I, [_P, _I64, _I64, _I, _P, _P, _P, _I, _P, _P, _P, _P, _D, _P, _P, _P, _SZ, _P]),
    'vt_glm_hvp_multi_workspace_bytes': (_SZ, [_I, _I]),
    'vt_glm_hvp_multi': (_I, [_P, _I64, _I64, _I, _P, _P, _I, _D, _P, _P, _SZ, _P]),
    'vt_glm_hvp': (_I, [_P, _I64, _I64, _I, _P, _P, _D, _P, _P, _SZ, _P]),
    'vt_glm_dirderiv_workspace_bytes': (_SZ, [_I64, _I]),
    'vt_glm_dirderiv': (_I, [_P, _I64, _I64, _I, _P, _P, _I, _P, _I, _P, _P, _SZ, _P]),
    'vt_glm_influence_max_directions': (_I, [_I]),
    'vt_glm_influence': (_I, [_P, _I64, _I64, _I, _P, _P, _I, _D, _P, _I64, _P]),
    'vt_potrf_dinv_doubles': (_SZ, [_I]),
    'vt_potrf': (_I, [_P, _I64, _I, _P, _P, _P]),
    'vt_potrs': (_I, [_P, _I64, _I, _P, _P, _I64, _I, _P]),
    'vt_trsm_lower': (_I, [_P, _I64, _I, _P, _P, _I64, _I, _I, _P]),
    'vt_quad_forms_workspace_bytes': (_SZ, [_I64, _I]),
    'vt_quad_forms': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _P, _SZ, _P]),
    'vt_ij_apply': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _P, _I64, _P]),
    'vt_tf32_gemm_workspace_bytes': (_SZ, [_I, _I, _I64, _I]),
    'vt_tf32_convert': (_I, [_P, _I64, _I64, _I, _P, _I, _P, _P, _I64, _P]),
    'vt_tf32_gemm': (_I, [_I, _I, _I64, _D, _P, _P, _I64, _I, _P, _P, _I64, _I, _P, _I64, _P, _P, _P, _SZ, _P]),
    'vt_ij_apply_tf32_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_ij_apply_tf32': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _P, _I64, _I, _P, _SZ, _P]),
    'vt_syrk_tf32_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_syrk_tf32': (_I, [_P, _I64, _I64, _I, _P, _D, _P, _I64, _I, _P, _SZ, _P]),
    'vt_ozaki_slice': (_I, [_P, _I64, _I64, _I, _P, _I64, _I64, _I, _P, _P, _P]),
    'vt_ozaki_slice_t': (_I, [_P, _I64, _I64, _I, _P, _P, _P, _I64, _I64, _I, _P, _P]),
    'vt_ozaki_gemm': (_I, [_I, _I, _I, _P, _I64, _I64, _P, _I64, _I64, _I, _D, _P, _P, _P, _I64, _P]),
    'vt_syrk_ozaki_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_syrk_ozaki': (_I, [_P, _I64, _I64, _I, _P, _D, _P, _I64, _I, _P, _P, _P, _SZ, _P]),
    'vt_ij_apply_ozaki_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_ij_apply_ozaki': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _P, _I64, _I, _P, _SZ, _P]),
    'vt_quad_forms_ozaki_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_quad_forms_ozaki': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _I, _P, _SZ, _P]),
    'vt_group_loo_workspace_bytes': (_SZ, [_I64, _I]),
    'vt_group_loo': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _I64, _P, _P, _P, _I, _P, _P, _P, _SZ, _P]),
    'vt_group_loo_ozaki_workspace_bytes': (_SZ, [_I64, _I, _I]),
    'vt_group_loo_ozaki': (_I, [_P, _I64, _P, _I64, _I64, _I, _P, _I64, _P, _P, _P, _I, _P, _P, _I, _P, _SZ, _P]),
    'vt_gemv_workspace_bytes': (_SZ, [_I, _I64]),
    'vt_gemv': (_I, [_P, _I64, _I, _I64, _P, _D, _P, _D, _P, _P, _SZ, _P]),
    'vt_cg_batch_init': (_I, [_I, _I, _P, _P, _P, _P, _D, _D, _I, _P]),
    'vt_cg_batch_update_p': (_I, [_I, _I, _P, _P, _P, _P, _P, _I, _P]),
    'vt_cg_batch_update_xr': (_I, [_I, _I, _P, _P, _P, _P, _P, _P]),
    'vt_block_potrf_batched': (_I, [_P, _I64, _I, _P, _P]),
    'vt_block_trsm_batched': (_I, [_P, _P, _I64, _I, _I, _P]),
    'vt_block_trsmt_batched': (_I, [_P, _P, _I64, _I, _I, _P]),
    'vt_block_solve_batched': (_I, [_P, _P, _I64, _I, _I, _P]),
    'vt_tall_gemv': (_I, [_P, _I64, _I, _P, _D, _P, _D, _P]),
    'vt_tall_colsum_workspace_bytes': (_SZ, [_I]),
    'vt_tall_colsum': (_I, [_P, _I64, _I, _P, _D, _P, _D, _P, _P, _SZ, _P]),
    'vt_gmm_blocks': (_I, [_P, _I64, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'vt_synth_design': (_I, [_P, _I64, _I64, _I64, _I, _U64, _D, _P]),
    'vt_synth_uniform': (_I, [_P, _I64, _I64, _U64, _P]),
    'vt_synth_bernoulli': (_I, [_P, _P, _I64, _I64, _U64, _P]),
}

_lib = None


def load():
    """Load the shared library (no GPU needed) and type every entry point."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                'vittles_b200: {} is missing. Build it with `python -m vittles_b200.build` '
                '(nvcc, sm_100a). There is no CPU fallback.'.format(LIB_PATH))
        lib = _c.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError('vittles_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback.')
    return load()


def check(status):
    """Map a C-ABI status to the exception type the reference raises
    (SURVEY.md section 8b: ValueError for validation, LinAlgError for a
    non-positive-definite matrix)."""
    if status == VT_OK:
        return
    msg = load().vt_last_error().decode('utf-8', 'replace')
    if status == VT_ERR_INVALID:
        raise ValueError(msg)
    if status == VT_ERR_NOT_PD:
        raise np.linalg.LinAlgError(msg)
    raise RuntimeError('vittles_b200: {} (status {})'.format(msg, status))


def ptr(t):
    """Device pointer of a float64 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not (isinstance(t, torch.Tensor) and t.is_cuda):
        raise TypeError('expected a CUDA tensor')
    return _c.c_void_p(t.data_ptr())


def stream():
    return _c.c_void_p(torch.cuda.current_stream().cuda_stream)


def exported_symbols():
    return sorted(SIGNATURES)
