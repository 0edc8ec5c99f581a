"""Weighted SYRK on the INT8 slicing engine: time per call and a hash of the result.
    python tools/syrk_probe.py [N D [N D ...]]"""
import hashlib
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vittles_b200 import ops  # noqa: E402


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def main():
    dev = torch.device('cuda', 0)
    args = [int(float(v)) for v in sys.argv[1:]] or [2_000_000, 1024]
    for N, D in zip(args[0::2], args[1::2]):
        X = ops.synth_design(7, 0, N, D, dev)
        s = torch.rand(N, device=dev, dtype=torch.float64, generator=torch.Generator(device=dev).manual_seed(N + D))
        if os.environ.get('VT_PROBE_UNWEIGHTED') == '1':       # X^T X (the Schur complement of config 3)
            s = None
        row = {'N': N, 'D': D, 'weighted': s is not None}
        for prec in ('f64_ozaki', 'f64'):
            ms, H = timed(lambda: ops.syrk_weighted(X, s, precision=prec), 3)
            row[prec + '_ms'] = ms
            row[prec + '_fp64_equiv_tflops'] = N * D * (D + 1.0) / ms / 1e9
            row[prec + '_sha'] = hashlib.sha256(H.cpu().numpy().tobytes()).hexdigest()[:16]
            if prec == 'f64_ozaki':
                Ho = H
        row['ozaki_vs_f64_rel'] = float((Ho - H).abs().max() / H.abs().max())
        if os.environ.get('VT_OGEMM_TIMING') == '1':       # where the MMA-issuing thread waits (clocks, mean over CTAs)
            import ctypes
            from vittles_b200 import _cabi
            lib = _cabi.require_cuda()
            buf = (ctypes.c_ulonglong * 8)()
            torch.cuda.synchronize()
            lib.vt_debug_ogemm_timing(buf)
            ms, _ = timed(lambda: ops.syrk_weighted(X, s, precision='f64_ozaki'), 1)
            lib.vt_debug_ogemm_timing(buf)
            n, nc = max(1, buf[4]), max(1, buf[6])
            row['timing'] = {'ctas_x_launches_x2': buf[4], 'mma_clk_total': buf[0] / n, 'clk_wait_accum': buf[1] / n,
                             'clk_wait_B': buf[2] / n, 'clk_wait_A': buf[3] / n, 'converter_clk': buf[5] / nc,
                             'converter_warps': buf[6]}
        print(json.dumps(row), flush=True)
        del X, s


if __name__ == '__main__':
    main()
