#!/usr/bin/env python3
"""Staged bring-up / timing probe of the INT8 error-free-slicing engine (csrc/ogemm.cu).

    python tools/ogemm_probe.py            # every stage, each in its own process
    python tools/ogemm_probe.py STAGE
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = ['i8_peak', 'slice', 'one', 'k1024', 'big', 'ragged', 's8', 'apply', 'time_apply', 'time_parts', 'syrk', 'time_syrk']


def run(stage):
    import torch
    from vittles_b200 import ops, _cabi
    from vittles_b200._cabi import ptr, stream, check
    dev = torch.device('cuda', 0)
    g = torch.Generator(device=dev).manual_seed(1)

    def rnd(*shape):
        return torch.randn(*shape, device=dev, dtype=torch.float64, generator=g)

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    def digits_reference(As, sa, Bs, sb, S):
        """what the kernel is asked to compute, from the digits, in float64 (exact up to 2^-53 per term)"""
        M, N = As.shape[1], Bs.shape[1]
        acc = torch.zeros((M, N), dtype=torch.float64, device=dev)
        for s in range(S):
            for t in range(S - s):
                P = As[s].double() @ Bs[t].double().T          # exact: |P| < 2^53
                acc += P * 2.0 ** (-8 * (s + t) - 12)
        return sa[:, None] * sb[None, :] * acc

    def gemm_case(name, M, N, K, S=7):
        A, B = rnd(M, K), rnd(N, K)
        out = ops.ozaki_gemm(A, B, nslices=S)
        torch.cuda.synchronize()
        As, sa = ops.ozaki_slice(A, S)
        Bs, sb = ops.ozaki_slice(B, S)
        refd = digits_reference(As, sa, Bs, sb, S)
        exact = A @ B.T
        d = (out - refd).abs()
        res = {'stage': name, 'shape': [M, N, K], 'S': S, 'rel_vs_digits': float(d.max() / refd.abs().max()),
               'rel_vs_f64': float((out - exact).abs().max() / exact.abs().max()),
               'elementwise_rel_vs_f64_p99': float(torch.quantile(((out - exact).abs() / exact.abs().clamp_min(1e-300)).flatten()[:1000000], 0.99)),
               'nan': bool(torch.isnan(out).any())}
        if res['rel_vs_digits'] > 1e-6 or res['nan']:
            res['row_bands'] = [round(float(d[i:i + 32].max()), 4) for i in range(0, min(M, 256), 32)]
            res['col_bands'] = [round(float(d[:, j:j + 16].max()), 4) for j in range(0, min(N, 128), 16)]
            res['out_00'] = [float(v) for v in out[0, :4]]
            res['ref_00'] = [float(v) for v in refd[0, :4]]
        print(json.dumps(res), flush=True)

    if stage == 'i8_peak':
        import ctypes
        lib = _cabi.require_cuda()
        secs = float(os.environ.get('VT_PEAK_SECS', '1.0'))
        for n in [int(v) for v in os.environ.get('VT_PEAK_N', '64,128,192,256').split(',')]:
            tops, clk = ctypes.c_double(), ctypes.c_double()
            check(lib.vt_i8_peak_probe(secs, n, ctypes.byref(tops), ctypes.byref(clk), stream()))
            print(json.dumps({'stage': stage, 'n_tile': n, 'seconds': secs, 'int8_tops': tops.value,
                              'sm_clocks_per_mma': clk.value}), flush=True)
    elif stage == 'slice':
        X = rnd(300, 102) * torch.exp(3 * rnd(300, 1))
        X[7] = 0.0
        for S in (6, 7):
            d, sc = ops.ozaki_slice(X, S)
            rec = torch.zeros_like(X)
            for s in range(S):
                rec += d[s, :, :102].double() * 2.0 ** (-8 * s - 6)
            rec *= sc[:, None]
            rowmax = X.abs().max(dim=1).values.clamp_min(1e-300)
            print(json.dumps({'stage': stage, 'S': S, 'max_digit': int(d.abs().max()), 'pad_zero': bool((d[:, :, 102:] == 0).all()),
                              'resid_rel_rowmax': float(((X - rec).abs().max(dim=1).values / rowmax).max()),
                              'bound': 2.0 ** (-(8 * S - 1)), 'scale_pow2': bool((torch.frexp(sc)[0] == 0.5).all()),
                              'scale_covers': bool((sc >= X.abs().max(dim=1).values).all())}), flush=True)
    elif stage == 'one':
        gemm_case(stage, 128, 64, 128)
        gemm_case(stage + '_n128', 128, 128, 128)
    elif stage == 'k1024':
        gemm_case(stage, 128, 64, 1024)
        gemm_case(stage + '_m256', 256, 128, 1024)
    elif stage == 'big':
        gemm_case(stage, 1024, 4096, 1024)
    elif stage == 'ragged':
        gemm_case(stage, 200, 300, 100)
        gemm_case(stage + '_k1000', 130, 515, 1000)
    elif stage == 's8':
        gemm_case(stage, 512, 512, 1024, S=5)
        gemm_case(stage + '_s6', 512, 512, 1024, S=6)
    elif stage in ('apply', 'time_apply'):
        D = 1024
        N = int(os.environ.get('VT_APPLY_N', '20000')) if stage == 'apply' else 1000000
        X = ops.synth_design(7, 0, N, D, dev)
        Hm = rnd(D, D)
        Hinv = torch.linalg.inv(Hm @ Hm.T / D + 0.05 * torch.eye(D, device=dev, dtype=torch.float64)).contiguous()
        resid = rnd(N)
        ref = ops.ij_apply(Hinv, X, resid)
        out = ops.ij_apply(Hinv, X, resid, precision='f64_ozaki')
        torch.cuda.synchronize()
        err = (out - ref).abs()
        res = {'stage': stage, 'N': N, 'rel_max': float(err.max() / ref.abs().max()),
               'elementwise_rel_max': float((err / ref.abs().clamp_min(1e-300)).max()),
               'rtol1e-8_atol1e-12max_ok': bool((err <= 1e-8 * ref.abs() + 1e-12 * ref.abs().max()).all())}
        if stage == 'time_apply':
            ms = timed(lambda: ops.ij_apply(Hinv, X, resid, out=out, precision='f64_ozaki'))
            ms64 = timed(lambda: ops.ij_apply(Hinv, X, resid, out=ref), reps=1)
            res.update({'ms': ms, 'fp64_equiv_tflops': 2.0 * D * D * N / ms / 1e9, 'ms_f64_dmma': ms64})
        print(json.dumps(res), flush=True)
    elif stage == 'time_parts':
        lib = _cabi.require_cuda()
        D = 1024
        for S in (5, 6, 7):
            nchunk = 37888
            X = ops.synth_design(7, 0, nchunk, D, dev)
            Hinv = rnd(D, D)
            ms_slice = timed(lambda: ops.ozaki_slice(X, S))
            Bs, sb = ops.ozaki_slice(X, S)
            As, sa = ops.ozaki_slice(Hinv, S)
            out = torch.empty((D, nchunk), dtype=torch.float64, device=dev)

            def gemm_only():
                check(lib.vt_ozaki_gemm(D, nchunk, D, ptr(As), As.stride(1), As.stride(0), ptr(Bs), Bs.stride(1),
                                        Bs.stride(0), S, -1.0, ptr(sa), ptr(sb), ptr(out), nchunk, stream()))
            ms_gemm = timed(gemm_only, reps=5)
            pairs = S * (S + 1) // 2
            print(json.dumps({'stage': stage, 'S': S, 'chunk_rows': nchunk, 'ms_slice': ms_slice,
                              'slice_gb_per_s': nchunk * D * (8 + S) / ms_slice / 1e6, 'ms_gemm': ms_gemm,
                              'fp64_equiv_tflops': 2.0 * D * D * nchunk / ms_gemm / 1e9,
                              'int8_tops': 2.0 * D * D * nchunk * pairs / ms_gemm / 1e9}), flush=True)
    elif stage == 'timing':
        # VT_OGEMM_TIMING=1 must be set: where the MMA-issuing thread waits (clocks, mean over CTAs)
        import ctypes
        lib = _cabi.require_cuda()
        D, S, nchunk = 1024, 7, 37888
        X = ops.synth_design(7, 0, nchunk, D, dev)
        Hinv = rnd(D, D)
        Bs, sb = ops.ozaki_slice(X, S)
        As, sa = ops.ozaki_slice(Hinv, S)
        out = torch.empty((D, nchunk), dtype=torch.float64, device=dev)

        def gemm_only():
            check(lib.vt_ozaki_gemm(D, nchunk, D, ptr(As), As.stride(1), As.stride(0), ptr(Bs), Bs.stride(1),
                                    Bs.stride(0), S, -1.0, ptr(sa), ptr(sb), ptr(out), nchunk, stream()))
        buf = (ctypes.c_ulonglong * 8)()
        gemm_only(); torch.cuda.synchronize()
        lib.vt_debug_ogemm_timing.restype = ctypes.c_int
        lib.vt_debug_ogemm_timing(buf)
        ms = timed(gemm_only, reps=1)
        rc = lib.vt_debug_ogemm_timing(buf)
        n = max(1, buf[4])
        print(json.dumps({'stage': stage, 'rc': rc, 'ms': ms, 'launches_x_ctas': buf[4], 'clk_total': buf[0] / n,
                          'clk_wait_accum': buf[1] / n, 'clk_wait_B': buf[2] / n, 'clk_wait_A': buf[3] / n,
                          'tiles_per_cta': 8 * (nchunk // 64) / 148}), flush=True)
        # the whole apply (D = 1024: the converter warps of each GEMM slice the next chunk)
        N = 20 * nchunk
        Xb = ops.synth_design(7, 0, N, D, dev)
        resid = rnd(N)
        outb = ops.ij_apply(Hinv, Xb, resid, precision='f64_ozaki')
        torch.cuda.synchronize()
        lib.vt_debug_ogemm_timing(buf)
        ms = timed(lambda: ops.ij_apply(Hinv, Xb, resid, out=outb, precision='f64_ozaki'), reps=1)
        lib.vt_debug_ogemm_timing(buf)
        n, nc = max(1, buf[4]), max(1, buf[6])
        print(json.dumps({'stage': stage + '_apply', 'chunks': 20, 'ms': ms, 'mma_clk_total_per_launch': buf[0] / n,
                          'clk_wait_accum': buf[1] / n, 'clk_wait_B': buf[2] / n, 'clk_wait_A': buf[3] / n,
                          'converter_clk_per_launch': buf[5] / nc, 'converter_warps': buf[6]}), flush=True)
    elif stage in ('syrk', 'time_syrk'):
        D = 1024
        for N in ((777, 50000) if stage == 'syrk' else (1000000,)):
            X = ops.synth_design(7, 0, N, D, dev)
            s = torch.rand(N, device=dev, dtype=torch.float64, generator=g) * 0.25
            ref = ops.syrk_weighted(X, s)
            out = ops.syrk_weighted(X, s, precision='f64_ozaki')
            torch.cuda.synchronize()
            err = (out - ref).abs()
            res = {'stage': stage, 'N': N, 'rel_max': float(err.max() / ref.abs().max()), 'symmetric': bool(torch.equal(out, out.T)),
                   'rtol1e-8_atol1e-12max_ok': bool((err <= 1e-8 * ref.abs() + 1e-12 * ref.abs().max()).all()),
                   'nan': bool(torch.isnan(out).any())}
            if res['rel_max'] > 1e-6 or res['nan']:
                res['row_bands'] = [round(float(err[i:i + 128].max()), 6) for i in range(0, D, 128)]
                res['col_bands'] = [round(float(err[:, j:j + 64].max()), 6) for j in range(0, D, 64)]
                res['out_00'] = [float(v) for v in out[0, :4]]
                res['ref_00'] = [float(v) for v in ref[0, :4]]
            if stage == 'time_syrk':
                ms = timed(lambda: ops.syrk_weighted(X, s, out=out, precision='f64_ozaki'))
                ms64 = timed(lambda: ops.syrk_weighted(X, s, out=ref), reps=1)
                res.update({'ms': ms, 'fp64_equiv_tflops_algorithmic': float(D) * (D + 1) * N / ms / 1e9, 'ms_f64_dmma': ms64})
            print(json.dumps(res), flush=True)
    else:
        raise SystemExit('unknown stage ' + stage)


if __name__ == '__main__':
    if len(sys.argv) > 1:
        run(sys.argv[1])
    else:
        for st in STAGES:
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), st], capture_output=True, text=True,
                                   timeout=150)
                sys.stdout.write(r.stdout)
                if r.returncode != 0:
                    print(json.dumps({'stage': st, 'rc': r.returncode, 'stderr': r.stderr[-700:]}), flush=True)
            except subprocess.TimeoutExpired:
                print(json.dumps({'stage': st, 'timeout': True}), flush=True)
