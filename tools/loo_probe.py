"""Measure the quadratic forms h_n = |L^{-1} x_n|^2 on the INT8 engine and approximate leave-one-out CV end to end.

    python tools/loo_probe.py [--n 10000000] [--d 1024] [--seconds 1.0] [--quad-only]

Prints one JSON line:
  * gpu, power_limit_w: the card and its power limit, read in the same run;
  * i8_peak_tops: dense INT8 TOP/s of the bare tcgen05.mma loop (ops.i8_peak_probe), the roofline's denominator;
  * quad_ozaki: ms per ops.quad_forms(..., 'f64_ozaki') at (N, D), X resident (82 GB at the default shape, far
    larger than the L2), and the INT8 TOP/s of the MMA work it executes (triangular: row block tm of L^{-1} meets
    k-blocks 0 .. tm; 28 digit products of 128 x 64 x 128 per k-block and tile) with its fraction of i8_peak_tops;
  * apply_ozaki: ms per ops.ij_apply(..., 'f64_ozaki') at the same shape (it writes the 82 GB of S) and
    quad_over_apply, the ratio of the two times;
  * quad_f64: ms per ops.quad_forms(..., 'f64') (the DMMA engine);
  * acv: ObservationInfluence(...).approximate_cv() on a fresh instance at the optimum of a logistic fit: seconds
    (host clock around work that ends in a device synchronise), peak allocated device memory (X included) and its
    growth over what was allocated before the call.
Each kernel timing is CUDA events around back-to-back calls for at least --seconds, after a warm-up call.
--quad-only measures i8_peak_tops and quad_ozaki alone (run it with VT_LIB_PATH pointing at a build compiled with
-DVT_QF_NAIVE_ORDER to time the unbalanced unit order).  Needs a GPU; writes nothing.
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))
import vittles_b200 as vt  # noqa: E402
from vittles_b200 import ops  # noqa: E402
from influence_probe import SEED, gpu_info, synth, timed  # noqa: E402

OBM, OBN, OBK, S7 = 128, 64, 128, 7
CHUNK_BYTES = 288 << 20


def chunk_rows(N, D, G):
    """ozaki_chunk_rows (ogemm.cu)."""
    ld = (D + 15) // 16 * 16
    nb = max(1, CHUNK_BYTES // (ld * S7) // OBN)
    tiles_m = (D + OBM - 1) // OBM
    best, best_eff, b = nb, 0.0, nb
    while b >= 1 and b > nb // 2:
        T = b * tiles_m
        eff = T / (G * ((T + G - 1) // G))
        if eff > best_eff + 1e-9:
            best, best_eff = b, eff
        b -= 1
    return min(best * OBN, N)


def quad_ops(N, D, G):
    """INT8 operations the triangular quadratic forms execute: per 64-row column tile, sum over row blocks tm of
    (tm + 1) k-blocks of 28 digit products of 128 x 64 x 128."""
    T = (D + OBM - 1) // OBM
    ch = chunk_rows(N, D, G)
    col_tiles = sum(-(-min(ch, N - r0) // OBN) for r0 in range(0, N, ch))
    return 2.0 * (S7 * (S7 + 1) // 2) * OBM * OBN * OBK * (T * (T + 1) // 2) * col_tiles


def fit(X, y, iters=12):
    n, d = X.shape
    obj = vt.objectives.GLMObjective(X, y, l2=1.0)
    w = torch.ones(n, dtype=torch.float64, device='cuda')
    theta = torch.zeros(d, dtype=torch.float64, device='cuda')
    for _ in range(iters):
        st, H = obj.vt_stats_and_hessian(theta, w)
        step = ops.potrf(H, overwrite=True).solve(st['grad'])
        theta = theta - step
        if float(torch.linalg.vector_norm(step)) < 1e-11:
            break
    return obj, theta, w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--d', type=int, default=1024)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--quad-only', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('loo_probe needs a GPU')
    n, d = args.n, args.d
    name, plim = gpu_info()
    G = ops.device_info()['sm_count']
    peak = ops.i8_peak_probe(seconds=args.seconds)['tops']
    X, y = synth(n, d)
    g = torch.Generator(device='cuda').manual_seed(SEED)
    A = torch.randn(d, d, dtype=torch.float64, device='cuda', generator=g)
    Linv = ops.potrf(A @ A.T / d + torch.eye(d, dtype=torch.float64, device='cuda')).inverse_factor()
    del A
    h = torch.empty(n, dtype=torch.float64, device='cuda')
    ms_q = timed(lambda: ops.quad_forms(Linv, X, precision='f64_ozaki', out=h), args.seconds)
    tops = quad_ops(n, d, G) / (ms_q * 1e-3) / 1e12
    res = dict(gpu=name, power_limit_w=plim, lib=os.path.relpath(vt._cabi.LIB_PATH, ROOT), N=n, D=d,
               i8_peak_tops=round(peak, 1),
               quad_ozaki=dict(ms=round(ms_q, 2), int8_tops=round(tops, 1), peak_fraction=round(tops / peak, 3)))
    if not args.quad_only:
        ms_f = timed(lambda: ops.quad_forms(Linv, X, precision='f64', out=h), args.seconds)
        res['quad_f64'] = dict(ms=round(ms_f, 2))
        del h
        ops.free_workspaces()
        obj, theta, w = fit(X, y)
        resid = obj.vt_stats(theta, w, want_grad=False)['resid']
        S = torch.empty((d, n), dtype=torch.float64, device='cuda')
        ms_a = timed(lambda: ops.ij_apply(Linv, X, resid, out=S, precision='f64_ozaki'), args.seconds)
        res['apply_ozaki'] = dict(ms=round(ms_a, 2))
        res['quad_over_apply'] = round(ms_q / ms_a, 3)
        del S, resid
        ops.free_workspaces()
        torch.cuda.empty_cache()
        oi = vt.ObservationInfluence(obj, theta, w)
        oi.approximate_cv()                                       # warm-up: workspaces, modules
        oi = vt.ObservationInfluence(obj, theta, w)
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        r = oi.approximate_cv()
        torch.cuda.synchronize()
        res['acv'] = dict(s=round(time.perf_counter() - t0, 4), peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 2),
                          growth_gb=round((torch.cuda.max_memory_allocated() - before) / 1e9, 3),
                          mean_loss=r.mean_loss, n_invalid=r.n_invalid,
                          max_leverage=float(r.leverage.max()))
    print(json.dumps(res))


if __name__ == '__main__':
    main()
