"""Measure leave-one-group-out on both engines and approximate_cv(groups=...) end to end.

    python tools/lgo_probe.py [--n 10000000] [--d 1024] [--seconds 1.0] [--sizes 1,8,32]

Prints one JSON line:
  * gpu, power_limit_w: the card and its power limit, read in the same run;
  * lgo_ozaki_<m>, lgo_f64_<m>: ms per ops.group_loo(..., 'ns') with groups of m rows at (N, D), X resident (82 GB at
    the default shape, far larger than the L2), on the INT8 engine and on the DMMA engine; lgo_ozaki_ij_<m>: the IJ
    predictor on the INT8 engine (no Cholesky of M);
  * quad_ozaki, apply_ozaki: ms per ops.quad_forms(..., 'f64_ozaki') and ops.ij_apply(..., 'f64_ozaki') at the same
    shape, for comparison (the apply writes the 82 GB of S);
  * acv_groups: ObservationInfluence(...).approximate_cv('ns', groups=...) with groups of 8 on a fresh instance at
    the optimum of a logistic fit: seconds (host clock around work that ends in a device synchronise), peak
    allocated device memory (X included) and its growth over what was allocated before the call.
Each kernel timing is CUDA events around back-to-back calls for at least --seconds, after a warm-up call.  Needs a
GPU; writes nothing.
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
from loo_probe import fit  # noqa: E402


def starts_of(n, m):
    s = torch.arange(0, n, m, dtype=torch.int64, device='cuda')
    return torch.cat([s, torch.full((1,), n, dtype=torch.int64, device='cuda')])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--d', type=int, default=1024)
    ap.add_argument('--seconds', type=float, default=1.0)
    ap.add_argument('--sizes', default='1,8,32')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('lgo_probe needs a GPU')
    n, d = args.n, args.d
    name, plim = gpu_info()
    X, y = synth(n, d)
    obj, theta, w = fit(X, y)
    st = obj.vt_stats(theta, w, want_grad=False)
    oi = vt.ObservationInfluence(obj, theta, w)
    Linv = oi.factor.inverse_factor()
    s, u, z = st['s'], w * st['resid'], st['z']
    res = dict(gpu=name, power_limit_w=plim, N=n, D=d)
    for m in (int(v) for v in args.sizes.split(',')):
        starts = starts_of(n, m)
        for engine, key in (('f64_ozaki', 'lgo_ozaki'), ('f64', 'lgo_f64')):
            ms = timed(lambda: ops.group_loo(Linv, X, starts, s, u, z, 'ns', precision=engine), args.seconds)
            res['{}_{}'.format(key, m)] = round(ms, 2)
        ms = timed(lambda: ops.group_loo(Linv, X, starts, s, u, z, 'ij', precision='f64_ozaki'), args.seconds)
        res['lgo_ozaki_ij_{}'.format(m)] = round(ms, 2)
    h = torch.empty(n, dtype=torch.float64, device='cuda')
    res['quad_ozaki'] = round(timed(lambda: ops.quad_forms(Linv, X, precision='f64_ozaki', out=h), args.seconds), 2)
    del h
    ops.free_workspaces()
    S = torch.empty((d, n), dtype=torch.float64, device='cuda')
    res['apply_ozaki'] = round(timed(lambda: ops.ij_apply(Linv, X, st['resid'], out=S, precision='f64_ozaki'),
                                     args.seconds), 2)
    del S, st, s, u, z, Linv
    ops.free_workspaces()
    torch.cuda.empty_cache()
    labels = torch.arange(n, device='cuda') // 8
    oi.approximate_cv('ns', groups=labels)                        # warm-up: workspaces, modules
    oi = vt.ObservationInfluence(obj, theta, w)
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    r = oi.approximate_cv('ns', groups=labels)
    torch.cuda.synchronize()
    res['acv_groups'] = dict(s=round(time.perf_counter() - t0, 4),
                             peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 2),
                             growth_gb=round((torch.cuda.max_memory_allocated() - before) / 1e9, 3),
                             mean_loss=r.mean_loss, n_invalid=r.n_invalid)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
