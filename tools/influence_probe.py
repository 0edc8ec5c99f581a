"""Measure the per-observation influence pass (vt_glm_influence) and the AMIP route end to end.

    python tools/influence_probe.py [--n 10000000] [--d 1024] [--seconds 0.5]

Prints one JSON line:
  * gpu, power_limit_w: the card and its power limit, read in the same run;
  * copy_gbs: device-to-device copy rate of a 4 GB buffer (read + write bytes over time), the reference rate;
  * passes: for K in {1, 2, 4, 8} at (N, D), and for K in {1, max} at D = 4096 and 8192 (N scaled to the same
    bytes of X): ms per call, GB/s with bytes = 8 N D + 8 N + 8 K N, and the fraction of copy_gbs.  Each timing is
    CUDA events around back-to-back calls for at least --seconds, after a warm-up call; X (82 GB at the default
    shape) is far larger than the L2;
  * e2e: ObservationInfluence(...) + amip for one QoI, against HyperparameterSensitivityLinearApproximation(...)
    followed by a @ get_dopt_dhyper(), on the same data: seconds (host clock around work that ends in a device
    synchronise) and peak allocated device memory of each, X included.
Needs a GPU; writes nothing.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vittles_b200 as vt  # noqa: E402
from vittles_b200 import ops  # noqa: E402

SEED = 20261020


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader,nounits', '-i',
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, plim = [s.strip() for s in out.strip().split(',')[:2]]
        return name, float(plim)
    except Exception:
        return torch.cuda.get_device_name(), None


def timed(fn, seconds):
    """ms per call of fn over at least `seconds` of back-to-back calls (CUDA events), after one warm-up call."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    reps = max(3, int(seconds * 1e3 / max(a.elapsed_time(b), 1e-3)) + 1)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def copy_rate(seconds):
    src = torch.empty(1 << 29, dtype=torch.float64, device='cuda')     # 4 GB
    src.fill_(1.0)
    dst = torch.empty_like(src)
    ms = timed(lambda: dst.copy_(src), seconds)
    return 2 * src.numel() * 8 / (ms * 1e-3) / 1e9


def pass_rates(X, Ks, copy_gbs, seconds):
    n, d = X.shape
    c = torch.randn(n, dtype=torch.float64, device='cuda')
    out = []
    for K in Ks:
        V = torch.randn(K, d, dtype=torch.float64, device='cuda')
        res = torch.empty((K, n), dtype=torch.float64, device='cuda')
        ms = timed(lambda: ops.glm_influence(X, c, V, alpha=-1.0, out=res), seconds)
        gb = (8.0 * n * d + 8.0 * n + 8.0 * K * n) / 1e9
        out.append(dict(N=n, D=d, K=K, passes=-(-K // ops.glm_influence_max_directions(d)), ms=round(ms, 3),
                        gbs=round(gb / (ms * 1e-3), 1), copy_fraction=round(gb / (ms * 1e-3) / copy_gbs, 3)))
        del res, V
    return out


def synth(n, d):
    X = ops.synth_design(SEED, 0, n, d, 'cuda')
    theta_star = ops.synth_theta(SEED, d, 'cuda')
    z = ops.glm_stats(X, theta_star, torch.zeros(n, dtype=torch.float64, device='cuda'), None, want_grad=False)[0]
    y = ops.synth_bernoulli(SEED, 0, z)
    return X, y


def end_to_end(X, y):
    n, d = X.shape
    w = torch.ones(n, dtype=torch.float64, device='cuda')
    obj = vt.objectives.GLMObjective(X, y)
    theta = torch.zeros(d, dtype=torch.float64, device='cuda')
    for _ in range(25):
        st, H = obj.vt_stats_and_hessian(theta, w)
        step = ops.potrf(H, overwrite=True).solve(st['grad'])
        theta = theta - step
        if float(torch.linalg.vector_norm(step)) < 1e-11:
            break
    del st, H, step
    a = torch.zeros(d, dtype=torch.float64, device='cuda')
    a[0] = 1.0
    value = float(theta[0])

    def influence_route():
        inf = vt.ObservationInfluence(obj, theta, w)
        return inf.amip((a, value), max_drop=0.01)

    def s_route():
        sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
        return a[None, :] @ sens.get_dopt_dhyper()

    res = {}
    for name, fn in (('influence_amip', influence_route), ('s_route', s_route)):
        r = fn()                                                            # warm-up: workspaces, modules
        del r
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        res[name] = dict(s=round(time.perf_counter() - t0, 4), peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 2))
        if name == 'influence_amip':
            res[name].update(n_drop=r.n_drop, max_change=r.max_change)
        del r
        torch.cuda.synchronize()
    res['speedup'] = round(res['s_route']['s'] / res['influence_amip']['s'], 2)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=10_000_000)
    ap.add_argument('--d', type=int, default=1024)
    ap.add_argument('--seconds', type=float, default=0.5)
    ap.add_argument('--no-e2e', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('influence_probe needs a GPU')
    name, plim = gpu_info()
    copy_gbs = copy_rate(args.seconds)
    X, y = synth(args.n, args.d)
    passes = pass_rates(X, [1, 2, 4, 8], copy_gbs, args.seconds)
    e2e = None if args.no_e2e else end_to_end(X, y)
    bytes_x = args.n * args.d
    del X, y
    ops.free_workspaces()
    torch.cuda.empty_cache()
    for d in (4096, 8192):
        Xw = ops.synth_design(SEED, 0, bytes_x // d, d, 'cuda')
        passes += pass_rates(Xw, sorted({1, ops.glm_influence_max_directions(d)}), copy_gbs, args.seconds)
        del Xw
        torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=name, power_limit_w=plim, copy_gbs=round(copy_gbs, 1), passes=passes, e2e=e2e)))


if __name__ == '__main__':
    main()
