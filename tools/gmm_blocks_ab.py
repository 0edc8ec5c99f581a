"""name: time gmm_blocks of two or more builds of the library against each other at the config-3 shape, in turn.

    python tools/gmm_blocks_ab.py BASE.so OTHER.so [MORE.so ...] [--n N] [--k K] [--d D] [--reps R] [--out FILE]

Each library is loaded on its own (ctypes, RTLD_LOCAL) and called through its C ABI (vt_gmm_blocks) on the same
device buffers: overlapping clusters (centers 0.35 randn), logits in [-1.5, 1.5].  One round times 5 back-to-back
launches of each library with CUDA events, the order of the libraries rotating from round to round; the output
buffers (48 GB of cross blocks at the default shape, far beyond L2) are written in full by every launch.  Prints one
JSON line with the card's name and power limit, the median and spread of the per-launch times of each library, and
how far each library's outputs are from the first one's (responsibilities and objective terms must be
bit-identical)."""
import argparse
import ctypes
import json
import subprocess

import numpy as np
import torch


def _lib(path):
    lib = ctypes.CDLL(path, mode=ctypes.RTLD_LOCAL)
    fn = lib.vt_gmm_blocks
    P, I, I64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    fn.argtypes = [P, I64, I, I, P, P, P, P, P, P, P, P, P]
    fn.restype = I
    return fn


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('libs', nargs='+', help='shared libraries exporting vt_gmm_blocks; the first is the baseline')
    ap.add_argument('--n', type=int, default=1000000)
    ap.add_argument('--k', type=int, default=20)
    ap.add_argument('--d', type=int, default=16)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    N, K, d = a.n, a.k, a.d
    M = K - 1
    assert len(a.libs) >= 2, 'need a baseline and at least one other library'
    names = ['lib{}'.format(i) for i in range(len(a.libs))]
    fns = {k: _lib(p) for k, p in zip(names, a.libs)}
    gen = torch.Generator(device='cuda').manual_seed(3)
    f64 = dict(dtype=torch.float64, device='cuda')
    centers = 0.35 * torch.randn(K, d, generator=gen, **f64)
    X = centers[torch.randint(0, K, (N,), generator=gen, device='cuda')] + torch.randn(N, d, generator=gen, **f64)
    m = (centers + 0.05 * torch.randn(K, d, generator=gen, **f64)).contiguous()
    rho = (3.0 * torch.rand(N, M, generator=gen, **f64) - 1.5).contiguous()
    log_pi = torch.log_softmax(0.3 * torch.randn(K, generator=gen, **f64), 0)
    cross = torch.empty(N, M, K * d, **f64)
    outs = {k: dict(blocks=torch.empty(N, M, M, **f64), r=torch.empty(N, K, **f64), grad_rho=torch.empty(N, M, **f64),
                    obj_terms=torch.empty(N, **f64)) for k in fns}
    stream = torch.cuda.current_stream().cuda_stream

    def call(k):
        o = outs[k]
        rc = fns[k](X.data_ptr(), N, d, K, m.data_ptr(), rho.data_ptr(), log_pi.data_ptr(), o['blocks'].data_ptr(),
                    cross.data_ptr(), o['r'].data_ptr(), o['grad_rho'].data_ptr(), o['obj_terms'].data_ptr(), stream)
        assert rc == 0, (k, rc)

    for k in fns:                        # warm-up: module load, first touch of the buffers
        call(k)
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    per_round = 5
    for rep in range(a.reps):
        sh = rep % len(names)
        for k in names[sh:] + names[:sh]:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(per_round):
                call(k)
            ev1.record()
            ev1.synchronize()
            times[k].append(ev0.elapsed_time(ev1) / per_round)
    # outputs against the baseline's: every output but the cross blocks in full, the cross blocks of the first 20000
    n_c = min(N, 20000)
    crosses = {}
    for k in names:
        call(k)
        crosses[k] = cross[:n_c].clone()
    torch.cuda.synchronize()
    o = outs[names[0]]

    def rel(x, y):
        return float(((x - y).abs().max() / y.abs().max()).item())
    diffs = {k: dict(blocks=rel(outs[k]['blocks'], o['blocks']), grad_rho=rel(outs[k]['grad_rho'], o['grad_rho']),
                     cross=rel(crosses[k], crosses[names[0]]), r_bit_identical=bool(torch.equal(outs[k]['r'], o['r'])),
                     obj_bit_identical=bool(torch.equal(outs[k]['obj_terms'], o['obj_terms']))) for k in names[1:]}
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i',
                          str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    stats = {k: dict(median_ms=float(np.median(v)), min_ms=float(np.min(v)), max_ms=float(np.max(v))) for k, v in
             times.items()}
    base = stats[names[0]]['median_ms']
    res = dict(shape=dict(N=N, K=K, d=d), gpu=smi, launches_per_sample=per_round, samples=a.reps,
               libs=dict(zip(names, a.libs)), times=stats,
               median_over_baseline={k: stats[k]['median_ms'] / base for k in names[1:]}, vs_baseline=diffs)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
