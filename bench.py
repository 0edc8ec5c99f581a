#!/usr/bin/env python3
"""Headline benchmark: all-observation infinitesimal-jackknife sensitivities for
logistic regression, N = 10M, D = 1024, float64 (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" is the whole hot path over the whole data set:
    GLM statistics pass  ->  H = X^T diag(s) X  (-> all-reduce of H)  ->
    Cholesky factor + inverse  ->  S = -H^{-1} G^T  (D x N, device resident)
through the public API (HyperparameterSensitivityLinearApproximation on a
GLMObjective).  Observations are sharded over the ranks (strong scaling of the
fixed N = 10M problem); the only collective is the all-reduce of the D x D
Hessian.  Prints ONE JSON line on rank 0 (contract in the task statement).
"""
import argparse
import json
import os

# Keep the caching allocator from carving small workspaces out of a cached 82 GB block (the (D, N) result):
# the next 82 GB request would then no longer fit on the device.
os.environ.setdefault('PYTORCH_CUDA_ALLOC_CONF', 'max_split_size_mb:512')
import subprocess
import sys
import threading
import time

if '--impl' in sys.argv and 'reference' in sys.argv:
    # The CPU arm uses every host core.  torch.distributed.run exports OMP_NUM_THREADS=1 to its workers and the BLAS
    # pools of numpy and scipy size themselves from the environment when they are first loaded - so set it before
    # either is imported (use_all_host_cores() additionally resizes the pools that are already there).
    _n = str(len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1))
    for _k in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_k] = _n

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = 'per-obs IJ sensitivities/sec (logit N=10M,D=1024)'
UNIT = 'obs/s'
SEED = 20261017
ORIG_AFFINITY = os.sched_getaffinity(0) if hasattr(os, 'sched_getaffinity') else None
FP64_PEAK_FALLBACK_TFLOPS = 37.18      # profiles/fp64_peak_r01.jsonl (tools/fp64_peak.cu on this pool's B200)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=4)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--n-total', type=int, default=10_000_000)
    ap.add_argument('--dim', type=int, default=1024)
    ap.add_argument('--cpu-sample', type=int, default=0,
                    help='rows of the CPU-baseline sample (0: sized from a calibration run, 1e5 .. 1e6 rows)')
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-e2e-full', action='store_true', help='skip the leg that also brings the (D, N) result to the host')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-tf32', action='store_true', help='skip the rows of the other engines (f64 DMMA, tf32x3, tf32)')
    ap.add_argument('--precision', default='auto', choices=['auto', 'f64', 'f64_ozaki', 'tf32x3', 'tf32'],
                    help="engine of the two contractions for the headline and e2e legs (default 'auto': the library's "
                         "default, which is the FP64-grade INT8 error-free-slicing engine at this size)")
    ap.add_argument('--no-configs', action='store_true', help='skip BASELINE configs 3, 4, 5 (tools/bench_configs.py)')
    ap.add_argument('--engine-rows-only', action='store_true', help=argparse.SUPPRESS)   # child mode, see main()
    ap.add_argument('--engines', action='store_true', help='also measure the other engines when --gpus > 1 '
                    '(by default they are measured on 1 GPU only)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed as float64 .npy files in DIR: '
                         'hessian_at_opt (D, D) and dopt_dhyper_sample, the columns of the (D, N) sensitivities at a '
                         'fixed seeded sample of observations (see dump_outputs)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    if args.dump_outputs and dump_columns(args.n_total, args.dim) < 1:
        ap.error('--dump-outputs: the {0} x {0} Hessian alone exceeds {1} bytes'.format(args.dim, DUMP_BYTES))
    return args


# ---------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores
# ---------------------------------------------------------------------------

def cpu_reference_step(n, d, seed=SEED):
    """One bounded CPU step: closed-form H and cross-Hessian in numpy (autograd
    assembly cannot run in this image - BASELINE.md section 3), then the
    reference's own solver path get_cholesky_solver(H)(cross) = cho_factor +
    cho_solve (solver_lib.py:27,29; sensitivity_lib.py:389,226).  Returns
    seconds for the n-row sample (data generation excluded)."""
    from oracle import models, solver_lib as osl
    X, y, theta_star = models.synth_logistic(seed, n, d)
    w = np.ones(n)
    theta = theta_star          # timing does not depend on being at the optimum
    t0 = time.perf_counter()
    cf = models.glm_closed_form(X, y, theta, w)
    solve = osl.get_cholesky_solver(cf['hessian'])
    S = -1 * solve(cf['cross_hessian'])
    t1 = time.perf_counter()
    assert S.shape == (d, n)
    return t1 - t0


def use_all_host_cores():
    """BLAS threads := all host cores, whatever OMP_NUM_THREADS says (torch.distributed.run exports
    OMP_NUM_THREADS=1 to its workers, which made the r01 reference arm single-threaded at N > 1).  Returns the
    number of threads the BLAS pool now uses."""
    if hasattr(os, 'sched_setaffinity'):
        os.sched_setaffinity(0, ORIG_AFFINITY)      # undo the NUMA binding of the GPU legs
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        import scipy.linalg                         # noqa: F401  (load scipy's own BLAS before resizing the pools)
        from threadpoolctl import threadpool_limits, threadpool_info
        threadpool_limits(limits=ncores)           # stays in force for the life of the process
        return max([p.get('num_threads', 1) for p in threadpool_info()] + [1])
    except Exception:
        return 1


def cpu_sample_rows(args, cores, steps_total):
    """Rows of the CPU sample: as many as fit a budget of ~150 s for `steps_total` steps (and host memory),
    between 1e5 and 1e6, from a 20 000-row calibration step."""
    if args.cpu_sample > 0:
        return args.cpu_sample
    d = args.dim
    cpu_reference_step(5000, d)                      # BLAS warm-up
    per_row = cpu_reference_step(20000, d) / 20000.0
    n = int(150.0 / (steps_total * per_row))
    try:
        import psutil
        n = min(n, int(0.25 * psutil.virtual_memory().available / (4 * 8 * d)))   # X, cross-Hessian, S + slack
    except Exception:
        pass
    return int(max(100_000, min(1_000_000, n)) // 1000 * 1000)


def run_reference_arm(args):
    """--impl reference: the reference's CPU path for this metric on all host cores (oracle port: numpy closed-form
    assembly + the reference's cho_factor / cho_solve), each step a bounded sample of the workload."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    cores = use_all_host_cores()
    d = args.dim
    warm = max(1, args.warmup)
    n = cpu_sample_rows(args, cores, args.steps + warm)
    for _ in range(warm):
        cpu_reference_step(n, d)
    times = [cpu_reference_step(n, d) for _ in range(max(1, args.steps))]
    sec = float(np.mean(times))
    value = n / sec
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': len(times), 'warmup': warm, 'ms_per_step': sec * 1e3 * (args.n_total / n),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'logistic IJ N=10M D=1024 f64 (BASELINE configs[1])', 'n_obs': args.n_total,
                   'dim': d, 'sample_rows_per_step': n},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '{} of {} observations per step, D={} (cost is linear in N beyond the D^3/3 '
                                   'factorisation; ms_per_step is scaled to the full N); numpy closed-form assembly + '
                                   'cho_factor/cho_solve on {} BLAS threads'.format(n, args.n_total, d, cores)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------
# clock sampling during the timed region
# ---------------------------------------------------------------------------

class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,' \
        'clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                 '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(np.max(mx)), 'power_w_max': float(np.max(pw)),
                'samples': len(sm), 'reasons': sorted(reasons)}


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------

def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import vittles_b200 as vt
    from vittles_b200 import ops

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus and world > 1:
        raise SystemExit('--gpus {} but WORLD_SIZE={}'.format(args.gpus, world))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    numa_note = numa_bind_to_gpu(local_rank)      # before any pinned allocation: first touch places the pages
    group = None
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
        group = dist.group.WORLD

    N, D = args.n_total, args.dim
    r0 = (N * rank) // world
    r1 = (N * (rank + 1)) // world
    n_loc = r1 - r0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- synthetic data, generated on the device (counter-based) ------------
    X = ops.synth_design(SEED, r0, n_loc, D, dev)
    theta_star = ops.synth_theta(SEED, D, dev)
    zeros = torch.zeros(n_loc, dtype=torch.float64, device=dev)
    z_star = ops.glm_stats(X, theta_star, zeros, None, 'logistic', want_grad=False)[0]
    y = ops.synth_bernoulli(SEED, r0, z_star)
    del z_star, zeros
    w = torch.ones(n_loc, dtype=torch.float64, device=dev)
    obj = vt.objectives.GLMObjective(X, y, family='logistic', group=group, precision=args.precision)

    # ---- optimum by Newton's method on the same kernels (setup, untimed) ----
    theta = torch.zeros(D, dtype=torch.float64, device=dev)
    for it in range(25):
        st = obj.vt_stats(theta, w)
        H = obj.vt_hessian(theta, w, st)
        step = ops.potrf(H, overwrite=True).solve(st['grad'])
        theta = theta - step
        if float(torch.linalg.vector_norm(step)) < 1e-11:
            break
    grad_norm = float(torch.linalg.vector_norm(obj.vt_stats(theta, w)['grad']))
    del st, H, step

    def one_step():
        sens = vt.HyperparameterSensitivityLinearApproximation(obj, theta, w)
        return sens

    peak_tflops = ops.fp64_peak_probe(0.25)
    engine = ops.resolve_precision(args.precision, n_loc, D, w)        # what 'auto' means at this shard size
    i8_peak = ops.i8_peak_probe(1.0, 256) if engine == 'f64_ozaki' else None   # sustained: a 1 s bare-MMA loop

    # ---- timed region: device-resident inputs --------------------------------
    for _ in range(args.warmup):
        s_ = one_step(); del s_
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        s_ = None             # release the previous step's (D, N) result before the next one is allocated
        s_ = one_step()
    e1.record()
    barrier()
    launches = ops.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item()) / args.steps
    value = N / (ms_per_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, s_, torch, dist, world, rank, r0, N, dev)
    del s_

    # ---- per-kernel timing (same stream, CUDA events) -> roofline ------------
    def timed(fn, reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = fn()
        torch.cuda.synchronize()
        a.record()
        for _ in range(reps):
            del out
            out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps, out
    reps = max(2, min(args.steps, 3))
    t_stats, st = timed(lambda: obj.vt_stats(theta, w, for_hessian=True), reps)     # as the step runs it: on the INT8
    # engine the statistics pass also produces the per-feature scales of the Hessian assembly
    t_syrk, H = timed(lambda: ops.syrk_weighted(X, st['s'], precision=engine, colmax=st.get('colmax')), reps)
    if world > 1:
        dist.all_reduce(H)
    t_chol, hinv = timed(lambda: ops.potrf(H).inverse(), reps)
    t_apply, S = timed(lambda: ops.ij_apply(hinv, X, st['resid'], precision=engine), reps)
    apply_tflops = 2.0 * D * D * n_loc / (t_apply * 1e-3) / 1e12
    syrk_tflops = float(D) * (D + 1) * n_loc / (t_syrk * 1e-3) / 1e12
    stats_gbs = 8.0 * D * n_loc / (t_stats * 1e-3) / 1e9
    # the dominant kernel on its own, sustained: the GEMM of one pre-sliced chunk in a >= 0.5 s loop (no slicing, no
    # converter job) - the kernel's own fraction of the INT8 peak, next to the whole-call figure of `roofline`
    gemm_alone = None
    if engine == 'f64_ozaki':
        try:
            from vittles_b200._cabi import check, ptr, require_cuda, stream
            lib = require_cuda()
            S_ = ops.OZAKI_SLICES
            rows_c = min(37888, n_loc)
            Bs, sb = ops.ozaki_slice(X[:rows_c], S_)
            As, sa = ops.ozaki_slice(hinv, S_)
            out_c = torch.empty((D, rows_c), dtype=torch.float64, device=dev)

            def gemm_only():
                check(lib.vt_ozaki_gemm(D, rows_c, D, ptr(As), As.stride(1), As.stride(0), ptr(Bs), Bs.stride(1),
                                        Bs.stride(0), S_, -1.0, ptr(sa), ptr(sb), ptr(out_c), rows_c, stream()))
            for _ in range(20):
                gemm_only()
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nrep = 700
            g0.record()
            for _ in range(nrep):
                gemm_only()
            g1.record()
            torch.cuda.synchronize()
            ms_g = g0.elapsed_time(g1) / nrep
            tops_g = 2.0 * D * D * rows_c * (S_ * (S_ + 1) // 2) / (ms_g * 1e-3) / 1e12
            gemm_alone = {'kernel': 'ogemm_kernel<{}> (vt_ozaki_gemm on one pre-sliced chunk of {} observations)'.format(S_, rows_c),
                          'launches': nrep, 'ms_per_launch': ms_g, 'achieved': tops_g, 'peak': i8_peak['tops'],
                          'unit': 'INT8 TOP/s', 'frac': tops_g / i8_peak['tops'],
                          'fp64_equiv_tflops': 2.0 * D * D * rows_c / (ms_g * 1e-3) / 1e12}
            del Bs, As, out_c
        except Exception as exc:                  # report, never hide
            gemm_alone = {'error': repr(exc)[:200]}
    # conditioning of the Hessian at the optimum (reported: the fused path multiplies by an explicit inverse
    # only while kappa eps stays far below the parity tolerance - sensitivity_lib.EXPLICIT_INVERSE_MAX_COND)
    ev = torch.linalg.eigvalsh(H)
    kappa = float(ev[-1] / ev[0])
    del ev

    # size-independent correctness properties at full size (sampled columns)
    idx = torch.randint(0, n_loc, (256,), device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    G_cols = (X[idx] * st['resid'][idx, None]).T.contiguous()                # (D, 256)
    resid_check = ops.gemm(H, S[:, idx].contiguous().T.contiguous(), 'KC', 'KC') + G_cols
    rel_resid = float(torch.max(torch.abs(resid_check)) / torch.max(torch.abs(G_cols)))
    S_cols64 = S[:, idx].clone()
    del S, G_cols, resid_check

    # ---- other engines for the two contractions, reported next to the FP64 DMMA headline, never
    # instead of it: 'f64_ozaki' (FP64-grade contractions on the INT8 tensor cores, same parity bar) and the
    # optional reduced-precision 'tf32x3' / 'tf32' rows (tcgen05 TF32 engine, stated tolerances).
    # On one GPU they are measured in a CHILD process after everything else (see the end of main): a device
    # fault in an optional engine must never cost the headline line.  With several ranks (--engines) they run here.
    engine_rows = None
    want_rows = not args.no_tf32 and (world == 1 or args.engines)
    if args.engine_rows_only or (want_rows and world > 1):
        import gc
        engine_rows = {}
        for prec in (('f64',) if engine == 'f64_ozaki' else ('f64_ozaki',)) + ('f64_ozaki_s6', 'tf32x3', 'tf32'):
            slices0 = ops.OZAKI_SLICES
            try:
                if prec == 'f64_ozaki_s6':    # the same engine with six digits per operand (46 bits, 21 digit products)
                    ops.OZAKI_SLICES = 6
                engine_rows[prec] = engine_row(prec.replace('_s6', ''), vt, ops, torch, dist, world, group, dev, X, y, theta,
                                               w, st, hinv, idx, S_cols64, N, D, n_loc, reps, timed, note_key=prec)
            except Exception as exc:          # report, never hide
                engine_rows[prec] = {'error': repr(exc)[:300]}
            finally:
                ops.OZAKI_SLICES = slices0
            gc.collect()
            torch.cuda.empty_cache()
        if args.engine_rows_only:
            print(json.dumps({'other_engines': engine_rows}))
            return
    del S_cols64

    peaks = {}
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks = json.load(f)
    except Exception:
        pass
    traffic = traffic_i8 = None
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as f:
            tj = json.load(f)
        traffic = tj.get('ij_apply_dram_bytes_per_obs')
        traffic = None if traffic is None else traffic * n_loc      # per call at this run's shard size
        traffic_i8 = tj.get('ogemm_apply_dram_bytes_per_obs')
        traffic_i8 = None if traffic_i8 is None else traffic_i8 * n_loc
    except Exception:
        pass

    # ---- end to end: HOST buffers in, host result out ---------------------------
    e2e = e2e_full = None
    freed = False
    if not args.no_e2e:
        try:
            room0 = host_headroom_bytes()
            need0 = world * pinned_cost(8 * n_loc * D) + host_reserve_bytes()
            if room0 is not None and room0 < need0:
                raise MemoryError('host memory headroom {:.0f} GB < {:.0f} GB needed to stage the inputs (pinned blocks '
                                  'come in powers of two) and keep a reserve'.format(room0 / 1e9, need0 / 1e9))
            memlog('before staging')
            host = stage_to_host(torch, X, y, theta)
            memlog('inputs staged')
            # free every device-resident tensor of the resident phase: the e2e step brings its own
            obj.X = obj.y = obj = None
            del X, y, st, H, hinv, w
            freed = True
            ops.free_workspaces()
            torch.cuda.empty_cache()
            e2e = run_e2e(args, vt, torch, dist, dev, group, world, host)
            memlog('after e2e')
            e2e['numa'] = numa_note
            e2e['host_memory_headroom_gb_before_staging'] = None if room0 is None else room0 / 1e9
        except Exception as exc:      # report, never hide
            e2e = {'value': None, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                   'error': repr(exc)[:300]}
        if e2e.get('value') and not args.no_e2e_full:
            # the (D, N) result needs as much host memory again as the inputs already staged (all ranks of the node
            # together); without clear headroom the leg is skipped - an out-of-memory kill would take the whole line
            need = world * pinned_cost(8 * n_loc * D) + host_reserve_bytes()
            room = host_headroom_bytes()
            ok = torch.tensor([1 if (room is None or room >= need) else 0], device=dev)
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 1:
                try:
                    e2e_full = run_e2e(args, vt, torch, dist, dev, group, world, host, full=True)
                except Exception as exc:      # report, never hide
                    e2e_full = {'value': None, 'unit': UNIT, 'error': repr(exc)[:300]}
            else:
                e2e_full = {'value': None, 'unit': UNIT,
                            'skipped': 'host memory headroom {:.0f} GB < {:.0f} GB needed to hold the (D, N) result next '
                                       'to the staged inputs'.format((room or 0) / 1e9, need / 1e9)}

    memlog('after e2e_full')
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = use_all_host_cores()
        n_s = args.cpu_sample if args.cpu_sample > 0 else cpu_sample_rows(args, cores, 8)    # ~20 s of CPU work
        sec = cpu_reference_step(n_s, D)
        cpu_baseline = {'value': n_s / sec, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                        'sample': '{} of {} observations, D={}; numpy closed-form assembly + '
                                  'cho_factor/cho_solve (oracle port of the reference path)'.format(n_s, N, D)}

    if want_rows and world == 1:
        # the other engines, in a child process with the device to itself (this process keeps only its context)
        import gc
        if not freed:
            obj.X = obj.y = obj = None
            del X, y, st, H, hinv, w
            freed = True
        host = None
        ops.free_workspaces()
        gc.collect()
        torch.cuda.empty_cache()
        cmd = [sys.executable, os.path.abspath(__file__), '--engine-rows-only', '--n-total', str(N), '--dim', str(D),
               '--steps', str(min(args.steps, 3)), '--warmup', '1', '--no-e2e', '--no-cpu-baseline', '--no-configs',
               '--precision', args.precision]
        try:
            child = subprocess.run(cmd, capture_output=True, text=True, timeout=1500)
            lines = [ln for ln in child.stdout.splitlines() if ln.startswith('{')]
            engine_rows = json.loads(lines[-1])['other_engines'] if lines else {
                'error': 'child exited with code {}: {}'.format(child.returncode, child.stderr[-300:])}
        except Exception as exc:              # report, never hide
            engine_rows = {'error': repr(exc)[:300]}

    # ---- BASELINE configs 3, 4, 5 (block-arrow factorisation, dense LR covariance, Taylor + CG), measured by the
    # same driver-run command on the same ranks; every device tensor of the headline legs is gone by now
    configs = None
    if not args.no_configs:
        try:
            import gc
            if not freed:
                obj.X = obj.y = obj = None
                del X, y, st, H, hinv, w
                freed = True
            host = None
            ops.free_workspaces()
            gc.collect()
            torch.cuda.empty_cache()
            sys.path.insert(0, os.path.join(ROOT, 'tools'))
            import bench_configs
            memlog('before configs')
            configs = bench_configs.run_all(dev, group, peak=peak_tflops)
            memlog('after configs')
        except Exception as exc:              # report, never hide
            configs = {'error': repr(exc)[:300]}

    if rank == 0:
        S_ = ops.OZAKI_SLICES
        nprod = S_ * (S_ + 1) // 2
        if engine == 'f64_ozaki':
            apply_tops = 2.0 * D * D * n_loc * nprod / (t_apply * 1e-3) / 1e12
            roofline = {
                'bound': 'tensor', 'kernel': 'ogemm_kernel<{}> + in-kernel slicing (vt_ij_apply_ozaki: S = -Hinv G^T on '
                                             'tcgen05.mma.kind::i8)'.format(S_),
                'achieved': apply_tops, 'peak': i8_peak['tops'], 'unit': 'TFLOP/s', 'frac': apply_tops / i8_peak['tops'],
                'unit_note': 'INT8 tera-operations per second (multiply + add = 2 ops), reported under the contract\'s '
                             'TFLOP/s key',
                'peak_source': 'bare tcgen05.mma.kind::i8 128x256x32 issue loop measured in this run for 1 s '
                               '(vt_i8_peak_probe: {:.0f} TOP/s, {:.1f} SM clocks per instruction; power-capped '
                               'clocks - the nominal 4500 TOP/s needs 1.86 GHz); MEASURED_PEAKS.json has no INT8 '
                               'entry'.format(i8_peak['tops'], i8_peak['clocks_per_mma']),
                'algorithmic': '{} exact digit products x 2*D^2 INT8 ops per observation ({} balanced base-256 slices '
                               'per operand); whole vt_ij_apply_ozaki call incl. slicing'.format(nprod, S_),
                'fp64_equivalent': {'achieved_tflops': apply_tflops, 'fp64_dmma_peak_tflops': peak_tflops,
                                    'ratio_to_fp64_pipe_peak': apply_tflops / peak_tflops,
                                    'algorithmic': '2*D^2 flop per observation'},
                'gemm_kernel_alone': gemm_alone,
                'traffic': traffic_i8,
                'traffic_source': 'profiles/ncu_traffic.json: dram__bytes_read+write of one ncu --set full launch of '
                                  'ogemm_kernel<7> (GEMM of a 37888-row chunk + in-kernel slicing of the next), scaled per '
                                  'observation to the whole call; algorithmic = 30*D bytes/obs (8D x_n + 7D digits written '
                                  '+ 7D digits read + 8D S_n)',
            }
        else:
            roofline = {'bound': 'tensor', 'kernel': 'dgemm_kernel<KC,KC> (vt_ij_apply: S = -Hinv G^T)',
                        'achieved': apply_tflops, 'peak': peak_tflops, 'unit': 'TFLOP/s',
                        'frac': apply_tflops / peak_tflops,
                        'peak_source': 'FP64 DMMA probe measured in this run (vt_fp64_peak_probe); '
                                       'MEASURED_PEAKS.json has no FP64 entry; tools/fp64_peak.cu gave '
                                       '{} TFLOP/s'.format(FP64_PEAK_FALLBACK_TFLOPS),
                        'traffic': traffic,
                        'traffic_source': 'profiles/ncu_traffic.json: dram__bytes_read+write of one ncu --set full '
                                          'launch at N=1e6, scaled per observation; algorithmic = 16*D bytes/obs',
                        'algorithmic': '2*D^2 flop per observation'}
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None,
            'dtype': {'f64': 'f64', 'f64_ozaki': 'f64 (contractions: exact i8 digit products -> f64, error-free slicing)',
                      'tf32x3': 'tf32x3', 'tf32': 'tf32'}[engine], 'data': 'synthetic',
            'config': {'workload': 'logistic IJ N=10M D=1024 f64 (BASELINE configs[1])', 'n_obs': N, 'dim': D,
                       'precision': args.precision, 'engine': engine,
                       'sharding': 'observations over {} rank(s), one all-reduce of the DxD Hessian'.format(world),
                       'l2': 'inputs ({:.1f} GB per rank) exceed the 126 MB L2'.format(8.0 * n_loc * D / 1e9),
                       'grad_norm_at_opt': grad_norm, 'sampled_residual_rel': rel_resid,
                       'hessian_condition_number': kappa},
            'clocks': clocks,
            'gpu_launches': launches,
            'roofline': roofline,
            'kernels': {
                'ij_apply': {'ms': t_apply, 'fp64_equiv_tflops': apply_tflops, 'ratio_to_fp64_pipe_peak': apply_tflops / peak_tflops},
                'syrk_weighted': {'ms': t_syrk, 'fp64_equiv_tflops_algorithmic_D(D+1)': syrk_tflops,
                                  'ratio_to_fp64_pipe_peak': syrk_tflops / peak_tflops},
                'glm_stats': {'ms': t_stats, 'gb_per_s': stats_gbs,
                              'frac_hbm_peak': stats_gbs / peaks['hbm_gbs'] if 'hbm_gbs' in peaks else None},
                'potrf_plus_inverse': {'ms': t_chol},
                'fp64_dmma_peak_tflops': peak_tflops, 'int8_peak': i8_peak,
            },
            'cpu_baseline': cpu_baseline,
            'e2e': e2e,
            'e2e_full': e2e_full,
            'other_engines': engine_rows,
            'configs': configs,
        }
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


ENGINE_NOTES = {
    'f64': 'both contractions on the FP64 DMMA engine (mma.sync m8n8k4, cp.async ring) - the r01 default',
    'f64_ozaki': ('both contractions on tcgen05.mma.kind::i8: 7 balanced base-256 slices per operand (54 bits), 28 exact '
                  'INT8 products, INT32 accumulators in TMEM, FP64 recombination; statistics, Cholesky and inverse in '
                  'FP64; held to the same rtol 1e-8 bar as the FP64 DMMA path'),
    'f64_ozaki_s6': ('the INT8 slicing engine with 6 slices per operand (46 bits, 21 exact digit products; VT_OZAKI_SLICES=6): '
                     'still inside the rtol 1e-8 bar, about two digits less than the 7-slice default'),
    'tf32x3': 'both contractions on tcgen05.mma.kind::tf32 with a three-term hi/lo split; the rest in FP64',
    'tf32': 'both contractions on tcgen05.mma.kind::tf32 (TMEM accumulators, TMA operands); the rest in FP64',
}
ENGINE_TOL = {'f64': 1e-8, 'f64_ozaki': 1e-8, 'tf32x3': 2e-4, 'tf32': 5e-3}


def engine_row(prec, vt, ops, torch, dist, world, group, dev, X, y, theta, w, st, hinv, idx, S_cols64, N, D, n_loc, reps,
               timed, note_key=None):
    """One full step through the public API with GLMObjective(precision=prec), max over ranks, plus the
    two contraction kernels timed alone and the sampled-column error against the FP64 DMMA result."""
    o32 = vt.objectives.GLMObjective(X, y, family='logistic', group=group, precision=prec)
    t_step, sens32 = timed(lambda: vt.HyperparameterSensitivityLinearApproximation(o32, theta, w), reps)
    tms = torch.tensor([t_step], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    t_step = float(tms.item())
    S32 = sens32.get_dopt_dhyper()
    del sens32
    diff = torch.abs(S32[:, idx] - S_cols64)
    smax = torch.max(torch.abs(S_cols64))
    err_norm = float(torch.max(diff) / smax)
    # the parity bar of tests/conftest.py::assert_close: |diff| <= rtol |ref| + 1e-12 max|ref|, as the worst ratio
    bar = float(torch.max(diff / (1e-8 * torch.abs(S_cols64) + 1e-12 * smax)))
    t_ap, _ = timed(lambda: ops.ij_apply(hinv, X, st['resid'], out=S32, precision=prec), reps)
    row = {'value': N / (t_step * 1e-3), 'unit': UNIT, 'ms_per_step': t_step,
           'sampled_sens_err_vs_headline_engine': {'normwise': err_norm, 'worst_ratio_to_rtol1e-8_bar': bar},
           'tolerance': ('rtol 1e-8 elementwise + 1e-12 max|ref| floor (the FP64 parity bar)' if prec in ('f64', 'f64_ozaki')
                         else '{:g} normwise'.format(ENGINE_TOL[prec])),
           'within_tolerance': bool(bar <= 1.0) if prec in ('f64', 'f64_ozaki') else bool(err_norm <= ENGINE_TOL[prec]),
           'ij_apply_ms': t_ap, 'ij_apply_fp64_equiv_tflops': 2.0 * D * D * n_loc / (t_ap * 1e-3) / 1e12,
           'engine': ENGINE_NOTES[note_key or prec]}
    t_sy, _h = timed(lambda: ops.syrk_weighted(X, st['s'], precision=prec), reps)
    row.update({'syrk_ms': t_sy, 'syrk_fp64_equiv_tflops_algorithmic': float(D) * (D + 1) * n_loc / (t_sy * 1e-3) / 1e12})
    return row


DUMP_BYTES = 60 << 20          # the whole --dump-outputs directory stays under 64 MB
DUMP_MAX_COLUMNS = 4096


def dump_columns(n, d):
    """How many columns of the (D, N) sensitivity matrix --dump-outputs keeps: all up to 4096, fewer when D is so
    wide that they and the D x D Hessian would not fit in DUMP_BYTES."""
    return min(n, DUMP_MAX_COLUMNS, (DUMP_BYTES - 8 * d * d) // (8 * d))


def dump_outputs(out_dir, sens, torch, dist, world, rank, r0, n, dev):
    """--dump-outputs: what the caller of the last timed step receives, in float64.  hessian_at_opt.npy is the whole
    D x D Hessian; dopt_dhyper_sample.npy holds the columns of the (D, N) sensitivity matrix at dump_columns(N, D)
    observations drawn without replacement by numpy's RandomState(SEED), in increasing order, gathered from the ranks
    that hold them.  The inputs depend only on the arguments, so two builds can be compared file by file."""
    S = sens.get_dopt_dhyper()                   # this rank's (D, n_loc) block, on the device
    d, n_loc = S.shape
    cols = np.sort(np.random.RandomState(SEED).choice(n, dump_columns(n, d), replace=False))
    mine = (cols >= r0) & (cols < r0 + n_loc)
    sample = torch.zeros((d, len(cols)), dtype=torch.float64, device=dev)
    sample[:, torch.from_numpy(np.flatnonzero(mine)).to(dev)] = S[:, torch.from_numpy(cols[mine] - r0).to(dev)]
    if world > 1:
        dist.all_reduce(sample)                  # every column comes from exactly one rank; the others add zeros
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, 'hessian_at_opt.npy'), sens.get_hessian_at_opt().double().cpu().numpy())
        np.save(os.path.join(out_dir, 'dopt_dhyper_sample.npy'), sample.cpu().numpy())


def memlog(tag):
    """VT_BENCH_MEMLOG=1: available host memory at the stations of the run, on stderr (every rank)."""
    if os.environ.get('VT_BENCH_MEMLOG') != '1':
        return
    room = host_headroom_bytes()
    print('[mem] rank {} {:<28s} available {:.1f} GB'.format(os.environ.get('RANK', '0'), tag, (room or 0) / 1e9),
          file=sys.stderr, flush=True)


def stage_to_host(torch, X, y, theta):
    """Pinned host copies of this rank's inputs (set-up for the e2e leg)."""
    n_loc, D = X.shape
    X_host = torch.empty((n_loc, D), dtype=torch.float64, pin_memory=True)
    X_host.copy_(X)
    y_host = torch.empty(n_loc, dtype=torch.float64, pin_memory=True)
    y_host.copy_(y)
    w_host = torch.ones(n_loc, dtype=torch.float64).pin_memory()
    w1 = torch.ones(n_loc, dtype=torch.float64)
    w1[::7] = 0.0
    return dict(X=X_host, y=y_host, w=w_host, w1=w1.pin_memory(), theta=theta.cpu().pin_memory())


def pinned_cost(nbytes):
    """What a pinned tensor of `nbytes` takes from the host: torch's caching host allocator hands out blocks whose
    sizes are powers of two (82 GB of inputs occupy 128 GB; measured: 2 x 41 GB shards took 139 GB)."""
    n = int(nbytes)
    return 1 << max(n - 1, 1).bit_length()


def host_reserve_bytes():
    """Host memory that must stay free after a staging allocation (page cache, NCCL's shared segments, the driver's
    own processes on the box): a tenth of the machine, at least 16 GB."""
    try:
        import psutil
        return max(16 << 30, int(0.10 * psutil.virtual_memory().total))
    except Exception:
        return 32 << 30


def host_headroom_bytes():
    """Bytes of host memory this process may still take: the smaller of the system's available memory and the
    headroom of the memory cgroup it runs in (pinned pages count against both).  The e2e legs stage 82 GB of inputs
    - and e2e_full another 82 GB of results - in host memory; taking more than there is gets the whole process
    killed (and the bench line with it), so those legs check first and report why they were skipped."""
    avail = None
    try:
        import psutil
        avail = int(psutil.virtual_memory().available)
    except Exception:
        pass
    for lim_path, cur_path in (('/sys/fs/cgroup/memory.max', '/sys/fs/cgroup/memory.current'),
                               ('/sys/fs/cgroup/memory/memory.limit_in_bytes', '/sys/fs/cgroup/memory/memory.usage_in_bytes')):
        try:
            with open(lim_path) as f:
                lim = f.read().strip()
            with open(cur_path) as f:
                cur = int(f.read().strip())
            if lim != 'max' and int(lim) < (1 << 60):
                room = int(lim) - cur
                avail = room if avail is None else min(avail, room)
        except Exception:
            continue
    return avail


def numa_bind_to_gpu(local_rank):
    """Run this process (and first-touch its pinned staging memory) on the host NUMA node of its GPU, when the box
    exposes more than one node.  Returns a short description for the report."""
    try:
        nodes = [d for d in os.listdir('/sys/devices/system/node') if d.startswith('node') and d[4:].isdigit()]
        if len(nodes) < 2:
            return '{} NUMA node visible: nothing to bind'.format(len(nodes))
        import subprocess as sp
        q = sp.run(['nvidia-smi', '-i', str(local_rank), '--query-gpu=pci.bus_id', '--format=csv,noheader'],
                   capture_output=True, text=True).stdout.strip().lower()
        dom = q[4:] if q.startswith('0000') and len(q) > 12 else q          # 00000000:1B:00.0 -> 0000:1b:00.0
        with open('/sys/bus/pci/devices/{}/numa_node'.format(dom)) as f:
            node = int(f.read().strip())
        if node < 0:
            return 'GPU {} reports no NUMA node'.format(local_rank)
        with open('/sys/devices/system/node/node{}/cpulist'.format(node)) as f:
            cpus = set()
            for part in f.read().strip().split(','):
                lo, _, hi = part.partition('-')
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return 'NUMA node {} of GPU {} has no CPU this process may use'.format(node, local_rank)
        os.sched_setaffinity(0, allowed)
        return 'bound to NUMA node {} ({} CPUs) of GPU {}'.format(node, len(allowed), local_rank)
    except Exception as exc:
        return 'not bound: {!r}'.format(exc)[:160]


def run_e2e(args, vt, torch, dist, dev, group, world, host, full=False):
    """The same metric through the public API with HOST buffers: every step
    copies this rank's X, y, w and theta from pinned host memory to the device,
    runs the whole path, and reads the result summary (the linear-approximation
    prediction for a leave-k-out weight vector, D doubles, plus the D x D
    Hessian) back to the host.  full=False: the (D, N) sensitivity matrix itself
    stays on the device, as a user of an 82 GB result would keep it.  full=True:
    get_dopt_dhyper() is called as well and returns the whole matrix on the HOST
    (what the reference's get_dopt_dhyper returns, sensitivity_lib.py:230-231)."""
    X_host, y_host, w_host, w1_host, theta_host = host['X'], host['y'], host['w'], host['w1'], host['theta']
    n_loc, D = X_host.shape
    N = args.n_total
    h2d = (X_host.numel() + y_host.numel() + 2 * w_host.numel() + theta_host.numel()) * 8
    d2h = (D + D * D) * 8 + (D * n_loc * 8 if full else 0)

    def step():
        # host (pinned) buffers straight into the public API: GLMObjective starts chunked
        # asynchronous copies and the statistics + Hessian sweep runs behind them
        o = vt.objectives.GLMObjective(X_host, y_host, family='logistic', group=group, precision=args.precision)
        sens = vt.HyperparameterSensitivityLinearApproximation(o, theta_host, w_host)
        pred = sens.predict_opt_par_from_hyper_par(w1_host)      # D doubles, returned on the host
        hess = sens.get_hessian_at_opt()                         # D x D, returned on the host
        assert not pred.is_cuda and not hess.is_cuda
        if full:
            S_host = sens.get_dopt_dhyper()                      # (D, n_loc) on the host (pinned staging)
            assert not S_host.is_cuda and tuple(S_host.shape) == (D, n_loc)
            return pred, hess, S_host
        return pred, hess

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    out = step(); del out
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        out = step(); del out
    e1.record()
    barrier()
    wall = time.perf_counter() - t0
    ms = torch.tensor([max(e0.elapsed_time(e1), wall * 1e3)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms.item()) / args.e2e_steps
    res = {'value': N / (ms_step * 1e-3), 'unit': UNIT, 'ms_per_step': ms_step, 'steps': args.e2e_steps,
           'h2d_bytes_per_step': h2d * world, 'd2h_bytes_per_step': d2h * world,
           'api': 'HyperparameterSensitivityLinearApproximation(GLMObjective(host X, host y), theta, w)'
                  '.predict_opt_par_from_hyper_par(w1) + get_hessian_at_opt()' + (' + get_dopt_dhyper() -> host' if full else '')}
    if not full:
        # the bound of this leg: every rank's bare pinned H2D copy of its shard of X, all ranks at once
        Xd = torch.empty((n_loc, D), dtype=torch.float64, device=dev)
        Xd.copy_(X_host, non_blocking=True)
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        Xd.copy_(X_host, non_blocking=True)
        c1.record()
        barrier()
        cms = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(cms, op=dist.ReduceOp.MAX)
        del Xd
        agg = X_host.numel() * 8 * world / (float(cms.item()) * 1e-3) / 1e9
        res['h2d_ceiling'] = {'bare_pinned_copy_of_X_all_ranks_at_once_gb_per_s': agg, 'ms': float(cms.item()),
                              'e2e_h2d_gb_per_s': h2d * world / (ms_step * 1e-3) / 1e9,
                              'e2e_fraction_of_bare_copy_time': float(cms.item()) / ms_step}
    return res


if __name__ == '__main__':
    main()
