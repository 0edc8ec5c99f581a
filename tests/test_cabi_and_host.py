"""CPU: the C-ABI library loads and exports every symbol the header declares;
host-side logic that needs no GPU (term bookkeeping, argument validation, the
fail-loudly rule)."""
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT


def test_library_exports_every_declared_symbol():
    from vittles_b200 import _cabi
    header = open(os.path.join(ROOT, 'include', 'vittles_b200.h')).read()
    declared = set(re.findall(r'\b(vt_[a-z0-9_]+)\s*\(', header))
    assert len(declared) >= 30
    lib = _cabi.load()                                   # no GPU needed to load and type the entry points
    for name in declared:
        assert hasattr(lib, name), 'library does not export ' + name
    assert declared == set(_cabi.exported_symbols()), declared ^ set(_cabi.exported_symbols())
    assert isinstance(lib.vt_last_error(), bytes)
    # inverted 128-blocks + scratch panel + flags + inverted 256-blocks + (D >= 1024) inverted 512-blocks + solve scratch + split-K tiles of the solve (148 SMs assumed without a GPU) + second panel (look-ahead)
    head = 8 * 128 * 128 + 1024 * 128 + 10 + 4 * 256 * 256 + 2 * 512 * 512 + 512 * 512
    assert lib.vt_potrf_dinv_doubles(1024) == (head + 31) // 32 * 32 + 2 * 148 * 128 * 128 + 1024 * 128
    assert lib.vt_potrf_dinv_doubles(130) == 2 * 128 * 128 + 130 * 128 + 4 + 1 * 256 * 256 + 130 * 128


def test_abi_version():
    """Version 2: vt_ozaki_slice_t takes no selector of the instruction sequence, and only vt_ozaki_slice slices rows."""
    from vittles_b200 import _cabi
    assert _cabi.load().vt_abi_version() == 2


def test_no_cpu_fallback():
    """Without a CUDA device every compute entry fails loudly."""
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    import vittles_b200 as vt
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        vt.solver_lib.get_cholesky_solver(np.eye(3))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        vt.objectives.GLMObjective(np.ones((4, 2)), np.ones(4))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        vt.HyperparameterSensitivityLinearApproximation(lambda t, l: (t * l).sum(), np.ones(2), np.ones(2))


def test_product_never_imports_the_oracle():
    import subprocess, sys
    code = ("import sys; sys.path.insert(0, %r); import vittles_b200; "
            "bad=[m for m in sys.modules if m == 'oracle' or m.startswith('oracle.')]; assert not bad, bad" % ROOT)
    subprocess.check_call([sys.executable, '-c', code])
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'vittles_b200')):
        for fn in files:
            if fn.endswith('.py'):
                src = open(os.path.join(dirpath, fn)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', src, re.M), fn


def test_derivative_terms_host_logic(golden):
    """tests/test_sensitivity_lib.py:354-401 (differentiate / consolidate)."""
    from vittles_b200 import sensitivity_lib as sl
    t = sl.DerivativeTerm(eps_order=1, eta_orders=[1, 0], prefactor=2.0)
    assert t.order() == 2 and t.total_eta_order == 1
    kids = t.differentiate()
    assert len(kids) == 3                                                          # reference :363-381
    sig = sorted((k.eps_order, tuple(k.eta_orders), k.prefactor) for k in kids)
    assert sig == [(1, (0, 1, 0), 2.0), (1, (2, 0, 0), 2.0), (2, (1, 0, 0), 2.0)]
    a = sl.DerivativeTerm(0, [1], 1.0)
    merged = sl._consolidate_terms([a, sl.DerivativeTerm(0, [1], 2.5), sl.DerivativeTerm(1, [0], 1.0)])
    assert len(merged) == 2 and merged[0].prefactor == 3.5                         # reference :384-401
    assert a.check_similarity(sl.DerivativeTerm(0, [1], 9.0))
    assert str(a).startswith('Order: 1')
    with pytest.raises(AssertionError):
        sl.DerivativeTerm(0, [1, 1], 1.0)          # len(eta_orders) must equal the order
    g = golden('taylor')
    terms = [sl._get_taylor_base_terms()]
    for k in range(1, 5):
        nxt = []
        for term in terms[-1]:
            nxt += term.differentiate()
        terms.append(sl._consolidate_terms(nxt))
    for k in range(5):
        ref = {(int(r[1]), tuple(int(x) for x in r[2:2 + k + 1])): r[0] for r in g['table_order{}'.format(k + 1)]}
        assert {(t.eps_order, tuple(t.eta_orders)): t.prefactor for t in terms[k]} == ref

    # _evaluate_term_fwd expands the directions as the reference does (:720-734)
    calls = []

    def fake_eval(eta0, eps0, eta_dirs, eps_dirs, validate=False):
        calls.append((list(eta_dirs), list(eps_dirs)))
        return 1.0
    term = sl.DerivativeTerm(eps_order=2, eta_orders=[1, 0, 1, 0, 0, 0], prefactor=3.0)
    out = sl._evaluate_term_fwd(term, 'e0', 'p0', 'D', ['d1', 'd2', 'd3', 'd4', 'd5'], fake_eval)
    assert out == 3.0 and calls[0] == (['d1', 'd3'], ['D', 'D'])
    with pytest.raises(ValueError):
        sl._evaluate_term_fwd(term, 'e0', 'p0', 'D', ['d1'], fake_eval, validate=True)


def test_shard_ranges():
    from vittles_b200.distributed import shard_range
    for n, w in [(10_000_000, 8), (1000, 3), (7, 8)]:
        pieces = [shard_range(n, r, w) for r in range(w)]
        assert pieces[0][0] == 0 and pieces[-1][1] == n
        assert all(pieces[i][1] == pieces[i + 1][0] for i in range(w - 1))
        sizes = [b - a for a, b in pieces]
        assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(10, 3, 2)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the CPU arm) prints one JSON line."""
    import json, subprocess, sys
    out = subprocess.check_output([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1',
                                   '--warmup', '1', '--cpu-sample', '2000', '--dim', '64'], text=True)
    line = json.loads(out.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['value'] > 0 and line['cpu_baseline']['kind'] == 'port'
    assert line['e2e']['h2d_bytes_per_step'] == 0


def test_block_arrow_detection_host_logic():
    """detect_block_arrow (SURVEY 8f item 3): recovers the blocks of a permuted block-arrow COO
    matrix, sums duplicate entries, and rejects matrices without that structure."""
    import scipy.sparse
    from vittles_b200.sparse_hessian_lib import detect_block_arrow
    rng = np.random.RandomState(0)
    G, M, Dg = 40, 5, 90
    d = G * M + Dg
    perm = rng.permutation(d)
    sa, gi = perm[:G * M].reshape(G, M), np.sort(perm[G * M:])
    dense = np.zeros((d, d))
    blocks = rng.normal(size=(G, M, M))
    blocks = blocks + blocks.transpose(0, 2, 1) + 10 * np.eye(M)
    cross = rng.normal(size=(G, M, Dg))
    hgg = rng.normal(size=(Dg, Dg))
    hgg = hgg + hgg.T
    for g in range(G):
        dense[np.ix_(sa[g], sa[g])] = blocks[g]
        dense[np.ix_(sa[g], gi)] = cross[g]
        dense[np.ix_(gi, sa[g])] = cross[g].T
    dense[np.ix_(gi, gi)] = hgg
    coo = scipy.sparse.coo_matrix(dense)
    # duplicates: split every value into two halves, as the reference's assembly does (:147-153)
    dup = scipy.sparse.coo_matrix((np.concatenate([coo.data / 2, coo.data / 2]),
                                   (np.concatenate([coo.row, coo.row]), np.concatenate([coo.col, coo.col]))), (d, d))
    for mat in (coo, dup):
        sa2, gi2, b2, c2, h2 = detect_block_arrow(mat)
        assert np.array_equal(gi2, gi)
        rebuilt = np.zeros((d, d))
        for g in range(sa2.shape[0]):
            rebuilt[np.ix_(sa2[g], sa2[g])] = b2[g]
            rebuilt[np.ix_(sa2[g], gi2)] = c2[g]
            rebuilt[np.ix_(gi2, sa2[g])] = c2[g].T
        rebuilt[np.ix_(gi2, gi2)] = h2
        np.testing.assert_allclose(rebuilt, dense, rtol=0, atol=1e-15)
        assert sa2.shape == (G, M)
    r = scipy.sparse.random(80, 80, density=0.1, random_state=2)
    assert detect_block_arrow((r @ r.T + scipy.sparse.eye(80)).tocoo()) is None
    ragged = scipy.sparse.block_diag([np.ones((3, 3)), np.ones((4, 4))])
    assert detect_block_arrow(ragged) is None


def test_engine_selection_host_logic():
    """precision= is validated on the host before anything touches a device; workspace queries of the
    tensor-core engines need no GPU and grow the way the chunked drivers slice."""
    import vittles_b200 as vt
    from vittles_b200 import _cabi, ops
    assert ops._split('f64') == 0 and ops._split('f64_ozaki') == 0 and ops._split('tf32') == 1 and ops._split('tf32x3') == 3
    with pytest.raises(ValueError, match='precision'):
        ops._split('bf16')
    with pytest.raises(ValueError, match='precision'):
        vt.objectives.GLMObjective(np.ones((4, 2)), np.ones(4), precision='fp16')
    assert ops.OZAKI_SLICES in (6, 7, 8)
    lib = _cabi.load()
    # INT8 engine: slices of H^-1 + two chunk buffers of X slices (chunk: a whole number of 64-row tiles, < 64K rows)
    small = lib.vt_ij_apply_ozaki_workspace_bytes(1000, 1024, 8)
    big = lib.vt_ij_apply_ozaki_workspace_bytes(10_000_000, 1024, 8)
    assert 8 * 1024 * 1024 < small < big < (1 << 30)
    assert lib.vt_ij_apply_ozaki_workspace_bytes(10_000_000, 1024, 7) < big
    # Hessian assembly: N doubles of sqrt(s) + two chunk buffers + split-K partial Hessians
    w = lib.vt_syrk_ozaki_workspace_bytes(10_000_000, 1024, 8)
    assert 8 * 10_000_000 < w < (1 << 30)
    # TF32 engine: FP32 copies of one chunk (x2 for the hi/lo split)
    t1 = lib.vt_ij_apply_tf32_workspace_bytes(10_000_000, 1024, 1)
    t3 = lib.vt_ij_apply_tf32_workspace_bytes(10_000_000, 1024, 3)
    assert 0 < t1 < (1 << 29) and t1 < t3 < (1 << 30)
    assert lib.vt_syrk_tf32_workspace_bytes(10_000_000, 1024, 1) > 0
    assert lib.vt_tf32_gemm_workspace_bytes(1024, 1024, 1 << 20, 1) > 0     # long K: split-K partial tiles
    assert lib.vt_tf32_gemm_workspace_bytes(1024, 1 << 20, 1024, 1) == 0    # many tiles, short K: direct epilogue


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs next to ours) on a tiny shape: one JSON line with the
    contract's keys, all host cores in use even when OMP_NUM_THREADS=1 is exported (as torch.distributed.run does)."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, OMP_NUM_THREADS='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dim', '16',
                          '--cpu-sample', '3000', '--steps', '2', '--warmup', '1'], capture_output=True, text=True,
                         env=env, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['steps'] == 2 and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    ncores = len(os.sched_getaffinity(0))
    assert d['cpu_baseline']['cores'] == ncores or ncores > 64      # every core, whatever OMP_NUM_THREADS says
    # rank != 0 of a torchrun job exits quietly
    out2 = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dim', '16',
                           '--cpu-sample', '3000'], capture_output=True, text=True, env=dict(env, RANK='1', WORLD_SIZE='2'),
                          timeout=120)
    assert out2.returncode == 0 and out2.stdout.strip() == ''


def test_bench_host_memory_accounting():
    """The e2e legs of bench.py stage tens of GB in pinned host memory; their guards must count what torch's
    caching host allocator really takes (powers of two) and keep a reserve - an over-committed pinned allocation
    does not raise, it gets every rank killed (seen at 2 GPUs on a 251 GB host)."""
    import importlib.util
    import sys
    spec = importlib.util.spec_from_file_location('bench_for_test', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    argv = sys.argv
    sys.argv = ['bench.py']
    try:
        spec.loader.exec_module(bench)
    finally:
        sys.argv = argv
    GB = 1 << 30
    assert bench.pinned_cost(82 * 10 ** 9) == 128 * GB           # the inputs of the headline config on one GPU
    assert bench.pinned_cost(41 * 10 ** 9) == 64 * GB            # ... and per rank on two
    assert bench.pinned_cost(64 * GB) == 64 * GB and bench.pinned_cost(64 * GB + 1) == 128 * GB
    assert bench.host_reserve_bytes() >= 16 * GB
    room = bench.host_headroom_bytes()
    assert room is None or room > 0
    # --dump-outputs: the headline shape keeps 4096 sampled columns, and no accepted --dim goes over 64 MB
    assert bench.dump_columns(10_000_000, 1024) == 4096 and bench.dump_columns(1000, 16) == 1000
    for d in (1, 1024, 2048, 2700, 2800):
        k = bench.dump_columns(10_000_000, d)
        assert k < 1 or 8 * d * (d + k) + 2 * 128 <= 64 * 10 ** 6


def test_bench_rejects_bad_arguments(tmp_path):
    """--steps is the number of timed steps, so at least one; --dump-outputs belongs to the GPU path and needs room
    for the Hessian.  Each is refused before any work starts."""
    import subprocess
    import sys
    for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', str(tmp_path)],
                  ['--dim', '4096', '--dump-outputs', str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True,
                             timeout=120)
        assert out.returncode == 2 and 'error:' in out.stderr, (extra, out.stderr[-300:])
    assert os.listdir(str(tmp_path)) == []
