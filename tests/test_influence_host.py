"""CPU tests of the observation-influence API (``vittles_b200.influence_lib``): argument checks that run before any
device work, the exact merge of per-rank AMIP candidates (ties included) and, over gloo at world sizes 2 and 3 with
uneven shards, that the sharded AMIP selection equals the single-process one.  Also the numpy oracle
(``oracle/influence.py``) against brute force on a tiny problem."""
import itertools
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _bare(n_total, dim):
    """An ObservationInfluence with no device state: a call that touched the device would fail."""
    from vittles_b200 import ObservationInfluence
    obj = ObservationInfluence.__new__(ObservationInfluence)
    obj.n_total, obj.dim, obj.offset = n_total, dim, 0
    return obj


@pytest.mark.parametrize('max_drop', [-1, 11, 0.0, 1.5, -0.2, True, '3', None])
def test_max_drop_out_of_range_is_refused_before_device_work(max_drop):
    obj = _bare(10, 3)
    with pytest.raises(ValueError):
        obj.amip((np.ones(3), 1.0), max_drop=max_drop)


def test_max_drop_resolution():
    from vittles_b200.influence_lib import resolve_max_drop
    assert resolve_max_drop(0, 10) == 0
    assert resolve_max_drop(10, 10) == 10
    assert resolve_max_drop(np.int64(4), 10) == 4
    assert resolve_max_drop(1.0, 10) == 10
    assert resolve_max_drop(0.01, 1001) == 10
    assert resolve_max_drop(0.05, 10) == 0


@pytest.mark.parametrize('shape', [(0, 3), (4,), (2, 4), (1, 2), (3, 3, 1)])
def test_qoi_jacobian_of_the_wrong_shape_is_refused(shape):
    obj = _bare(10, 3)
    a = np.zeros(shape)
    with pytest.raises(ValueError):
        obj.influence(a)
    if len(shape) == 1 or shape[0] == 1:
        with pytest.raises(ValueError):
            obj.amip((a, 1.0), max_drop=2)


def test_non_glm_objective_is_not_implemented():
    from vittles_b200 import ObservationInfluence

    def f(theta, w):
        return (theta * theta).sum()

    with pytest.raises(NotImplementedError) as err:
        ObservationInfluence(f, np.zeros(3))
    assert 'HyperparameterSensitivityLinearApproximation' in str(err.value)
    assert 'get_dopt_dhyper' in str(err.value)


def test_merge_of_hand_made_candidates():
    from vittles_b200.influence_lib import merge_candidates, local_candidates
    # rank 0 holds rows 0..5, rank 1 rows 6..9: ties across and within ranks, padding (key 0, index -1)
    k0 = torch.tensor([3.0, 1.0, 0.0, 3.0, -2.0, 2.0], dtype=torch.float64)
    k1 = torch.tensor([3.0, 2.0, 5.0, 1.0], dtype=torch.float64)
    a_k, a_i = local_candidates(k0, 0, 4)
    b_k, b_i = local_candidates(k1, 6, 4)
    assert a_i.tolist() == [0, 3, 5, 1] and a_k.tolist() == [3.0, 3.0, 2.0, 1.0]
    assert b_i.tolist() == [8, 6, 7, 9]
    pad_k = torch.cat([b_k, torch.zeros(1, dtype=torch.float64)])
    pad_i = torch.cat([b_i, torch.tensor([-1])])
    for m in range(0, 8):
        k, i = merge_candidates([a_k, pad_k], [a_i, pad_i], m)
        assert i.tolist() == [8, 0, 3, 6, 5, 7, 1, 9][:m], m
        assert k.tolist() == [5.0, 3.0, 3.0, 3.0, 2.0, 2.0, 1.0, 1.0][:m]
    # the order of the lists does not matter
    k, i = merge_candidates([pad_k, a_k], [pad_i, a_i], 8)
    assert i.tolist() == [8, 0, 3, 6, 5, 7, 1, 9]


def test_amip_from_scores_matches_the_oracle():
    from vittles_b200.influence_lib import amip_from_scores
    from oracle import influence as oinf
    rng = np.random.default_rng(3)
    score = np.round(rng.normal(size=400), 2)                 # many exact ties
    score[::7] = 0.0
    for value, target, m in [(1.0, 0.0, 40), (-1.0, 0.0, 40), (1.0, 0.5, 400), (3.0, -100.0, 25), (0.0, 0.0, 5),
                             (-2.0, 1.0, 0)]:
        got = amip_from_scores(torch.as_tensor(score), value, target, m)
        ref = oinf.amip_greedy(score, value, target, m)
        assert got.n_drop == ref['n_drop']
        assert got.indices.tolist() == ref['indices'].tolist()
        assert got.predicted_value == ref['predicted_value']
        assert got.max_change == ref['max_change']
        assert got.direction == ref['direction']


def test_oracle_against_brute_force():
    """psi against central differences of the refitted optimum, the greedy selection against every subset, and the
    refit against Newton with zero weights."""
    from oracle import influence as oinf, models
    n, d = 9, 3
    X, y, _ = models.synth_logistic(11, n, d)
    X = X * 3.0
    w = np.linspace(0.5, 1.5, n)
    l2 = 0.1
    theta = models.glm_newton(X, y, w, l2=l2)
    A = np.array([[1.0, 0.0, 0.0], [0.3, -1.0, 2.0]])
    psi = oinf.psi(X, y, w, theta, A, l2=l2)
    h = 1e-5
    for j in range(n):
        wp, wm = w.copy(), w.copy()
        wp[j] += h
        wm[j] -= h
        fd = (models.glm_newton(X, y, wp, l2=l2) - models.glm_newton(X, y, wm, l2=l2)) / (2 * h)
        np.testing.assert_allclose(psi[:, j], A @ fd, rtol=1e-6, atol=1e-9)
    score = w * psi[0]
    value = float(theta[0])
    for target in (0.0, value - 0.5 * np.sign(value), value + 0.2):
        ref = oinf.amip_greedy(score, value, target, n)
        sign = 1.0 if value >= target else -1.0
        best = None
        for m in range(1, n + 1):
            top = max(sum(score[list(c)]) * sign for c in itertools.combinations(range(n), m))
            pred = value - sign * top
            if (pred <= target) if sign > 0 else (pred >= target):
                best = m
                break
        assert ref['n_drop'] == best, (target, ref['n_drop'], best)
    drop = [2, 5]
    w0 = w.copy()
    w0[drop] = 0.0
    np.testing.assert_allclose(oinf.refit(X, y, w, drop, l2=l2), models.glm_newton(X, y, w0, l2=l2), rtol=1e-10)


# ---------------------------------------------------------------------------------------- gloo, uneven shards ----
def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _scores(n):
    """Scores with exact ties (also across ranks) and zero-weight rows."""
    rng = np.random.default_rng(7)
    s = np.round(rng.normal(size=n), 2)
    s[::5] = 0.0
    return s


def _amip_worker(rank, world, port, sizes, cases, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    from vittles_b200 import distributed as vd
    from vittles_b200.influence_lib import amip_from_scores, row_offset
    _, _, group = vd.init_from_env(backend='gloo')
    offset, n_total = row_offset(sizes[rank], group)
    assert offset == sum(sizes[:rank]) and n_total == sum(sizes)
    score = torch.as_tensor(_scores(n_total)[offset:offset + sizes[rank]])
    res = {}
    for c, (value, target, m) in enumerate(cases):
        r = amip_from_scores(score, value, target, m, offset, group)
        res['n{}'.format(c)] = np.array(-1 if r.n_drop is None else r.n_drop)
        res['i{}'.format(c)] = r.indices
        res['p{}'.format(c)] = np.array([r.predicted_value, r.max_change])
    np.savez(os.path.join(out_dir, 'amip_rank{}.npz'.format(rank)), **res)
    dist.barrier()
    dist.destroy_process_group()


CASES = [(1.0, 0.0, 60), (-1.0, 0.0, 60), (2.0, 1.5, 300), (0.5, -50.0, 30), (-0.3, 0.2, 1)]


@pytest.mark.parametrize('sizes', [(300, 701), (100, 650, 251)])
def test_sharded_amip_selection_matches_single_process(tmp_path, sizes):
    from vittles_b200.influence_lib import amip_from_scores
    world = len(sizes)
    mp.spawn(_amip_worker, args=(world, _free_port(), list(sizes), CASES, str(tmp_path)), nprocs=world, join=True)
    score = torch.as_tensor(_scores(sum(sizes)))
    for rank in range(world):
        got = np.load(os.path.join(str(tmp_path), 'amip_rank{}.npz'.format(rank)))
        for c, (value, target, m) in enumerate(CASES):
            ref = amip_from_scores(score, value, target, m)
            assert int(got['n{}'.format(c)]) == (-1 if ref.n_drop is None else ref.n_drop), (rank, c)
            assert got['i{}'.format(c)].tolist() == ref.indices.tolist(), (rank, c)
            assert got['p{}'.format(c)].tolist() == [ref.predicted_value, ref.max_change], (rank, c)
