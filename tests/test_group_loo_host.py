"""CPU tests of leave-one-group-out cross-validation (``approximate_cv(groups=...)``): malformed labels are refused
before any device work, the oracle's closed forms against brute-force refits, and, over gloo at world sizes 2 and 3
with uneven shards, that the group starts, mean_loss and n_invalid equal the single-process values and that a group
straddling two ranks is refused on every rank."""
import os
import types

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import lgo_reference as lgo
from conftest import ROOT
from test_influence_host import _bare, _free_port


def _bare_grouped(n):
    obj = _bare(n, 3)
    obj._obj = types.SimpleNamespace(n_obs=n, group=None)     # no X, no device: device work would fail
    return obj


BAD_GROUPS = {
    'short': np.zeros(9, dtype=np.int64),
    'long': np.zeros(11, dtype=np.int64),
    '2d': np.zeros((10, 1), dtype=np.int64),
    'float': np.arange(10, dtype=np.float64),
    'bool': np.ones(10, dtype=bool),
    'strings': np.array(['a'] * 10),
    'decreasing': np.array([0, 0, 1, 1, 2, 1, 3, 3, 4, 4]),
    'torch float': torch.arange(10, dtype=torch.float64),
}


@pytest.mark.parametrize('name', sorted(BAD_GROUPS))
@pytest.mark.parametrize('method', ['ns', 'ij'])
def test_malformed_groups_are_refused_before_device_work(name, method):
    obj = _bare_grouped(10)
    with pytest.raises(ValueError):
        obj.approximate_cv(method, groups=BAD_GROUPS[name])
    with pytest.raises(ValueError):
        obj.loo_linear_predictor(method, groups=BAD_GROUPS[name])


def test_groups_of_more_than_32_rows_are_refused():
    obj = _bare_grouped(70)
    labels = np.repeat([0, 1, 2], [20, 33, 17])
    with pytest.raises(ValueError, match='33 rows'):
        obj.approximate_cv('ns', groups=labels)
    with pytest.raises(ValueError):
        obj.loo_linear_predictor('ij', groups=list(labels))


def test_group_starts_of_valid_labels():
    from vittles_b200.influence_lib import group_starts
    for labels in ([5, 5, 7, 9, 9, 9], np.array([5, 5, 7, 9, 9, 9], dtype=np.int32), torch.tensor([5, 5, 7, 9, 9, 9])):
        starts, lab = group_starts(labels, 6)
        assert starts.tolist() == [0, 2, 3, 6] and lab.dtype == torch.int64
    starts, _ = group_starts(np.repeat(np.arange(3), 32), 96)
    assert starts.tolist() == [0, 32, 64, 96]
    starts, _ = group_starts(np.zeros(0, dtype=np.int64), 0)
    assert starts.tolist() == [0]


# ---------------------------------------------------------------------------------------------------- the oracle ----
def _fit(family, n, d, seed, l2):
    from oracle import models
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, d))
    X[:, 0] = 1.0
    z0 = X @ (0.5 * rng.normal(size=d))
    if family == 'logistic':
        y = (rng.uniform(size=n) < 1 / (1 + np.exp(-z0))).astype(np.float64)
    elif family == 'poisson':
        y = rng.poisson(np.exp(np.clip(z0, -4, 2))).astype(np.float64)
    else:
        y = z0 + rng.normal(size=n)
    w = rng.uniform(0.5, 2.0, size=n)
    w[3] = 0.0
    return X, y, w, models.glm_newton(X, y, w, family, l2)


STARTS = np.array([0, 1, 4, 5, 11, 19, 20, 23, 31, 36, 40])


@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
@pytest.mark.parametrize('l2', [0.0, 0.1])
def test_oracle_group_predictors_against_refits(family, l2):
    """z^NS = X_R of one Newton step from theta_hat without the group; for the Gaussian family the exact
    leave-group-out optimum.  z^IJ = X_R (theta_hat + H^{-1} sum_{n in R} w_n r_n x_n).  Groups of one row give the
    leave-one-out forms."""
    from oracle import loo as oloo, models
    X, y, w, theta = _fit(family, 40, 4, seed=len(family) + 3, l2=l2)
    ref = lgo.group_loo(X, y, w, theta, STARTS, family, l2)
    cf = models.glm_closed_form(X, y, theta, w, family, l2)
    for a, b in zip(STARTS[:-1], STARTS[1:]):
        rows = np.arange(a, b)
        np.testing.assert_allclose(ref['z_ns'][rows], lgo.newton_step_without_rows(X, y, w, theta, rows, family, l2),
                                   rtol=1e-9, atol=1e-12)
        g = (w[rows] * cf['r'][rows]) @ X[rows]
        np.testing.assert_allclose(ref['z_ij'][rows], X[rows] @ (theta + np.linalg.solve(cf['hessian'], g)),
                                   rtol=1e-9, atol=1e-12)
        if family == 'gaussian':
            np.testing.assert_allclose(ref['z_ns'][rows], lgo.exact_lgo(X, y, w, rows, family, l2), rtol=1e-9,
                                       atol=1e-12)
    one = oloo.loo(X, y, w, theta, family, l2)
    single = lgo.group_loo(X, y, w, theta, np.arange(41), family, l2)
    for k in ('h', 'leverage', 'z_ij', 'z_ns'):
        np.testing.assert_allclose(single[k], one[k], rtol=1e-12, atol=1e-14)


def test_oracle_singular_group_is_nan():
    """Feature 3 is nonzero on the rows of one group only and l2 = 0: without the group the Hessian is singular."""
    from oracle import models
    X, y, w, _ = _fit('gaussian', 40, 4, seed=2, l2=0.0)
    X[:, 3] = 0.0
    X[5:11, 3] = np.linspace(1.0, 2.0, 6)
    theta = models.glm_newton(X, y, w, 'gaussian', 0.0)
    ref = lgo.group_loo(X, y, w, theta, STARTS, 'gaussian', 0.0)
    assert np.isnan(ref['z_ns'][5:11]).all()
    assert np.isfinite(np.delete(ref['z_ns'], np.arange(5, 11))).all()


# ---------------------------------------------------------------------------------------- gloo, uneven shards ----
def _labels(n):
    rng = np.random.default_rng(5)
    sizes = rng.integers(1, 33, size=n)
    return np.repeat(np.arange(sizes.size) * 3, sizes)[:n]


def _rows(n, labels):
    rng = np.random.default_rng(11)
    loss = rng.exponential(size=n)
    w = rng.uniform(0.0, 2.0, size=n)
    w[::7] = 0.0
    invalid = np.isin(labels, labels[[2, n // 2, n - 1]])      # whole groups
    loss[invalid] = np.nan
    return loss, w, invalid


def _cut_between_groups(labels, sizes):
    """Shard boundaries near the given sizes, moved forward to the next group boundary."""
    cuts, a = [], 0
    for s in sizes[:-1]:
        b = a + s
        while 0 < b < labels.size and labels[b] == labels[b - 1]:
            b += 1
        cuts.append(b)
        a = b
    bounds = [0] + cuts + [labels.size]
    return [bounds[i + 1] - bounds[i] for i in range(len(sizes))]


def _lgo_worker(rank, world, port, sizes, straddle, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from vittles_b200 import distributed as vd
    from vittles_b200.influence_lib import cv_totals, group_starts
    _, _, group = vd.init_from_env(backend='gloo')
    n = sum(sizes)
    labels = _labels(n)
    a = sum(sizes[:rank])
    b = a + sizes[rank]
    mine = labels[a:b].copy()
    if straddle and rank == 1:
        mine[0] = labels[a - 1]                                 # rank 1 continues the last group of rank 0
    try:
        starts, _ = group_starts(mine, b - a, group)
        err = ''
    except ValueError as e:
        starts, err = None, str(e)
    if not straddle:
        loss, w, invalid = _rows(n, labels)
        ml, nbad = cv_totals(torch.as_tensor(loss[a:b]), torch.as_tensor(w[a:b]), torch.as_tensor(invalid[a:b]), group)
        np.save(os.path.join(out_dir, 'lgo_rank{}.npy'.format(rank)), np.array([ml, nbad]))
        np.save(os.path.join(out_dir, 'lgo_starts{}.npy'.format(rank)), starts.numpy() + a)
    with open(os.path.join(out_dir, 'lgo_err{}.txt'.format(rank)), 'w') as f:
        f.write(err)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('sizes', [(300, 701), (100, 650, 251)])
def test_sharded_group_cv_matches_single_process(tmp_path, sizes):
    from oracle import loo as oloo
    from vittles_b200.influence_lib import cv_totals, group_starts
    n = sum(sizes)
    labels = _labels(n)
    sizes = _cut_between_groups(labels, list(sizes))
    world = len(sizes)
    mp.spawn(_lgo_worker, args=(world, _free_port(), sizes, False, str(tmp_path)), nprocs=world, join=True)
    loss, w, invalid = _rows(n, labels)
    ml, nbad = cv_totals(torch.as_tensor(loss), torch.as_tensor(w), torch.as_tensor(invalid))
    ml_ref, nbad_ref = oloo.mean_loss(loss, w, invalid)
    assert nbad == nbad_ref > 3
    np.testing.assert_allclose(ml, ml_ref, rtol=1e-14)
    starts, _ = group_starts(labels, n)
    merged = [0]
    for rank in range(world):
        got = np.load(os.path.join(str(tmp_path), 'lgo_rank{}.npy'.format(rank)))
        np.testing.assert_allclose(got[0], ml, rtol=1e-14)
        assert int(got[1]) == nbad
        assert open(os.path.join(str(tmp_path), 'lgo_err{}.txt'.format(rank))).read() == ''
        merged += np.load(os.path.join(str(tmp_path), 'lgo_starts{}.npy'.format(rank))).tolist()[1:]
    assert merged == starts.tolist()


@pytest.mark.parametrize('sizes', [(300, 701), (100, 650, 251)])
def test_straddling_group_is_refused_on_every_rank(tmp_path, sizes):
    labels = _labels(sum(sizes))
    sizes = _cut_between_groups(labels, list(sizes))
    world = len(sizes)
    mp.spawn(_lgo_worker, args=(world, _free_port(), sizes, True, str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        err = open(os.path.join(str(tmp_path), 'lgo_err{}.txt'.format(rank))).read()
        assert 'straddles' in err or 'malformed' in err, (rank, err)
