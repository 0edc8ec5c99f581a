"""CPU tests of approximate leave-one-out cross-validation (``ObservationInfluence.approximate_cv``): the method is
refused before any device work, the torch predictors and losses against the numpy oracle, the oracle's closed forms
against brute force (a one-step Newton refit without the row; for the Gaussian family the exact leave-one-out
refit), and, over gloo at world sizes 2 and 3 with uneven shards, that mean_loss and n_invalid equal the
single-process values."""
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from conftest import ROOT
from test_influence_host import _bare, _free_port


@pytest.mark.parametrize('method', ['NS', 'exact', '', None, 1])
def test_method_is_refused_before_device_work(method):
    obj = _bare(10, 3)
    with pytest.raises(ValueError):
        obj.approximate_cv(method)
    with pytest.raises(ValueError):
        obj.loo_linear_predictor(method)


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


@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
@pytest.mark.parametrize('l2', [0.0, 0.1])
def test_oracle_predictors_against_refits(family, l2):
    """z^NS = x_n^T of one Newton step from theta_hat without row n; for the Gaussian family that step lands on
    the exact leave-one-out optimum.  z^IJ = x_n^T (theta_hat + H^{-1} w_n r_n x_n)."""
    from oracle import loo as oloo, models
    X, y, w, theta = _fit(family, 40, 4, seed=len(family), l2=l2)
    ref = oloo.loo(X, y, w, theta, family, l2)
    cf = models.glm_closed_form(X, y, theta, w, family, l2)
    for n in range(X.shape[0]):
        ns = oloo.newton_step_without(X, y, w, theta, n, family, l2)
        np.testing.assert_allclose(ref['z_ns'][n], ns, rtol=1e-9, atol=1e-12)
        ij = X[n] @ (theta + np.linalg.solve(cf['hessian'], w[n] * cf['r'][n] * X[n]))
        np.testing.assert_allclose(ref['z_ij'][n], ij, rtol=1e-9, atol=1e-12)
        if family == 'gaussian':
            np.testing.assert_allclose(ref['z_ns'][n], oloo.exact_loo(X, y, w, n, family, l2), rtol=1e-9, atol=1e-12)
    assert np.all((ref['leverage'] >= 0) & (ref['leverage'] < 1))


@pytest.mark.parametrize('family', ['logistic', 'poisson', 'gaussian'])
def test_torch_closed_forms_match_the_oracle(family):
    from oracle import loo as oloo, models
    from vittles_b200.influence_lib import cv_totals, glm_loss, loo_predictor
    X, y, w, theta = _fit(family, 60, 5, seed=9, l2=0.1)
    X[:, 4] = 0.0
    X[5, 4] = 1.0                         # feature 4 carries row 5 alone: with l2 = 0 its Newton step is undefined
    theta = models.glm_newton(X, y, w, family, 0.0)
    ref = oloo.loo(X, y, w, theta, family, 0.0)
    cf = models.glm_closed_form(X, y, theta, w, family, 0.0)
    t = {k: torch.as_tensor(v) for k, v in dict(z=cf['z'], r=cf['r'], s=cf['s'], w=w, h=ref['h'], y=y).items()}
    for method, zr in (('ns', ref['z_ns']), ('ij', ref['z_ij'])):
        z = loo_predictor(t['z'], t['r'], t['s'], t['w'], t['h'], method)
        np.testing.assert_array_equal(np.isnan(z.numpy()), np.isnan(zr))
        np.testing.assert_allclose(z.numpy(), zr, rtol=1e-14, equal_nan=True)
        loss = glm_loss(z, t['y'], family)
        np.testing.assert_allclose(loss.numpy(), oloo.glm_loss(zr, y, family), rtol=1e-13, equal_nan=True)
        ml, nbad = cv_totals(loss, t['w'], torch.isnan(z))
        ml_ref, nbad_ref = oloo.mean_loss(oloo.glm_loss(zr, y, family), w, np.isnan(zr))
        assert nbad == nbad_ref == (1 if method == 'ns' else 0)
        np.testing.assert_allclose(ml, ml_ref, rtol=1e-13)


def test_logistic_loss_is_stable_in_both_tails():
    from vittles_b200.influence_lib import glm_loss
    z = torch.tensor([-800.0, -40.0, 0.0, 40.0, 800.0], dtype=torch.float64)
    for y in (0.0, 1.0):
        got = glm_loss(z, torch.full_like(z, y), 'logistic').numpy()
        ref = np.logaddexp(0.0, z.numpy()) - y * z.numpy()
        np.testing.assert_allclose(got, ref, rtol=1e-15)


# ---------------------------------------------------------------------------------------- gloo, uneven shards ----
def _rows(n):
    """Losses, weights (zeros included) and invalid rows of a global problem."""
    rng = np.random.default_rng(11)
    loss = rng.exponential(size=n)
    w = rng.uniform(0.0, 2.0, size=n)
    w[::7] = 0.0
    invalid = np.zeros(n, dtype=bool)
    invalid[[2, n // 2, n - 1]] = True
    loss[invalid] = np.nan
    return loss, w, invalid


def _cv_worker(rank, world, port, sizes, out_dir):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    from vittles_b200 import distributed as vd
    from vittles_b200.influence_lib import cv_totals
    _, _, group = vd.init_from_env(backend='gloo')
    loss, w, invalid = _rows(sum(sizes))
    a = sum(sizes[:rank])
    b = a + sizes[rank]
    ml, nbad = cv_totals(torch.as_tensor(loss[a:b]), torch.as_tensor(w[a:b]), torch.as_tensor(invalid[a:b]), group)
    np.save(os.path.join(out_dir, 'cv_rank{}.npy'.format(rank)), np.array([ml, nbad]))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize('sizes', [(300, 701), (100, 650, 251)])
def test_sharded_mean_loss_matches_single_process(tmp_path, sizes):
    from oracle import loo as oloo
    from vittles_b200.influence_lib import cv_totals
    world = len(sizes)
    mp.spawn(_cv_worker, args=(world, _free_port(), list(sizes), str(tmp_path)), nprocs=world, join=True)
    loss, w, invalid = _rows(sum(sizes))
    ml, nbad = cv_totals(torch.as_tensor(loss), torch.as_tensor(w), torch.as_tensor(invalid))
    ml_ref, nbad_ref = oloo.mean_loss(loss, w, invalid)
    assert nbad == nbad_ref == 3
    np.testing.assert_allclose(ml, ml_ref, rtol=1e-14)
    for rank in range(world):
        got = np.load(os.path.join(str(tmp_path), 'cv_rank{}.npy'.format(rank)))
        np.testing.assert_allclose(got[0], ml, rtol=1e-14)
        assert int(got[1]) == nbad
