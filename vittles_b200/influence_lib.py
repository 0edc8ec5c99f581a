"""Per-observation influence on quantities of interest, and dropped-data robustness (AMIP), for GLM objectives.

For weighted GLM objectives the infinitesimal jackknife is ``S = d theta_hat / d w = -H^{-1} G^T`` with column n
equal to ``-resid_n H^{-1} x_n``.  Users of the IJ usually want the effect of the weights on a few quantities of
interest phi_k(theta) rather than S itself:

    psi[k, n] = d phi_k(theta_hat(w)) / d w_n = a_k^T S[:, n] = -resid_n x_n . v_k,   v_k = H^{-1} a_k,  a_k = grad phi_k

That is K solves against the Cholesky factor of H and one pass over X that writes K values per observation
(``ops.glm_influence``); nothing of size D x N is formed, so the (D, N) matrix of
``HyperparameterSensitivityLinearApproximation`` and its memory are never needed.

Approximate leave-one-out cross-validation (:meth:`ObservationInfluence.approximate_cv`) needs one scalar per
observation, h_n = x_n^T H^{-1} x_n = |L^{-1} x_n|^2 (``ops.quad_forms``: a sum of squares, N D^2 / 2 multiply-adds
on the tensor cores).  With the statistics r_n = b'(z_n) - y_n and s_n = w_n b''(z_n) at theta_hat:

    leverage_n = s_n h_n
    z_n^IJ = z_n + w_n r_n h_n                          (x_n^T of predict_opt_par_without([n]))
    z_n^NS = z_n + w_n r_n h_n / (1 - s_n h_n)          (one Newton step from theta_hat without row n)

The Newton-step ("ALO") form equals the exact leave-one-out prediction for the Gaussian family.

With ``groups`` (one integer label per row, non-decreasing; a group is one label of at most 32 rows, all on one
rank), the same methods leave out whole groups.  For the rows R of a group, Q = X_R H^{-1} X_R^T, u = (w r)_R and
S = diag(s_R) (``ops.group_loo``: the rows of U = L^{-1} X^T as for h_n, then a per-group Gram and solve):

    z_R^IJ = z_R + Q u                                  (X_R of predict_opt_par_without(R))
    z_R^NS = z_R + t + Q S^1/2 M^{-1} S^1/2 t,  t = Q u,  M = I - S^1/2 Q S^1/2

which is z_R + X_R H_{-R}^{-1} X_R^T u by Woodbury (one Newton step without the group; exact for the Gaussian
family).  At groups of one row both reduce to the leave-one-out forms.

On top of psi, :meth:`ObservationInfluence.amip` computes the Approximate Maximum Influence Perturbation of
Broderick, Giordano & Meager: the smallest set of observations whose removal is predicted to move a quantity of
interest to a target (zero: a sign change), and :meth:`ObservationInfluence.refit` re-optimises without that set to
check the prediction.

Observation sharding: with ``objective.group`` set, every rank holds a contiguous block of rows, in rank order (the
layout ``distributed.shard_range`` produces).  Global observation indices are the local ones plus the exclusive
prefix sum of the ranks' row counts.  ``influence`` stays sharded; the AMIP selection is merged exactly (see
:func:`merge_candidates`).
"""
import math
import warnings
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch
import torch.distributed as dist

from . import ops, solver_lib
from ._arrays import to_device, kind_of, as_kind
from .objectives import GLMObjective


def _world(group):
    if group is None or not dist.is_initialized():
        return 1
    return dist.get_world_size(group)


def _all_gather(t, group):
    """The tensors of every rank, in rank order (all of the same shape)."""
    outs = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(outs, t.contiguous(), group=group)
    return outs


def row_offset(n_local, group=None, device=None):
    """(offset, n_total): this rank's first global row (the exclusive prefix of the ranks' row counts in rank order)
    and the number of rows over all ranks.  Assumes the contiguous rank-order layout of ``distributed.shard_range``."""
    if _world(group) == 1:
        return 0, int(n_local)
    counts = _all_gather(torch.tensor([int(n_local)], dtype=torch.int64, device=device), group)
    counts = [int(c.item()) for c in counts]
    rank = dist.get_rank(group)
    return sum(counts[:rank]), sum(counts)


def resolve_max_drop(max_drop, n_total):
    """The number of observations ``max_drop`` stands for: an int count in [0, n_total], or a float fraction in
    (0, 1] of n_total (rounded down)."""
    if isinstance(max_drop, (bool, np.bool_)):
        raise ValueError('max_drop must be an int count or a float fraction, not a bool')
    if isinstance(max_drop, (int, np.integer)):
        if not 0 <= int(max_drop) <= n_total:
            raise ValueError('max_drop = {} is outside [0, {}]'.format(int(max_drop), n_total))
        return int(max_drop)
    if isinstance(max_drop, (float, np.floating)):
        if not 0.0 < float(max_drop) <= 1.0:
            raise ValueError('a fractional max_drop must lie in (0, 1], got {}'.format(float(max_drop)))
        return int(math.floor(float(max_drop) * n_total))
    raise ValueError('max_drop must be an int count or a float fraction, not {}'.format(type(max_drop).__name__))


def qoi_matrix(qoi_jacobian, dim, device=None):
    """(A (K, D) float64, was_vector) from a (D,) or (K, D) QoI Jacobian; K >= 1."""
    a = qoi_jacobian if isinstance(qoi_jacobian, torch.Tensor) else torch.as_tensor(np.asarray(qoi_jacobian,
                                                                                             dtype=np.float64))
    vec = a.dim() == 1
    A = a.reshape(1, -1) if vec else a
    if A.dim() != 2 or A.shape[1] != dim or A.shape[0] < 1:
        raise ValueError('the QoI Jacobian must have shape ({},) or (K, {}) with K >= 1, got {}'.format(
            dim, dim, tuple(a.shape)))
    if device is not None:
        A = to_device(A, device)
    return A, vec


def _order(key, index):
    """Positions of the entries sorted by key descending, ties by index ascending."""
    by_index = torch.argsort(index, stable=True)
    by_key = torch.argsort(-key[by_index], stable=True)
    return by_index[by_key]


def local_candidates(key, offset, m):
    """This rank's top-m candidates (key, global index): key > 0, largest first, ties to the lower index.  The
    selection touches the N_local keys, not X."""
    idx = torch.nonzero(key > 0).reshape(-1)
    k = key[idx]
    o = _order(k, idx)[:m]
    return k[o], idx[o] + int(offset)


def merge_candidates(keys, indices, m):
    """The global top-m (key, index) from per-rank candidate lists (tensors; padding has key <= 0), by key descending
    and ties to the lower global index.  Each rank's global top-m elements are among its local top-m under the same
    order, so merging the local lists gives exactly the single-process selection."""
    k = torch.cat([t.reshape(-1) for t in keys])
    i = torch.cat([t.reshape(-1) for t in indices])
    keep = k > 0
    k, i = k[keep], i[keep]
    o = _order(k, i)[:m]
    return k[o], i[o]


def select_candidates(key, offset, m, group=None):
    """(keys, global indices) of the m observations with the largest positive key over all ranks, ties to the lower
    global index; identical on every rank."""
    k, i = local_candidates(key, offset, m)
    if _world(group) == 1:
        return k, i
    pk = torch.zeros(m, dtype=k.dtype, device=k.device)
    pi = torch.full((m,), -1, dtype=torch.int64, device=k.device)
    pk[:k.numel()] = k
    pi[:i.numel()] = i
    return merge_candidates(_all_gather(pk, group), _all_gather(pi, group), m)


@dataclass
class AMIPResult:
    """Outcome of :meth:`ObservationInfluence.amip`.

    ``n_drop``: the least number m <= max_drop of observations whose removal is predicted to reach the target, or
    None.  ``indices``: global int64 indices in selection order - the first ``n_drop`` of them, or all candidates up
    to max_drop when the target is out of reach.  ``predicted_value``: the first-order prediction of the quantity of
    interest without ``indices``.  ``max_change``: the predicted change when the first max_drop candidates are
    dropped.  ``direction``: 'decrease' (phi_hat > target) or 'increase'.  ``value``: phi at the optimum."""
    n_drop: Optional[int]
    indices: np.ndarray
    predicted_value: float
    max_change: float
    direction: str
    value: float
    target: float


@dataclass
class ApproximateCVResult:
    """Outcome of :meth:`ObservationInfluence.approximate_cv`.

    Per local row, in the array kind of the weights: ``z_loo``, the leave-one-out linear predictor of ``method``
    ('ns' or 'ij'); ``loss``, the family's negative log-likelihood of y_n at z_loo (up to terms in y only);
    ``leverage``, s_n h_n.  Over all ranks: ``mean_loss`` = sum w_n loss_n / sum w_n over the rows with a nonzero
    weight and a defined prediction, and ``n_invalid``, the rows whose Newton step is not defined (NaN in z_loo and
    loss: without row n the Hessian is singular to working accuracy)."""
    method: str
    z_loo: object
    loss: object
    leverage: object
    mean_loss: float
    n_invalid: int


LOO_METHODS = ('ns', 'ij')
# s_n h_n at or above this: H - s_n x_n x_n^T is singular to working accuracy (an exactly singular case computes
# s_n h_n only to within a few ulps of 1)
NS_SINGULAR = 1.0 - 2.0 ** -40


def check_loo_method(method):
    if method not in LOO_METHODS:
        raise ValueError("method must be 'ns' (Newton step) or 'ij' (infinitesimal jackknife), not {!r}".format(method))
    return method


def loo_predictor(z, resid, s, w, h, method):
    """z_n^NS (NaN where s_n h_n >= 1 - 2^-40) or z_n^IJ from the statistics at theta_hat and h_n."""
    step = w * resid * h
    if method == 'ij':
        return z + step
    lev = s * h
    return torch.where(lev < NS_SINGULAR, z + step / (1.0 - lev), torch.full_like(z, float('nan')))


GROUP_MAX_ROWS = ops.GROUP_LOO_MAX_ROWS


def group_starts(groups, n_local, group=None, device=None):
    """(starts, labels): the int64 group starts (G + 1 entries, 0 .. n_local) of this rank's rows and the labels as
    an int64 tensor (both on the labels' device), from one integer label per local row in any array kind.  Labels must be non-decreasing (a group
    is one label), no group may have more than GROUP_MAX_ROWS rows, and no label may continue on the next rank: the
    last label of rank r must be less than the first label of rank r + 1.  One all-gather of each rank's first and
    last label (and of whether its labels are well formed, so that every rank raises the same ValueError instead of
    leaving the others in the collective; ``device`` carries it for NCCL)."""
    err, labels, starts = None, None, None
    try:
        lab = groups.detach() if isinstance(groups, torch.Tensor) else torch.as_tensor(np.asarray(groups))
    except (TypeError, ValueError, RuntimeError) as e:
        lab, err = None, 'groups cannot be read as integer labels ({})'.format(e)
    if err is None:
        if lab.dim() != 1 or lab.numel() != n_local:
            err = 'groups has shape {}, this rank holds {} observations'.format(tuple(lab.shape), n_local)
        elif lab.dtype == torch.bool or lab.dtype.is_floating_point or lab.dtype.is_complex:
            err = 'groups must hold integer labels, not {}'.format(lab.dtype)
    if err is None:
        labels = lab.to(dtype=torch.int64)
        step = labels[1:] - labels[:-1]
        if bool((step < 0).any()):
            err = 'group labels must be non-decreasing (each group a run of consecutive rows)'
        else:
            cut = torch.nonzero(step).reshape(-1) + 1
            ends = [cut, torch.full((1,), n_local, dtype=torch.int64, device=labels.device)] if n_local else []
            starts = torch.cat([torch.zeros(1, dtype=torch.int64, device=labels.device)] + ends)
            size = starts[1:] - starts[:-1]
            if size.numel() and int(size.max()) > GROUP_MAX_ROWS:
                g = int(torch.argmax(size))
                err = 'group {} has {} rows; at most {} are supported'.format(int(labels[starts[g]]), int(size[g]),
                                                                             GROUP_MAX_ROWS)
    if _world(group) > 1:
        dev = device if _nccl(group) else None
        mine = torch.tensor([err is None, n_local > 0 if err is None else 0,
                             int(labels[0]) if err is None and n_local else 0,
                             int(labels[-1]) if err is None and n_local else 0], dtype=torch.int64, device=dev)
        every = [t.cpu().tolist() for t in _all_gather(mine, group)]
        if err is None:
            bad = [r for r, e in enumerate(every) if not e[0]]
            if bad:
                err = 'the group labels of rank(s) {} are malformed'.format(bad)
        if err is None:
            prev = None
            for r, (_, nonempty, first, last) in enumerate(every):
                if not nonempty:
                    continue
                if prev is not None and not prev[1] < first:
                    err = ('group {} straddles ranks {} and {}: a group must lie on one rank (labels increasing '
                           'across ranks)'.format(first, prev[0], r))
                    break
                prev = (r, last)
    if err is not None:
        raise ValueError(err)
    return starts, labels


def glm_loss(z, y, family):
    """The family's negative log-likelihood of y at the linear predictor z, up to terms in y only."""
    if family == 'logistic':
        return torch.clamp(z, min=0.0) + torch.log1p(torch.exp(-torch.abs(z))) - y * z
    if family == 'poisson':
        return torch.exp(z) - y * z
    if family == 'gaussian':
        return 0.5 * (y - z) ** 2
    raise ValueError('unknown GLM family {!r}'.format(family))


def cv_totals(loss, w, invalid, group=None):
    """(mean_loss, n_invalid) over all ranks: sum w_n loss_n / sum w_n over the rows with w_n != 0 that are not
    ``invalid`` (bool mask of the rows without a prediction), and the number of invalid rows.  One all-reduce of
    three numbers, on the device for NCCL and on the host otherwise."""
    keep = (w != 0) & ~invalid
    t = torch.stack([torch.where(keep, w * loss, torch.zeros_like(loss)).sum(),
                     torch.where(keep, w, torch.zeros_like(w)).sum(),
                     invalid.sum().to(loss.dtype)])
    if _world(group) > 1:
        t = t if _nccl(group) else t.cpu()
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    num, den, nbad = (float(v) for v in t.cpu())
    return (num / den if den != 0 else float('nan')), int(nbad)


def amip_from_scores(score, value, target, max_drop, offset=0, group=None):
    """AMIP selection from the per-observation scores w_n psi_n of this rank (dropping a set A changes phi by about
    -sum_{n in A} w_n psi_n).  Pure torch over the N_local scores and the candidate lists, so it runs on any device
    and any process group."""
    value, target = float(value), float(target)
    sign = 1.0 if value >= target else -1.0
    ks, idx = select_candidates(sign * score, offset, max_drop, group)
    # the prefix sums run on the host in float64, sequentially: at most max_drop values
    delta = -sign * np.cumsum(ks.cpu().numpy().astype(np.float64))
    idx = idx.cpu().numpy().astype(np.int64)
    pred = value + delta
    reached = (pred <= target) if sign > 0 else (pred >= target)
    if value == target:
        n_drop = 0
    else:
        hit = np.nonzero(reached)[0]
        n_drop = int(hit[0]) + 1 if hit.size else None
    total = float(delta[-1]) if delta.size else 0.0
    take = idx.size if n_drop is None else n_drop
    return AMIPResult(n_drop=n_drop, indices=idx[:take].copy(), predicted_value=value + (float(delta[take - 1])
                                                                                       if take else 0.0),
                      max_change=total, direction='decrease' if sign > 0 else 'increase', value=value,
                      target=target)


class ObservationInfluence:
    """Influence of every observation on quantities of interest of a weighted GLM optimum, without forming the
    (D, N) sensitivity matrix.

    ``objective``: a :class:`~vittles_b200.objectives.GLMObjective` (any family, ``l2`` and weights allowed).
    ``opt_par_value``: theta_hat, the optimum at ``weights`` (None: all ones).  ``hessian_at_opt``: optional (D, D)
    Hessian; otherwise the statistics pass and the Hessian assembly run as for
    ``HyperparameterSensitivityLinearApproximation`` (same engines, same all-reduce).  ``validate_optimum`` raises
    ``ValueError`` when |grad| > ``grad_tol``.  Results come back in the array kind of ``weights`` (of
    ``opt_par_value`` when ``weights`` is None): a CUDA tensor stays on the device."""

    def __init__(self, objective, opt_par_value, weights=None, hessian_at_opt=None, validate_optimum=False,
                 grad_tol=1e-8):
        if not isinstance(objective, GLMObjective):
            raise NotImplementedError(
                'ObservationInfluence is implemented for GLMObjective only; for {} build '
                'HyperparameterSensitivityLinearApproximation and use A @ get_dopt_dhyper()'.format(
                    type(objective).__name__))
        self._obj = objective
        self._kind = kind_of(opt_par_value if weights is None else weights)
        self._theta_kind = kind_of(opt_par_value)
        dev = objective.device
        n, d = objective.n_obs, objective.dim
        self.dim = d
        self._theta = to_device(opt_par_value, dev).reshape(-1)
        if self._theta.numel() != d:
            raise ValueError('opt_par_value has {} entries, the objective {}'.format(self._theta.numel(), d))
        self._w = (torch.ones(n, dtype=torch.float64, device=dev) if weights is None
                   else to_device(weights, dev).reshape(-1).contiguous())
        if self._w.numel() != n:
            raise ValueError('weights has {} entries, this rank holds {} observations'.format(self._w.numel(), n))
        if hessian_at_opt is None:
            self._stats, H = objective.vt_stats_and_hessian(self._theta, self._w)
        else:
            H = to_device(hessian_at_opt, dev)
            if tuple(H.shape) != (d, d):
                raise ValueError('``hessian_at_opt`` is the wrong shape.')
            self._stats = objective.vt_stats(self._theta, self._w, want_grad=validate_optimum)
        if validate_optimum:
            g = float(torch.linalg.vector_norm(self._stats['grad']))
            if g > grad_tol:
                raise ValueError('The gradient is not zero at the proposed optimum.  '
                                 '||grad|| = {} > {} = grad_tol'.format(g, grad_tol))
        self.factor = solver_lib.get_cholesky_solver(H).factor
        self.offset, self.n_total = row_offset(n, objective.group, dev if _nccl(objective.group) else None)
        self._h = None

    # -- influence ------------------------------------------------------------
    def _influence_device(self, A):
        V = self.factor.solve(A.T.contiguous())                                 # (D, K) = H^{-1} A^T
        return ops.glm_influence(self._obj.X, self._stats['resid'], V.T.contiguous(), alpha=-1.0)

    def influence(self, qoi_jacobian):
        """psi = d phi / d w for this rank's observations: (D,) -> (N_local,), (K, D) -> (K, N_local)."""
        A, vec = qoi_matrix(qoi_jacobian, self.dim)
        psi = self._influence_device(to_device(A, self._theta.device))
        return as_kind(psi[0] if vec else psi, self._kind)

    # -- dropping observations ------------------------------------------------
    def _local_rows(self, drop):
        """Local positions of the global indices in ``drop`` that this rank holds (validated, duplicates removed)."""
        d = np.unique(np.asarray(drop.cpu() if isinstance(drop, torch.Tensor) else drop, dtype=np.int64).reshape(-1))
        if d.size and (d[0] < 0 or d[-1] >= self.n_total):
            raise ValueError('observation indices must lie in [0, {})'.format(self.n_total))
        mine = d[(d >= self.offset) & (d < self.offset + self._obj.n_obs)] - self.offset
        return torch.as_tensor(mine, dtype=torch.int64, device=self._theta.device)

    def _predict_without(self, rows):
        dev = self._theta.device
        if rows.numel():
            coef = (self._w[rows] * self._stats['resid'][rows]).reshape(1, -1).contiguous()
            g = ops.gemm(coef, self._obj.X[rows], 'KC', 'KS').reshape(-1)    # sum_n w_n resid_n x_n
        else:
            g = torch.zeros(self.dim, dtype=torch.float64, device=dev)
        self._obj._allreduce(g)
        return self._theta + self.factor.solve(g)

    def predict_opt_par_without(self, drop):
        """First-order prediction of the optimum with the weights of the observations ``drop`` (global indices) set
        to zero: theta_hat + H^{-1} sum_{n in drop} w_n resid_n x_n."""
        return as_kind(self._predict_without(self._local_rows(drop)), self._theta_kind)

    def refit(self, drop, tol=1e-10, maxiter=25):
        """Newton's method on the same objective with the weights of ``drop`` set to zero, from
        ``predict_opt_par_without(drop)``; stops when |step| < tol.  Warns (UserWarning) if it has not converged
        after ``maxiter`` steps and returns the last iterate."""
        rows = self._local_rows(drop)
        w = self._w.clone()
        w[rows] = 0.0
        theta = self._predict_without(rows)
        converged = False
        for _ in range(int(maxiter)):
            st, H = self._obj.vt_stats_and_hessian(theta, w)
            step = ops.potrf(H, overwrite=True).solve(st['grad'])
            theta = theta - step
            if float(torch.linalg.vector_norm(step)) < tol:
                converged = True
                break
        if not converged:
            warnings.warn('refit: Newton did not converge to |step| < {} in {} iterations'.format(tol, maxiter),
                          UserWarning)
        return as_kind(theta, self._theta_kind)

    # -- approximate leave-one-out ---------------------------------------------
    def _quad_forms(self):
        """h_n = x_n^T H^{-1} x_n = |L^{-1} x_n|^2 for this rank's rows, computed once.  The engine follows the
        objective's precision; a TF32 objective gets 'auto' (the quadratic forms are always FP64-grade)."""
        if getattr(self, '_h', None) is None:
            precision = self._obj.precision
            if precision in ('tf32', 'tf32x3'):
                precision = 'auto'
            self._obj._wait_resident()
            Linv = self.factor.inverse_factor()
            self._h = ops.quad_forms(Linv, self._obj.X, precision=precision)
            del Linv
        return self._h

    def _loo(self, method):
        st = self._stats
        return loo_predictor(st['z'], st['resid'], st['s'], self._w, self._quad_forms(), method)

    def _group_loo(self, method, groups):
        """(z, h, labels) of leaving out each group; the labels are checked (:func:`group_starts`) before any
        device work.  The engine follows the objective's precision as for :meth:`_quad_forms`."""
        group = self._obj.group
        starts, labels = group_starts(groups, self._obj.n_obs, group, self._obj.device if _nccl(group) else None)
        dev = self._obj.X.device
        starts, labels = starts.to(dev), labels.to(dev)
        precision = self._obj.precision
        if precision in ('tf32', 'tf32x3'):
            precision = 'auto'
        self._obj._wait_resident()
        Linv = self.factor.inverse_factor()
        st = self._stats
        z, h = ops.group_loo(Linv, self._obj.X, starts, st['s'], self._w * st['resid'], st['z'], method,
                             precision=precision)
        del Linv
        return z, h, labels

    def leverage(self):
        """s_n h_n (the diagonal of the GLM hat matrix) for this rank's observations, shape (N_local,)."""
        return as_kind(self._stats['s'] * self._quad_forms(), self._kind)

    def loo_linear_predictor(self, method='ns', groups=None):
        """The approximate leave-one-out linear predictor x_n^T theta_hat_{-n} of this rank's rows, (N_local,):
        'ns' one Newton step without row n (NaN, with a UserWarning, where that step is not defined), 'ij' the
        infinitesimal jackknife x_n^T predict_opt_par_without([n]).  With ``groups`` (one integer label per local
        row, see :func:`group_starts`), row n's predictor leaves out its whole group instead."""
        check_loo_method(method)
        if groups is None:
            z = self._loo(method)
            if method == 'ns':
                _warn_invalid(int(torch.isnan(z).sum()))
            return as_kind(z, self._kind)
        z, _, labels = self._group_loo(method, groups)
        if method == 'ns':
            _warn_invalid_groups(int(torch.isnan(z).sum()), labels[torch.isnan(z)])
        return as_kind(z, self._kind)

    def approximate_cv(self, method='ns', groups=None):
        """Approximate leave-one-out cross-validation: the held-out loss of every observation at its approximate
        leave-one-out prediction, and their weighted mean over all ranks (:class:`ApproximateCVResult`).  With
        ``groups`` (one integer label per local row, non-decreasing, groups of at most 32 rows on one rank; see
        :func:`group_starts`), leave-one-group-out: each row is predicted without its whole group, and
        ``n_invalid`` counts the rows of the groups whose Newton step is not defined."""
        check_loo_method(method)
        if groups is None:
            z = self._loo(method)
            h = self._quad_forms()
        else:
            z, h, labels = self._group_loo(method, groups)
        loss = glm_loss(z, self._obj.y, self._obj.family)
        invalid = torch.isnan(z) if method == 'ns' else torch.zeros_like(z, dtype=torch.bool)
        mean_loss, n_invalid = cv_totals(loss, self._w, invalid, self._obj.group)
        if groups is None:
            _warn_invalid(n_invalid)
        else:
            _warn_invalid_groups(n_invalid, labels[invalid])
        return ApproximateCVResult(method=method, z_loo=as_kind(z, self._kind), loss=as_kind(loss, self._kind),
                                   leverage=as_kind(self._stats['s'] * h, self._kind),
                                   mean_loss=mean_loss, n_invalid=n_invalid)

    # -- AMIP -----------------------------------------------------------------
    def amip(self, qoi, target=0.0, max_drop=0.01):
        """Approximate Maximum Influence Perturbation: the fewest observations whose removal is predicted to move
        phi to ``target`` (the default 0 asks for a sign change).

        ``qoi``: a callable phi(theta) -> scalar torch value (its gradient at theta_hat is taken with
        ``torch.func.grad``), or a pair (a, phi_hat) of the gradient and the value.  ``max_drop``: an int count in
        [0, N] or a float fraction in (0, 1] of the N observations over all ranks.

        Dropping a set A changes phi by about -sum_{n in A} w_n psi_n.  If phi_hat > target the candidates are the
        observations with w_n psi_n > 0, largest first; if phi_hat < target those with w_n psi_n < 0, most negative
        first; ties go to the lower global index, zero-weight rows are never chosen.  The selection (a stable sort
        of the candidate scores, merged over the ranks) and the float64 prefix sum touch the N values of psi, not
        X: the pass over X that computes psi is the only step of size N x D."""
        m = resolve_max_drop(max_drop, self.n_total)
        if callable(qoi):
            theta = self._theta.detach()
            a = torch.func.grad(qoi)(theta)
            value = float(qoi(theta))
        else:
            a, value = qoi
            value = float(value)
        A, _ = qoi_matrix(a, self.dim)
        psi = self._influence_device(to_device(A, self._theta.device))[0]
        return amip_from_scores(self._w * psi, value, target, m, self.offset, self._obj.group)


def _warn_invalid(n):
    if n:
        warnings.warn('approximate leave-one-out: the Newton step is not defined for {} observation(s) (s_n h_n >= '
                      '1 - 2^-40: the Hessian without the row is singular); their prediction and loss are NaN and they '
                      'are left out of mean_loss'.format(n), UserWarning)


def _warn_invalid_groups(n, labels):
    """n rows over all ranks without a prediction; ``labels`` of this rank's such rows name the groups."""
    if n:
        names = torch.unique(labels).cpu().tolist()
        shown = ', '.join(str(v) for v in names[:10]) + (', ...' if len(names) > 10 else '')
        warnings.warn('approximate leave-one-group-out: the Newton step is not defined for {} observation(s) (the '
                      'Hessian without the group is singular to working accuracy: a squared Cholesky pivot of '
                      'I - S^1/2 Q S^1/2 <= 2^-40); their prediction and loss are NaN and they are left out of '
                      'mean_loss.  Groups on this rank: {}'.format(n, shown or 'none'), UserWarning)


def _nccl(group):
    return _world(group) > 1 and dist.get_backend(group) == 'nccl'
