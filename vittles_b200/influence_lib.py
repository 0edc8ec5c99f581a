"""Per-observation influence on quantities of interest, and dropped-data robustness (AMIP), for GLM objectives.

For weighted GLM objectives the infinitesimal jackknife is ``S = d theta_hat / d w = -H^{-1} G^T`` with column n
equal to ``-resid_n H^{-1} x_n``.  Users of the IJ usually want the effect of the weights on a few quantities of
interest phi_k(theta) rather than S itself:

    psi[k, n] = d phi_k(theta_hat(w)) / d w_n = a_k^T S[:, n] = -resid_n x_n . v_k,   v_k = H^{-1} a_k,  a_k = grad phi_k

That is K solves against the Cholesky factor of H and one pass over X that writes K values per observation
(``ops.glm_influence``); nothing of size D x N is formed, so the (D, N) matrix of
``HyperparameterSensitivityLinearApproximation`` and its memory are never needed.

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


def _nccl(group):
    return _world(group) > 1 and dist.get_backend(group) == 'nccl'
