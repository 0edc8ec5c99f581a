"""Factorise and solve block-arrow systems on the GPU (the B200 replacement for
"SuperLU on the COO matrix", ``solver_lib.py:46-48``).

    H = [ blockdiag(B_g)   C ]   ->   L_g = chol(B_g),  Z_g = L_g^{-1} C_g,
        [ C^T            Hgg ]        S = Hgg - Z^T Z = chol-factorised dense Schur complement

    solve(b):  y_g = L_g^{-1} b_g ;  x_glob = S^{-1} (b_glob - Z^T y) ;
               x_g = L_g^{-T} (y_g - Z_g x_glob)

Right-hand sides ``(d, K)`` are solved together: ``Z`` (the large array, 6 GB per
million observations at config 3) is read twice per solve whatever K is - once by
the GEMM ``Z^T Y`` and once by ``Y -= Z X_glob`` - instead of 2 K times.

Sharding (SURVEY.md section 8e, config 3): with ``h.group`` set every rank holds the
blocks and cross blocks of its own observations and a replica of the global block.
The only exchanges are one all-reduce of the Dg x Dg matrix ``Z^T Z`` at factor
time and one of the Dg x K matrix ``Z^T Y`` per solve; the local parts of right-hand
side and solution stay sharded, the global parts are replicated.
"""
import torch

from . import ops
from ._arrays import to_device, kind_of, as_kind
from .distributed import allreduce_sum_

BLOCK_MAXM = 32          # csrc/blockchol.cuh: one block per warp / CTA out of shared memory


class CudaBlockKernels:
    """The kernels the solver is made of (C ABI: vt_block_*, vt_dgemm, vt_syrk_weighted, vt_potrf / vt_potrs).
    The solver takes them through this one object so that its sharding logic can be exercised on CPU ranks
    (tests/test_distributed_cpu.py supplies a numpy stand-in); the product never constructs anything else."""

    @staticmethod
    def block_potrf(blocks):
        return ops.block_potrf(blocks)

    @staticmethod
    def block_trsm(Lb, C, transpose=False):
        return ops.block_trsm(Lb, C, transpose=transpose)

    @staticmethod
    def block_solve(Lb, y, transpose=False):
        """One right-hand side: y (G, M) in place, one warp per block."""
        return ops.block_solve(Lb, y, transpose=transpose)

    @staticmethod
    def gram(Z2):
        """Z^T Z on the FP64 DMMA engine, at every size.  The Schur complement Hgg - Z^T Z is a difference of large
        terms, and the INT8 slicing engine's error is relative to the column maxima of Z: with a few O(1) cross
        blocks among 1e-3 ones and S a thousandfold cancellation, its S misses the parity bar
        (tests/test_gpu_block_arrow.py), so 'auto' is not used here."""
        return ops.syrk_weighted(Z2, precision='f64')

    @staticmethod
    def dense_factor(S):
        return ops.potrf(S, overwrite=True)

    # Up to GEMV_MAX_RHS columns go through the HBM-bound matrix-vector kernels, one pass over Z per column; wider
    # right-hand sides through the GEMM engine, one pass over Z per 64 columns (its tiles are 64 wide, so a GEMM
    # with one or two columns would spend 30x the flops of the matrix-vector form on padding).
    GEMV_MAX_RHS = 2

    @classmethod
    def zt_times(cls, Z2, Y2):
        """Z^T Y, (Dg, K) (deterministic reduction over the long dimension)."""
        K = Y2.shape[1]
        if K <= cls.GEMV_MAX_RHS:
            return torch.stack([ops.tall_colsum(Z2, Y2[:, k].contiguous()) for k in range(K)], dim=1)
        return ops.gemm(Z2, Y2, 'KS', 'KS')

    @classmethod
    def sub_z_times(cls, Z2, Xg, Y2):
        """Y -= Z X_glob in place."""
        K = Y2.shape[1]
        if K <= cls.GEMV_MAX_RHS:
            for k in range(K):
                yk = Y2[:, k].contiguous()
                ops.tall_gemv(Z2, Xg[:, k].contiguous(), alpha=-1.0, y=yk, beta=1.0)
                if K > 1:
                    Y2[:, k] = yk
                else:
                    Y2.copy_(yk.reshape(-1, 1))
            return Y2
        return ops.gemm(Z2, Xg, 'KC', 'KS', alpha=-1.0, beta=1.0, out=Y2)


class BlockArrowSolver:
    def __init__(self, h, overwrite=False, kernels=None):
        self.k = CudaBlockKernels if kernels is None else kernels
        self.h = h
        self.group = getattr(h, 'group', None)
        self.d = h.shape[0]
        self.sa = h.sparsity_array
        self.gi = h.global_inds
        self.G, self.M = self.sa.shape
        self.Dg = int(self.gi.numel())
        if h.blocks is None:
            raise ValueError('the block-diagonal part of the Hessian is missing')
        covered = self.G * self.M + self.Dg
        if covered != self.d:
            raise ValueError('block-arrow solver: local and global indices cover {} of {} parameters'.format(
                covered, self.d))
        blocks = h.blocks if overwrite else h.blocks.clone()
        self.Lb = self.k.block_potrf(blocks.contiguous())
        self.Z = None
        self.schur = None
        if self.Dg > 0:
            if h.hgg is None:
                raise ValueError('the global block of the Hessian is missing')
            S = h.hgg.clone()                                 # replicated over the group
            if h.cross is not None:
                cross = h.cross if overwrite else h.cross.clone()
                self.Z = self.k.block_trsm(self.Lb, cross.contiguous())
                ZtZ = self.k.gram(self.Z.reshape(self.G * self.M, self.Dg))
                S = S - allreduce_sum_(ZtZ, self.group)       # the one exchange of the factorisation
            elif self.group is not None:
                pass                                          # no coupling: nothing to exchange
            self.schur = self.k.dense_factor(S)

    def _solve_mat(self, b):
        """b (d, K) -> H^{-1} b, all K columns together."""
        K = b.shape[1]
        Y = b[self.sa].contiguous()                           # (G, M, K) gather of the local right-hand sides
        if K == 1:
            self.k.block_solve(self.Lb, Y.reshape(self.G, self.M))
        else:
            self.k.block_trsm(self.Lb, Y)
        x = torch.empty_like(b)
        Y2 = Y.reshape(self.G * self.M, K)
        if self.Dg > 0:
            rhs = b[self.gi].contiguous()                     # (Dg, K), replicated over the group
            Z2 = None
            if self.Z is not None:
                Z2 = self.Z.reshape(self.G * self.M, self.Dg)
                rhs = rhs - allreduce_sum_(self.k.zt_times(Z2, Y2), self.group)   # the one exchange of a solve
            xg = self.schur.solve(rhs)
            x[self.gi] = xg
            if Z2 is not None:
                self.k.sub_z_times(Z2, xg.contiguous(), Y2)
        if K == 1:
            self.k.block_solve(self.Lb, Y.reshape(self.G, self.M), transpose=True)
        else:
            self.k.block_trsm(self.Lb, Y, transpose=True)
        x[self.sa] = Y
        return x

    def solve(self, v):
        kind = kind_of(v)
        b = to_device(v, self.Lb.device) if self.Lb.is_cuda else torch.as_tensor(v, dtype=torch.float64)
        if b.shape[0] != self.d or b.dim() > 2:
            raise ValueError('right-hand side has shape {}, expected ({},) or ({}, K)'.format(
                tuple(b.shape), self.d, self.d))
        if b.dim() == 1:
            return as_kind(self._solve_mat(b.reshape(self.d, 1).contiguous()).reshape(-1), kind)
        return as_kind(self._solve_mat(b.contiguous()), kind)
