#!/usr/bin/env python3
"""Small invocations of the round's new kernels for `compute-sanitizer --tool memcheck python tools/sanitize_run.py`
(pytest itself does not start under the sanitizer in this image): INT8 engine incl. the converter warps and ragged
shapes, fused column maxima, multi-output HVP, batched CG, block-arrow multi-RHS solve, dense solves."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
import vittles_b200 as vt  # noqa: E402
from vittles_b200 import ops  # noqa: E402
from oracle import slicing  # noqa: E402

dev = torch.device('cuda', 0)
g = torch.Generator(device=dev).manual_seed(0)


def rnd(*s):
    return torch.randn(*s, device=dev, dtype=torch.float64, generator=g)


def rel(a, b):
    return float((a - b).abs().max() / b.abs().max())


for (N, D) in ((3001, 77), (90000, 1024), (70000, 515)):
    X = ops.synth_design(3, 0, N, D, dev)
    Hinv = torch.eye(D, device=dev, dtype=torch.float64) + 0.01 * rnd(D, D)
    r = rnd(N)
    print('apply', N, D, rel(ops.ij_apply(Hinv, X, r, precision='f64_ozaki'), ops.ij_apply(Hinv, X, r)))
    s = torch.rand(N, device=dev, dtype=torch.float64, generator=g)
    print('syrk', N, D, rel(ops.syrk_weighted(X, s, precision='f64_ozaki'), ops.syrk_weighted(X, s)))
    theta = 0.3 * ops.synth_theta(3, D, dev)
    y = (torch.rand(N, device=dev, dtype=torch.float64, generator=g) < 0.5).double()
    st = ops.glm_stats(X, theta, y, None, want_colmax=True)
    H1 = ops.syrk_weighted(X, st[2], precision='f64_ozaki', colmax=st[4])
    print('fused colmax', torch.equal(H1, ops.syrk_weighted(X, st[2], precision='f64_ozaki')))
    V = rnd(7, D)
    ref = torch.stack([ops.glm_hvp(X, st[2], V[k].contiguous()) for k in range(7)])
    print('hvp_multi', rel(ops.glm_hvp_multi(X, st[2], V), ref))
    V2 = rnd(30, D)
    print('hvp_gemm', rel(ops.glm_hvp_multi(X, st[2], V2)[:7], ops.glm_hvp_multi(X, st[2], V2[:7].contiguous())))
A = rnd(130, 333)
B = rnd(70, 333)
print('ogemm', rel(ops.ozaki_gemm(A, B), A @ B.T))
# the stand-alone slicers against the CPU model at ragged shapes (rows held in registers, and rows wider than 1024
# that are re-read), and an unweighted Hessian whose later chunks are sliced inside the GEMM
def same_digits(got, ref):
    return np.array_equal(got[0][:, :, :ref[0].shape[2]].cpu().numpy(), ref[0]) and np.array_equal(got[1].cpu().numpy(), ref[1])


for Xr in (rnd(517, 333), rnd(67, 1100)):
    print('slicer', tuple(Xr.shape), same_digits(ops.ozaki_slice(Xr, 7), slicing.slice_rows(Xr.cpu().numpy(), 7)))
Xr = rnd(517, 333)
sqr = torch.rand(517, device=dev, dtype=torch.float64, generator=g).sqrt()
for sq_ in (sqr, None):
    W = (Xr if sq_ is None else Xr * sq_[:, None]).T.contiguous().cpu().numpy()
    print('transposed slicer', same_digits(ops.ozaki_slice_t(Xr, sq_, 7), slicing.slice_rows(W, 7)))
Xu = ops.synth_design(4, 0, 70001, 650, dev)
print('syrk unweighted', rel(ops.syrk_weighted(Xu, None, precision='f64_ozaki'), ops.syrk_weighted(Xu, None)))
# batched CG with a Jacobi preconditioner
d = 96
a = rnd(d, d + 4)
Hm = a @ a.T / d + torch.eye(d, device=dev, dtype=torch.float64)
Bm = rnd(d, 5)
solve = vt.solver_lib.get_cg_solver(lambda v: Hm @ v, d, {'tol': 1e-12, 'M': vt.solver_lib.JacobiPreconditioner(torch.diagonal(Hm))})
print('cg', rel(solve(Bm), torch.linalg.solve(Hm, Bm)))
# block-arrow solve, 1 / 2 / 40 columns
from vittles_b200.sparse_hessian_lib import BlockArrowHessian  # noqa: E402
G, M, Dg = 257, 19, 96
dd = G * M + Dg
perm = torch.randperm(dd, device=dev, generator=g)
sa, gi = perm[:G * M].reshape(G, M), perm[G * M:]
bl = rnd(G, M, M)
blocks = bl @ bl.transpose(1, 2) / M + torch.eye(M, device=dev, dtype=torch.float64)
cross = 0.02 * rnd(G, M, Dg)
g0 = rnd(Dg, Dg)
hgg = g0 @ g0.T / Dg + 3.0 * torch.eye(Dg, device=dev, dtype=torch.float64)
h = BlockArrowHessian(dd, sa, gi, blocks=blocks, cross=cross, hgg=hgg)
dense = h.to_dense_tensor()
for K in (1, 2, 40):
    b = rnd(dd, K)
    print('arrow', K, rel(vt.solver_lib.get_cholesky_solver(h)(b), torch.linalg.solve(dense, b)))
# dense factor / solves crossing the 128 / 256 / 512 blockings
for D, K in ((300, 37), (1100, 64), (1100, 3), (1300, 1400)):
    a = rnd(D, D + 8)
    Hd = a @ a.T / D + torch.eye(D, device=dev, dtype=torch.float64)
    b = rnd(D, K)
    print('potrs', D, K, rel(ops.potrf(Hd).solve(b), torch.linalg.solve(Hd, b)))
torch.cuda.synchronize()
print('sanitize run done')
