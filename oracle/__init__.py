"""CPU oracle for the vittles sensitivity hot path.

TEST INFRASTRUCTURE - NOT PRODUCT CODE.  Only ``tests/``,
``__graft_entry__.smoke()`` and the ``cpu_baseline`` / ``--impl reference``
legs of ``bench.py`` may import this package, and only as the checker or as the
timed CPU baseline.  ``vittles_b200`` never imports it: the product path fails
loudly when its CUDA library is missing.

What it is: a float64 restatement of the reference's algorithms
(the ``vittles`` package of rgiordan/vittles), module by module, with
``autograd.{grad,jacobian,hessian,make_jvp}`` replaced by
``torch.func.{grad,jacrev,hessian,jvp}`` on CPU and the reference's scipy calls
(``cho_factor``/``cho_solve``, ``factorized``, ``cg``) kept verbatim.  Each
function cites the reference ``file:line`` it follows.

Pinning (SURVEY.md section 8c): the reference itself cannot be imported here
(``autograd``/``paragami`` are not installed).  ``oracle/make_golden.py`` runs
the UNMODIFIED reference sources from a checkout of it on top of the
``oracle/refshim`` stand-ins for those two packages, checks this restatement
against the reference's outputs, and stores them under ``tests/golden/``.
The reference's own closed-form test fixtures (QuadraticModel, MVN KL, block
quadratic, weighted least squares) are re-created in ``oracle/fixtures.py`` and
asserted in ``tests/test_oracle.py``.
"""
from . import solver_lib, sensitivity, sparse_hessian, lr_cov, bivariate, models, fixtures, slicing  # noqa: F401
