"""Stand-in for HIPS ``autograd`` backed by ``torch.func`` (float64, CPU).

TEST INFRASTRUCTURE ONLY.  Without ``autograd`` installed, the unmodified
reference (the ``vittles`` package of rgiordan/vittles) cannot be imported as is.
``oracle/make_golden.py`` puts this directory on ``sys.path`` so that the
reference's own code runs here and its outputs can be stored as golden
fixtures under ``tests/golden/``.  Nothing in ``vittles_b200`` imports this.

Only the names the reference uses are provided (reference call sites:
``sensitivity_lib.py:170,181,354,360,382,470,822,829,1058,1062``,
``sparse_hessian_lib.py:59``, ``lr_cov_lib.py:77-80,191``).

Convention: objectives handed to the reference are written with ``torch``.
Every transformed function accepts numpy arrays or torch tensors; it returns
numpy iff none of its positional arguments was a torch tensor (i.e. it was
called from the reference's top-level numpy code and not from inside another
transform), which makes the transforms nestable exactly like autograd's.
"""
import numpy as _np
import torch as _torch
from torch import func as _func

from . import numpy  # noqa: F401  (autograd.numpy)
from . import core  # noqa: F401


def _to_torch(a):
    if isinstance(a, _torch.Tensor):
        return a
    return _torch.as_tensor(_np.asarray(a, dtype=_np.float64))


def _prep(args):
    want_numpy = not any(isinstance(a, _torch.Tensor) for a in args)
    return [_to_torch(a) for a in args], want_numpy


def _out(val, want_numpy):
    if not want_numpy:
        return val
    if isinstance(val, _torch.Tensor):
        return val.detach().numpy().copy()
    if isinstance(val, (tuple, list)):
        return type(val)(_out(v, True) for v in val)
    return val


def _as_tensor_fun(fun):
    """fun may return python floats / numpy for constant outputs."""
    def wrapped(*a):
        r = fun(*a)
        if not isinstance(r, _torch.Tensor):
            r = _torch.as_tensor(r, dtype=_torch.float64)
        return r
    return wrapped


def _unary(transform):
    def maker(fun, argnum=0):
        tfun = transform(_as_tensor_fun(fun), argnum)

        def wrapped(*args):
            targs, want_numpy = _prep(args)
            return _out(tfun(*targs), want_numpy)
        return wrapped
    return maker


grad = _unary(lambda f, argnum: _func.grad(f, argnums=argnum))
jacobian = _unary(lambda f, argnum: _func.jacrev(f, argnums=argnum))
hessian = _unary(lambda f, argnum: _func.jacfwd(_func.jacrev(f, argnums=argnum), argnums=argnum))


def make_jvp(fun, argnum=0):
    """autograd.make_jvp: ``make_jvp(f, argnum)(*args)(v) -> (f(*args), J v)``."""
    tfun = _as_tensor_fun(fun)

    def at(*args):
        targs, want_numpy = _prep(args)

        def jvp(v):
            tv = _to_torch(v)
            want = want_numpy and not isinstance(v, _torch.Tensor)

            def f_of_arg(x):
                a = list(targs)
                a[argnum] = x
                return tfun(*a)
            val, tan = _func.jvp(f_of_arg, (targs[argnum],), (tv,))
            return _out(val, want), _out(tan, want)
        return jvp
    return at


def hessian_vector_product(fun, argnum=0):
    g = _func.grad(_as_tensor_fun(fun), argnums=argnum)

    def hvp(*args):
        # autograd signature: hvp(*fun_args, vector)
        targs, want_numpy = _prep(args)
        fargs, v = targs[:-1], targs[-1]

        def g_of_arg(x):
            a = list(fargs)
            a[argnum] = x
            return g(*a)
        _, tan = _func.jvp(g_of_arg, (fargs[argnum],), (v,))
        return _out(tan, want_numpy)
    return hvp
