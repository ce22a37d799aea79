"""cplb_jacobian_products_device on the host side: every argument error is reported before any CUDA call (so these hold on a machine
without a GPU: the problems here are created with device = -1 and never bind to one)."""
import ctypes as C

import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic


def _call(prob, args):
    return _cabi.load().cplb_jacobian_products_device(None if prob is None else prob._h, None if args is None else C.byref(args), None)


def _args(N=4, **kw):
    """Every pointer a distinct non-NULL host address unless given (the checks never dereference them)."""
    buf = np.zeros(16)
    a = _cabi.JacobianProductsArgs(N, buf.ctypes.data)
    for k, v in kw.items():
        setattr(a, k, v)
    a._keep = buf
    return a


def _ptr():
    b = np.zeros(1)
    _ptr.keep.append(b)
    return b.ctypes.data


_ptr.keep = []


def test_argument_errors_come_before_any_device_work():
    lib = _cabi.load()
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    assert prob.GetDevice() == -1
    lam, of, xb, v, gd, fd = (_ptr() for _ in range(6))
    assert _call(None, _args(lambda_=lam, x_bar=xb)) == _cabi.NULL_POINTER
    assert _call(prob, None) == _cabi.NULL_POINTER and b"args" in lib.cplb_last_error()
    assert _call(prob, _args(x=None, lambda_=lam, x_bar=xb)) == _cabi.NULL_POINTER and b"x is NULL" in lib.cplb_last_error()
    assert _call(prob, _args(N=-1, lambda_=lam, x_bar=xb)) == _cabi.INVALID_ARGUMENT and b"negative" in lib.cplb_last_error()
    assert _call(prob, _args(x_bar=xb)) == _cabi.INVALID_ARGUMENT and b"lambda and obj_factor" in lib.cplb_last_error()
    assert _call(prob, _args(g_dot=gd)) == _cabi.NULL_POINTER and b"v is NULL" in lib.cplb_last_error()
    assert _call(prob, _args(f_dot=fd)) == _cabi.NULL_POINTER and b"v is NULL" in lib.cplb_last_error()
    assert _call(prob, _args(lambda_=lam, obj_factor=of, v=v)) == _cabi.INVALID_ARGUMENT and b"no output" in lib.cplb_last_error()
    assert _call(prob, _args(N=1 << 31, lambda_=lam, x_bar=xb)) == _cabi.INVALID_ARGUMENT and b"2^31" in lib.cplb_last_error()
    assert prob.GetDevice() == -1 and prob.launch_count() == 0


def test_empty_batch_launches_nothing():
    prob = cpl.BatchedCplProblem(["right", "left"], 100.0)
    assert _call(prob, _args(N=0, x=None, obj_factor=_ptr(), x_bar=_ptr())) == _cabi.OK
    assert _call(prob, _args(N=0, x=None, v=_ptr(), g_dot=_ptr(), f_dot=_ptr())) == _cabi.OK
    assert prob.launch_count() == 0 and prob.GetDevice() == -1


def test_python_entry_validates_before_calling():
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    with pytest.raises(ValueError, match="CUDA tensor"):
        prob.JacobianProducts(np.zeros((2, prob.n)), lam=np.zeros((2, prob.m)))


def test_per_instance_array_that_requires_grad_is_refused():
    torch = pytest.importorskip("torch")
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    x = torch.zeros(2, prob.n, dtype=torch.float64, requires_grad=True)
    with pytest.raises(ValueError, match="requires grad"):
        cpl.constraints_and_cost(prob, x, per_instance={"mu": torch.ones(2, dtype=torch.float64, requires_grad=True)})


@pytest.mark.gpu
def test_sharded_problem_is_refused(cuda_device):
    """Like cplb_solve_device: one batch per GPU.  (A sharded problem needs explicit device ordinals, hence a CUDA device.)"""
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground(), devices=[0, 0])
    assert _call(prob, _args(lambda_=_ptr(), x_bar=_ptr())) == _cabi.INVALID_ARGUMENT
    assert b"single-device problem" in _cabi.load().cplb_last_error()
