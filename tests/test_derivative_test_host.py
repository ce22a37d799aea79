"""cplb_derivative_test_device on the host side: default options, and every argument error reported before any CUDA call (so they
hold on a machine without a GPU: the problems here are created with device = -1 and never bind to one)."""
import ctypes as C

import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic


def _call(prob, N, x, options=None, out=None, per_instance=None):
    lib = _cabi.load()
    return lib.cplb_derivative_test_device(None if prob is None else prob._h, N, x, per_instance, None if options is None else C.byref(options),
                                           None if out is None else C.byref(out), None)


def test_default_options_are_ipopts():
    opt = _cabi.DerivativeTestOptions(-1.0, -1.0)
    _cabi.load().cplb_derivative_test_default_options(C.byref(opt))
    assert (opt.perturbation, opt.tol) == (1e-8, 1e-4)
    _cabi.load().cplb_derivative_test_default_options(None)   # a NULL pointer is ignored


def test_argument_errors_come_before_any_device_work():
    lib = _cabi.load()
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    assert prob.GetDevice() == -1
    x = np.zeros((4, prob.n))
    xp = x.ctypes.data
    out = _cabi.DerivativeTestOutputs()                        # every output NULL: allowed
    assert _call(None, 4, xp, out=out) == _cabi.NULL_POINTER
    assert _call(prob, 4, xp, out=None) == _cabi.NULL_POINTER and b"out" in lib.cplb_last_error()
    assert _call(prob, 4, None, out=out) == _cabi.NULL_POINTER and b"x" in lib.cplb_last_error()
    assert _call(prob, -1, xp, out=out) == _cabi.INVALID_ARGUMENT and b"negative" in lib.cplb_last_error()
    for bad in (0.0, -1e-8, float("inf"), float("nan")):
        assert _call(prob, 4, xp, _cabi.DerivativeTestOptions(bad, 1e-4), out) == _cabi.INVALID_ARGUMENT, bad
        assert b"perturbation" in lib.cplb_last_error()
    for bad in (0.0, -1.0, float("nan")):
        assert _call(prob, 4, xp, _cabi.DerivativeTestOptions(1e-8, bad), out) == _cabi.INVALID_ARGUMENT, bad
        assert b"tol" in lib.cplb_last_error()
    assert prob.GetDevice() == -1 and prob.launch_count() == 0


def test_empty_batch_launches_nothing():
    prob = cpl.BatchedCplProblem(["right", "left"], 100.0)
    out = _cabi.DerivativeTestOutputs()
    assert _call(prob, 0, None, out=out) == _cabi.OK
    assert _call(prob, 0, None, options=_cabi.DerivativeTestOptions(1e-6, 1e-3), out=out) == _cabi.OK
    assert prob.launch_count() == 0 and prob.GetDevice() == -1


def test_python_entry_needs_a_cuda_tensor():
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    with pytest.raises(ValueError, match="CUDA tensor"):
        prob.DerivativeTest(np.zeros((2, prob.n)))


@pytest.mark.gpu
def test_sharded_problem_is_refused(cuda_device):
    """Like cplb_solve_device: one batch per GPU.  (A sharded problem needs explicit device ordinals, hence a CUDA device.)"""
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground(), devices=[0, 0])
    out = _cabi.DerivativeTestOutputs()
    x = np.zeros((4, prob.n))
    assert _call(prob, 4, x.ctypes.data, out=out) == _cabi.INVALID_ARGUMENT
    assert b"single-device problem" in _cabi.load().cplb_last_error()
