"""Native lock-step solve round: `cplb_solve_device` (csrc/cplb_solver.cu) behind the interface of `LockStepInteriorPoint`.

Same algorithm as centroidalplanner_b200/lockstep_solver.py (the interior-point scheme IPOPT implements; see there and
include/cpl_batched.h), but a round is eight kernel launches -- four batched evaluations of the hot path and four solver
kernels that hold one instance's KKT system in shared memory -- instead of ~1,500 small torch launches and cuBLAS' batched
LU.  The two drivers agree to the solver tolerances, not bit for bit (different factorisation, different summation orders).
Its CPU replay (the same per-instance code on the host, the C oracle behind the evaluations) does agree bit for bit on Ground and
no-environment problems: every result field, in every mode, after any number of iterations.
The caller side of SURVEY 8(f) rank 1: cpl::CentroidalPlanner::Solve (src/CentroidalPlanner.cpp:22-34) for N instances.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _cabi
from .lockstep_solver import SolveResult
from .problem import _check


class NativeInteriorPoint:
    """Options carry IPOPT's names where the meaning is IPOPT's (`tol`, `max_iter`, `mu_init`, `bound_push`, `bound_frac`,
    `nlp_scaling_max_gradient`, `bound_relax_factor`)."""

    def __init__(self, tol=1e-3, max_iter=500, mu_init=0.1, bound_push=1e-2, bound_frac=1e-2, nlp_scaling_max_gradient=100.0,
                 constr_viol_tol=1e-4, polish_viol_tol=1e-9, bound_relax_factor=1e-8, max_backtracks=30, tail_instances=-1):
        self.options = _cabi.SolverOptions(float(tol), float(mu_init), float(bound_push), float(bound_frac), float(nlp_scaling_max_gradient),
                                           float(constr_viol_tol), float(polish_viol_tol), float(bound_relax_factor), int(max_iter),
                                           int(max_backtracks), int(tail_instances))

    def Solve(self, problem, x0, per_instance=None):
        """Solve all N instances from the starting points x0 (N, n), a CUDA tensor on the problem's device.  per_instance: dict of
        per-instance parameter arrays (contiguous float64 CUDA tensors, (N,) / (N, len): cplb_instance_params), every instance then
        solves its own planning problem."""
        x0 = torch.as_tensor(x0)
        if not x0.is_cuda:
            raise ValueError("cplb_solve_device needs device-resident starting points (there is no CPU solve path)")
        x0 = x0.to(torch.float64).contiguous()
        N, n = x0.shape
        if n != problem.n:
            raise ValueError(f"x0 has {n} columns, the problem {problem.n} variables")
        dev, f64, i32 = x0.device, torch.float64, torch.int32
        x = torch.empty(N, n, dtype=f64, device=dev)
        status = torch.empty(N, dtype=i32, device=dev)
        iters = torch.empty(N, dtype=i32, device=dev)
        cost = torch.empty(N, dtype=f64, device=dev)
        viol = torch.empty(N, dtype=f64, device=dev)
        dual = torch.empty(N, dtype=f64, device=dev)
        lam = torch.empty(N, problem.m, dtype=f64, device=dev)
        rounds, evals, inst, tail = C.c_int32(0), C.c_int64(0), C.c_int64(0), C.c_int64(0)
        out = _cabi.SolveOutputs(x.data_ptr(), status.data_ptr(), iters.data_ptr(), cost.data_ptr(), viol.data_ptr(), dual.data_ptr(),
                                 lam.data_ptr(), C.pointer(rounds), C.pointer(evals), C.pointer(inst), C.pointer(tail))
        stream = torch.cuda.current_stream(dev).cuda_stream
        pi, keep = problem._instance_params(per_instance, N, _cabi.INSTANCE_MAJOR, dev)
        with torch.cuda.device(dev):
            _check(problem._lib.cplb_solve_device(problem._h, N, x0.data_ptr(), None if pi is None else C.byref(pi), C.byref(self.options),
                                                  C.byref(out), C.c_void_p(stream)))
        del keep
        return SolveResult(x=x, status=status.to(torch.int64), iterations=iters.to(torch.int64), cost=cost, constr_viol=viol, dual_inf=dual,
                           rounds=rounds.value, evaluations=evals.value, instance_evaluations=inst.value, lam=lam, tail_instances=tail.value)
