"""Host-side mirrors of the reference's planner facades, batched: validation and parameter bookkeeping only.

`BatchedCentroidalPlanner` ~ cpl::CentroidalPlanner (include/CentroidalPlanner/CentroidalPlanner.h:19-189,
src/CentroidalPlanner.cpp) and `BatchedCoMPlanner` ~ cpl::CoMPlanner (CoMPlanner.h:10-89, src/CoMPlanner.cpp): the same
setters/getters with the same checks and exception types, on top of a `BatchedCplProblem` that evaluates N instances.
`Solve()` runs a batch of instances through a lock-step solver over the batched evaluator: IPOPT stays the production
host solver (INTEGRATION.md §2) but is not part of this repository nor installed in its image, so the default is the
native lock-step solve round (`NativeInteriorPoint`: cplb_solve_device); the facades also hand out the batched problem
(`GetCplProblem`) whose evaluation entry points any other solver drives.
"""
from __future__ import annotations

import numpy as np

from .problem import BatchedCplProblem


class BatchedCentroidalPlanner:
    def __init__(self, contact_names, robot_mass, env=None, device=None):
        if robot_mass <= 0.0:  # src/CentroidalPlanner.cpp:12-15
            raise ValueError("Invalid robot mass")
        self._contact_names = [str(s) for s in contact_names]
        self._robot_mass = float(robot_mass)
        self._env = env
        self._cpl_problem = BatchedCplProblem(self._contact_names, robot_mass, env, device=device)

    def Solve(self, x0=None, solver=None, per_instance=None, derivative_test=False):
        """cpl::CentroidalPlanner::Solve (src/CentroidalPlanner.cpp:22-34) for a batch: every row of `x0` (N, n) is one
        instance's starting point (default: one instance at `lockstep_solver.default_start` on the problem's device);
        returns one `Solution` dict per instance (CplProblem::GetSolution, sorted-name order) and keeps the solver's
        report in `last_solve`.  The reference runs ifopt::IpoptSolver here; IPOPT is not part of this repository, so the
        default `solver` is the native lock-step solve round (`NativeInteriorPoint`: same NLP, batched, on the GPU) --
        anything with `Solve(problem, x0, per_instance)` can take its place (e.g. `LockStepInteriorPoint`, the torch driver).  Like the reference, a failed solve is not
        raised (`:29-32`): inspect `last_solve.status`.
        derivative_test=True first runs the first-order derivative test the reference turns on before every solve (`:26`,
        BatchedCplProblem.DerivativeTest) at x0 with the same per-instance arrays and keeps its report in `last_derivative_test`;
        the solve itself is the same either way."""
        import torch

        from .lockstep_solver import default_start
        from .native_solver import NativeInteriorPoint

        prob = self._cpl_problem
        if x0 is None:
            if not torch.cuda.is_available():
                raise RuntimeError("Solve() evaluates on a CUDA device and none is available (there is no CPU evaluation path)")
            x0 = default_start(prob, 1, device=torch.device("cuda", torch.cuda.current_device()))
        if derivative_test:
            x0 = torch.as_tensor(x0)
            if not x0.is_cuda:
                raise ValueError("the derivative test needs device-resident starting points (there is no CPU evaluation path)")
            self.last_derivative_test = prob.DerivativeTest(x0.to(torch.float64).contiguous(), per_instance=per_instance)
        self.last_solve = (solver or NativeInteriorPoint()).Solve(prob, x0, per_instance)
        return [prob.GetSolution(xi) for xi in self.last_solve.x.detach().cpu().numpy()]

    # ---- helpers ------------------------------------------------------------------------------------
    def HasContact(self, contact_name):  # :359-370
        return contact_name in self._contact_names

    def _need(self, contact_name):
        if not self.HasContact(contact_name):
            raise ValueError(f"Invalid contact name: '{contact_name}'")  # std::invalid_argument, e.g. :41-44

    def GetCplProblem(self):
        return self._cpl_problem

    # ---- bounds (:37-124) ---------------------------------------------------------------------------
    def SetForceBounds(self, contact_name, force_lb, force_ub):
        self._need(contact_name)
        self._cpl_problem.SetForceBounds(contact_name, force_lb, force_ub)

    def GetForceBounds(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetForceBounds(contact_name)

    def SetPosBounds(self, contact_name, pos_lb, pos_ub):
        self._need(contact_name)
        self._cpl_problem.SetPosBounds(contact_name, pos_lb, pos_ub)

    def GetPosBounds(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetPosBounds(contact_name)

    def SetNormalBounds(self, contact_name, normal_lb, normal_ub):
        self._need(contact_name)
        self._cpl_problem.SetNormalBounds(contact_name, normal_lb, normal_ub)

    def GetNormalBounds(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetNormalBounds(contact_name)

    # ---- references and weights (:126-303) ------------------------------------------------------------
    def SetPosRef(self, contact_name, pos_ref):
        self._need(contact_name)
        self._cpl_problem.SetPosRef(contact_name, pos_ref)

    def GetPosRef(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetPosRef(contact_name)

    def SetForceRef(self, contact_name, force_ref):
        self._need(contact_name)
        self._cpl_problem.SetForceRef(contact_name, force_ref)

    def GetForceRef(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetForceRef(contact_name)

    def SetCoMRef(self, com_ref):
        self._cpl_problem.SetCoMRef(com_ref)

    def GetCoMRef(self):
        return self._cpl_problem.GetCoMRef()

    def SetCoMWeight(self, W_CoM):
        if W_CoM < 0.0:
            raise ValueError("Invalid weight")
        self._cpl_problem.SetCoMWeight(W_CoM)

    def GetCoMWeight(self):
        return self._cpl_problem.GetCoMWeight()

    def SetPosWeight(self, W_p):
        if W_p < 0.0:
            raise ValueError("Invalid weight")
        self._cpl_problem.SetPosWeight(W_p)

    def GetPosWeight(self):
        return {nm: self._cpl_problem.GetContactPosWeight(nm) for nm in self._contact_names}

    def SetContactPosWeight(self, contact_name, W_p):
        self._need(contact_name)
        if W_p < 0.0:
            raise ValueError("Invalid weight")
        self._cpl_problem.SetContactPosWeight(contact_name, W_p)

    def GetContactPosWeight(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetContactPosWeight(contact_name)

    def SetForceWeight(self, W_F):
        if W_F < 0.0:
            raise ValueError("Invalid weight")
        self._cpl_problem.SetForceWeight(W_F)

    def GetForceWeight(self):
        return {nm: self._cpl_problem.GetContactForceWeight(nm) for nm in self._contact_names}

    def SetContactForceWeight(self, contact_name, W_F):
        self._need(contact_name)
        if W_F < 0.0:
            raise ValueError("Invalid weight")
        self._cpl_problem.SetContactForceWeight(contact_name, W_F)

    def GetContactForceWeight(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetContactForceWeight(contact_name)

    # ---- wrench, friction, thresholds (:306-356) -----------------------------------------------------
    def SetManipulationWrench(self, wrench_manip):
        self._cpl_problem.SetManipulationWrench(wrench_manip)

    def GetManipulationWrench(self):
        return self._cpl_problem.GetManipulationWrench()

    def GetMu(self):
        return self._cpl_problem.GetMu()

    def SetForceThreshold(self, contact_name, F_thr):
        self._need(contact_name)
        if F_thr < 0.0:
            raise ValueError("Invalid force threshold")
        force_lb, force_ub = self._cpl_problem.GetForceBounds(contact_name)
        # :340 -- the threshold is only forwarded while the contact's force is not pinned to zero (a lifting contact)
        if (force_lb != 0.0).any() and (force_ub != 0.0).any():
            self._cpl_problem.SetForceThreshold(contact_name, F_thr)

    def GetForceThreshold(self, contact_name):
        self._need(contact_name)
        return self._cpl_problem.GetForceThreshold(contact_name)


class BatchedCoMPlanner(BatchedCentroidalPlanner):
    """cpl::CoMPlanner: no environment (FrictionCone rows only, src/CplProblem.cpp:63-71), contact positions and
    normals pinned through equal bounds, lifting contacts through zero force bounds."""

    def __init__(self, contact_names, robot_mass, device=None):
        super().__init__(contact_names, robot_mass, None, device=device)  # src/CoMPlanner.cpp:5-8
        self.SetPosWeight(0.0)      # :10-11
        self.SetForceWeight(0.0)
        self._F_thr_map = {}
        for nm in self._contact_names:
            self.SetContactNormal(nm, [0.0, 0.0, 1.0])  # :13-19
            self._F_thr_map[nm] = self.GetForceThreshold(nm)

    def SetLiftingContact(self, contact_name):  # :27-37
        self._F_thr_map[contact_name] = self.GetForceThreshold(contact_name)
        self.SetForceThreshold(contact_name, 0.0)
        self.SetForceBounds(contact_name, np.zeros(3), np.zeros(3))

    def GetLiftingContacts(self):  # :40-56
        out = []
        for nm in self._contact_names:
            lb, ub = self.GetForceBounds(nm)
            if (lb == 0.0).all() and (ub == 0.0).all():
                out.append(nm)
        return out

    def IsLiftingContact(self, contact_name):
        return contact_name in self.GetLiftingContacts()

    def ResetLiftingContact(self, contact_name):  # :74-88
        if not self.IsLiftingContact(contact_name):
            raise RuntimeError(f"'{contact_name}' is not a lifting contact.")
        self.SetForceBounds(contact_name, -1e3 * np.ones(3), 1e3 * np.ones(3))
        self.SetForceThreshold(contact_name, self._F_thr_map[contact_name])

    def SetContactPosition(self, contact_name, pos_ref):  # :91-97
        self.SetPosBounds(contact_name, pos_ref, pos_ref)

    def GetContactPosition(self, contact_name):  # :100-111
        lb, ub = self.GetPosBounds(contact_name)
        if (lb != ub).any():
            raise RuntimeError(f"Contact position for '{contact_name}' not set")
        return lb

    def SetContactNormal(self, contact_name, n_ref):  # :114-129
        self._need(contact_name)
        self.SetNormalBounds(contact_name, n_ref, n_ref)

    def GetContactNormal(self, contact_name):  # :132-143
        lb, ub = self.GetNormalBounds(contact_name)
        if (lb != ub).any():
            raise RuntimeError(f"Contact normal for '{contact_name}' not set")
        return lb

    def SetMu(self, mu):  # :146-156
        if mu <= 0.0:
            raise ValueError("Invalid friction coefficient")
        self._cpl_problem.SetMu(mu)
