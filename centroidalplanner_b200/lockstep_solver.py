"""Lock-step batched solve driver: N instances of one CplProblem shape solved together, one batched evaluation
(one kernel launch) per solver callback round.  SURVEY.md §8(f) rank 1 -- the caller side of the hot path.

What it stands in for.  The reference solves ONE instance per `cpl::CentroidalPlanner::Solve()` call with
`ifopt::IpoptSolver` (src/CentroidalPlanner.cpp:22-34; IPOPT's interior-point line-search method, `limited-memory`
Hessian approximation, ifopt's defaults listed in SURVEY Appendix B.8).  IPOPT is a host library that is NOT part of
this repository nor of its image.  The production integration keeps it: one IPOPT thread per instance over the IFOPT
views of `cplb/ifopt_views.hpp` in lock-step mode (INTEGRATION.md §2).  This module is the same driver loop with the
solver written out, so that the batched evaluator can be exercised -- and the reference's own post-solve assertions
(tests/TestBasic.cpp) checked -- by a real NLP solve without IPOPT:

  * the four IpoptAdapter callbacks become ONE `problem.eval(x, g, jac, cost, grad)` per iteration for all N instances,
    one widened `eval(jac, grad)` of N (n_free + 1) points for the Hessian differences and one widened `eval(g, cost)` per
    group of four line-search candidates;
  * the algorithm is the textbook primal-dual interior-point method IPOPT implements (Waechter & Biegler 2006, §2-3:
    slack reformulation of inequality rows, log barrier on bounds, fraction-to-boundary rule, monotone barrier update,
    gradient-based scaling with nlp_scaling_max_gradient = 100, bound_push / bound_frac initialisation, bound relaxation,
    kappa_sigma safeguard of the bound multipliers, fixed variables removed, second-order correction, `tol = 1e-3` as
    ifopt sets it).  Where it departs from IPOPT: the Lagrangian Hessian is a forward difference of the batched gradient
    and Jacobian instead of L-BFGS (the reference runs `limited-memory`), with an inertia-free curvature test and
    Levenberg-Marquardt damping for the directions the cost is flat in (ForceWeight 0); an l1 merit backtracking line
    search with slack reset replaces the filter; and a minimum-norm feasibility polish takes the constraints from
    IPOPT's constr_viol_tol (1e-4) to 1e-9 after the optimality test has passed.
    It is NOT IPOPT: iterates differ, solutions agree to the tolerance (local minima of the same NLP).

Everything is torch on the device of `x0` (fp64): the evaluation kernels read x where the linear algebra left it, so a
solve never crosses PCIe.  The problem object only needs `n, m, nnz, eval(), GetJacobianStructure(),
GetBoundsOnOptimizationVariables(), GetBoundsOnConstraints()`; tests drive the identical loop with the CPU oracle
behind that interface to compare trajectories.
"""
from __future__ import annotations

import dataclasses

import numpy as np
import torch

INF = 1.0e19  # ifopt: inf = 1.0e20 (SURVEY Appendix B.9); anything beyond 1e19 counts as "no bound" (IPOPT nlp_*_bound_inf)

SUCCESS = 0
MAX_ITER = 1
INVALID_NUMBER = 2
STATUS_NAMES = {SUCCESS: "Solve_Succeeded", MAX_ITER: "Maximum_Iterations_Exceeded", INVALID_NUMBER: "Invalid_Number_Detected"}


@dataclasses.dataclass
class SolveResult:
    x: torch.Tensor            # (N, n) final iterates (instance-major, IPOPT column order)
    status: torch.Tensor       # (N,) int64, see STATUS_NAMES
    iterations: torch.Tensor   # (N,) iterations each instance needed
    cost: torch.Tensor         # (N,) unscaled objective at x
    constr_viol: torch.Tensor  # (N,) max unscaled violation of constraint bounds at x
    dual_inf: torch.Tensor     # (N,) scaled dual infeasibility at x
    rounds: int                # lock-step rounds executed (= batched full evaluations - 1)
    evaluations: int           # batched evaluator calls (kernel launches) in total: full + Hessian differences + line-search trials
    instance_evaluations: int  # instances evaluated in total over those calls
    lam: torch.Tensor          # (N, m) constraint multipliers (unscaled)
    tail_instances: int = 0    # native round only: instances that finished on their own after the lock-step rounds

    def ok(self):
        return bool((self.status == SUCCESS).all())


class LockStepInteriorPoint:
    """Batched primal-dual interior-point solver; see the module docstring.  Options carry IPOPT's names where the
    meaning is IPOPT's (`tol`, `max_iter`, `mu_init`, `bound_push`, `bound_frac`, `nlp_scaling_max_gradient`)."""

    def __init__(self, tol=1e-3, max_iter=500, mu_init=0.1, bound_push=1e-2, bound_frac=1e-2,
                 nlp_scaling_max_gradient=100.0, constr_viol_tol=1e-4, polish_viol_tol=1e-9, bound_relax_factor=1e-8,
                 max_backtracks=30, compact=True, compact_min=64, verbose=False):
        self.tol = float(tol)
        self.max_iter = int(max_iter)
        self.mu_init = float(mu_init)
        self.bound_push = float(bound_push)
        self.bound_frac = float(bound_frac)
        self.max_gradient = float(nlp_scaling_max_gradient)
        self.constr_viol_tol = float(constr_viol_tol)
        self.polish_viol_tol = float(polish_viol_tol)
        self.bound_relax = float(bound_relax_factor)
        self.max_backtracks = int(max_backtracks)
        self.compact = bool(compact)
        self.compact_min = int(compact_min)
        self.verbose = verbose

    # ---- helpers -----------------------------------------------------------------------------------------------
    @staticmethod
    def _push_inside(v, lo, hi, has_lo, has_hi, k1, k2):
        """IPOPT's starting-point projection (Waechter & Biegler 2006, §3.6)."""
        span = torch.where(has_lo & has_hi, hi - lo, torch.full_like(lo, float("inf")))
        pl = torch.minimum(k1 * torch.clamp(lo.abs(), min=1.0), k2 * span)
        pu = torch.minimum(k1 * torch.clamp(hi.abs(), min=1.0), k2 * span)
        v = torch.where(has_lo, torch.maximum(v, lo + pl), v)
        v = torch.where(has_hi, torch.minimum(v, hi - pu), v)
        return v

    def Solve(self, problem, x0, per_instance=None):
        """Solve all N instances from the starting points x0 (N, n).  `per_instance` is forwarded to every evaluation
        (instances that are different problems of one shape, INTEGRATION.md §4b)."""
        x = torch.as_tensor(x0).to(torch.float64).contiguous().clone()
        dev, f64 = x.device, torch.float64
        N, n = x.shape
        m = problem.m
        assert n == problem.n

        iRow, jCol = problem.GetJacobianStructure()
        iRow_t = torch.as_tensor(iRow.astype(np.int64), device=dev)
        jCol_t = torch.as_tensor(jCol.astype(np.int64), device=dev)
        flat = iRow_t * n + jCol_t
        xl_np, xu_np = problem.GetBoundsOnOptimizationVariables()
        cl_np, cu_np = problem.GetBoundsOnConstraints()
        xl, xu = torch.as_tensor(xl_np, device=dev), torch.as_tensor(xu_np, device=dev)
        cl, cu = torch.as_tensor(cl_np, device=dev), torch.as_tensor(cu_np, device=dev)
        fixed = xl == xu                              # fixed_variable_treatment = make_parameter
        x_orig_lo, x_orig_hi = xl.clone(), xu.clone()
        rl = self.bound_relax * torch.clamp(xl.abs(), min=1.0)       # bound_relax_factor: an active row or variable keeps an interior
        ru = self.bound_relax * torch.clamp(xu.abs(), min=1.0)
        xl = torch.where(fixed, xl, xl - rl)
        xu = torch.where(fixed, xu, xu + ru)
        x_lo, x_hi = (xl > -INF) & ~fixed, (xu < INF) & ~fixed
        is_eq = cl == cu
        cl_r = torch.where(is_eq, cl, cl - self.bound_relax * torch.clamp(cl.abs(), min=1.0))
        cu_r = torch.where(is_eq, cu, cu + self.bound_relax * torch.clamp(cu.abs(), min=1.0))
        s_lo, s_hi = (cl > -INF) & ~is_eq, (cu < INF) & ~is_eq
        ineq = ~is_eq
        x = torch.where(fixed, xl.expand_as(x), x)
        x = self._push_inside(x, xl, xu, x_lo, x_hi, self.bound_push, self.bound_frac)
        free_f = (~fixed).to(f64)
        ineq_f = ineq.to(f64)
        free_idx = torch.nonzero(~fixed).flatten()
        nf = int(free_idx.numel())

        def repeat_params(k):
            """per-instance parameter arrays repeated k times along the instance axis (difference points of instance i
            are instances i*k .. i*k+k-1 of the widened batch)."""
            if per_instance is None:
                return {}
            return {"per_instance": {key: torch.repeat_interleave(torch.as_tensor(v, device=dev), k, dim=0) for key, v in per_instance.items()}}

        kw1 = {} if per_instance is None else {"per_instance": {k: torch.as_tensor(v, device=dev) for k, v in per_instance.items()}}
        kwh = repeat_params(nf + 1)
        evaluations = 0
        instance_evals = 0

        slot_free = ~fixed[jCol_t]                     # Jacobian slots in columns of fixed variables never enter (they may be 0/0, SURVEY Q3)

        def dense(jac_vals, rows):
            J = torch.zeros(rows, m * n, dtype=f64, device=dev)
            J[:, flat] = torch.where(slot_free, jac_vals, torch.zeros_like(jac_vals))
            return J.view(rows, m, n)

        def on_dev(out):
            # the host path of the product returns NumPy arrays, the device path torch tensors
            return {k: (None if v is None else torch.as_tensor(v, device=dev)) for k, v in out.items() if k in ("g", "jac", "cost", "grad")}

        def full_eval(xx):
            nonlocal evaluations, instance_evals
            evaluations += 1
            instance_evals += N
            out = on_dev(problem.eval(xx, g=True, jac=True, cost=True, grad=True, **kw1))
            return out["cost"], torch.where(fixed, torch.zeros_like(out["grad"]), out["grad"]), out["g"], dense(out["jac"], N)

        kw_rep = {1: kw1}

        def trial_eval(xx, K=1):
            nonlocal evaluations, instance_evals
            evaluations += 1
            instance_evals += N * K
            if K not in kw_rep:
                kw_rep[K] = repeat_params(K)
            out = on_dev(problem.eval(xx, g=True, jac=False, cost=True, grad=False, **kw_rep[K]))
            return out["cost"], out["g"]

        f, df, c, J = full_eval(x)
        bad0 = ~(torch.isfinite(f) & torch.isfinite(df).all(1) & torch.isfinite(c).all(1) & torch.isfinite(J).all(2).all(1))
        # gradient-based scaling at the starting point (nlp_scaling_method = gradient-based)
        Jn = torch.nan_to_num(J, nan=0.0, posinf=0.0, neginf=0.0) * free_f
        dc = torch.clamp(self.max_gradient / Jn.abs().amax(2).clamp(min=1e-300), max=1.0)             # (N, m)
        dfn = torch.nan_to_num(df, nan=0.0, posinf=0.0, neginf=0.0) * free_f
        dobj = torch.clamp(self.max_gradient / dfn.abs().amax(1).clamp(min=1e-300), max=1.0)          # (N,)
        sl, su = dc * cl_r, dc * cu_r                                                                   # scaled (relaxed) slack bounds

        def scaled(f, df, c, J):
            return dobj * f, dobj[:, None] * df, dc * c, dc[:, :, None] * J

        def lagrangian_hessian(xx, df_s, J_s, lam_s):
            """Hessian of f + lam^T c in x (scaled problem) by forward differences of the batched gradient and Jacobian:
            the nf difference points of every instance ride in ONE widened evaluation of N*(nf+1) instances -- what a
            per-instance CPU solver cannot afford (IPOPT in the reference runs `limited-memory`) costs the batched
            evaluator a fraction of a millisecond."""
            nonlocal evaluations, instance_evals
            eps = 1e-7 * torch.clamp(xx[:, free_idx].abs(), min=1.0)                                  # (N, nf)
            X = xx[:, None, :].repeat(1, nf + 1, 1)                                                     # (N, nf+1, n); slot nf = base point
            ar = torch.arange(nf, device=dev)
            X[:, ar, free_idx] += eps
            evaluations += 1
            instance_evals += N * (nf + 1)
            out = on_dev(problem.eval(X.view(N * (nf + 1), n), g=False, jac=True, cost=False, grad=True, **kwh))
            w = (dc * lam_s)[:, iRow_t]                                                                 # (N, nnz) row multipliers per slot
            gl = dobj[:, None, None] * out["grad"].view(N, nf + 1, n)
            jv = out["jac"].view(N, nf + 1, -1)
            gl = gl.index_add(2, jCol_t, torch.where(slot_free, jv, torch.zeros_like(jv)) * w[:, None, :])   # grad f + J^T lam at every point
            gl = torch.where(fixed, torch.zeros_like(gl), gl)
            Hc = (gl[:, :nf, :] - gl[:, nf:, :]) / eps[:, :, None]                                      # row a = d(grad L)/d x_free[a]
            H = torch.zeros(N, n, n, dtype=f64, device=dev)
            H[:, free_idx, :] = Hc
            H = H * free_f[:, None] * free_f[None, :]
            return 0.5 * (H + H.transpose(1, 2))

        f, df, c, J = scaled(f, df, c, J)
        # slacks: s = c(x) pushed inside its bounds on inequality rows, the bound itself on equality rows
        s = torch.where(is_eq, sl, self._push_inside(c, sl, su, s_lo.expand_as(c), s_hi.expand_as(c), self.bound_push, self.bound_frac))
        one = torch.ones((), dtype=f64, device=dev)
        vxl = torch.where(x_lo, one, 0 * one).expand(N, n).clone()
        vxu = torch.where(x_hi, one, 0 * one).expand(N, n).clone()
        vsl = torch.where(s_lo, one, 0 * one).expand(N, m).clone()
        vsu = torch.where(s_hi, one, 0 * one).expand(N, m).clone()
        lam = torch.zeros(N, m, dtype=f64, device=dev)
        mu = torch.full((N,), self.mu_init, dtype=f64, device=dev)
        status = torch.full((N,), -1, dtype=torch.int64, device=dev)
        status[bad0] = INVALID_NUMBER
        iters = torch.zeros(N, dtype=torch.int64, device=dev)
        big = torch.full((), float("inf"), dtype=f64, device=dev)
        x_lo_f, x_hi_f, s_lo_f, s_hi_f = x_lo.to(f64), x_hi.to(f64), s_lo.to(f64), s_hi.to(f64)
        delta_last = torch.zeros(N, dtype=f64, device=dev)
        delta_lm = torch.zeros(N, dtype=f64, device=dev)
        polish = torch.zeros(N, dtype=torch.bool, device=dev)
        eyeK = torch.eye(n + m, dtype=f64, device=dev)

        def gaps(x, s):
            gxl = torch.where(x_lo, x - xl, one)
            gxu = torch.where(x_hi, xu - x, one)
            gsl = torch.where(s_lo, s - sl, one)
            gsu = torch.where(s_hi, su - s, one)
            return gxl, gxu, gsl, gsu

        def barrier(f, x, s, mu):
            gxl, gxu, gsl, gsu = gaps(x, s)
            lb = (torch.log(gxl) * x_lo_f + torch.log(gxu) * x_hi_f).sum(1) + (torch.log(gsl) * s_lo_f + torch.log(gsu) * s_hi_f).sum(1)
            return f - mu * lb

        comp_mask = torch.cat([x_lo_f, x_hi_f, s_lo_f, s_hi_f])

        def kkt_residuals(df, c, J, s, lam, vxl, vxu, vsl, vsu, x):
            """Scaled optimality error of Waechter & Biegler eq. (5) without its mu-dependent part: dual and primal
            infeasibility, the multiplier scaling s_d, and the gap x multiplier products the complementarity error is made of."""
            gxl, gxu, gsl, gsu = gaps(x, s)
            rx = (df + torch.einsum("nij,ni->nj", J, lam) - vxl + vxu) * free_f
            rs = (-lam - vsl + vsu) * ineq_f
            h = c - s
            nmul = (m + 2 * n + 2 * m)
            sd = torch.clamp((lam.abs().sum(1) + vxl.sum(1) + vxu.sum(1) + vsl.sum(1) + vsu.sum(1)) / nmul, min=100.0) / 100.0
            dual = torch.maximum(rx.abs().amax(1), rs.abs().amax(1)) / sd
            prim = h.abs().amax(1)
            prods = torch.cat([gxl * vxl, gxu * vxu, gsl * vsl, gsu * vsu], dim=1)
            return dual, prim, sd, prods

        def complementarity(prods, sd, mu_t):
            return ((prods - mu_t[:, None]) * comp_mask).abs().amax(1) / sd

        eq_f = is_eq.to(f64)
        cu_s, cl_s = dc * cu, dc * cl                     # scaled ORIGINAL row bounds (sl / su are the relaxed ones)

        def polish_residual(cc):
            """What the feasibility polish drives to zero: equality residuals and excess over the original inequality bounds."""
            exc = torch.clamp(cc - cu_s, min=0.0) * s_hi_f + torch.clamp(cl_s - cc, min=0.0) * s_lo_f
            return torch.maximum(((cc - sl) * eq_f).abs().amax(1), exc.amax(1))

        N0 = N
        orig = torch.arange(N0, device=dev)            # original index of every instance still in the working set
        out = {"x": torch.empty(N0, n, dtype=f64, device=dev), "status": torch.empty(N0, dtype=torch.int64, device=dev),
               "iters": torch.empty(N0, dtype=torch.int64, device=dev), "cost": torch.empty(N0, dtype=f64, device=dev),
               "viol": torch.empty(N0, dtype=f64, device=dev), "dual": torch.empty(N0, dtype=f64, device=dev),
               "lam": torch.empty(N0, m, dtype=f64, device=dev)}

        def flush():
            """Current state of the working set -> the full-size result buffers."""
            out["x"][orig] = torch.minimum(torch.maximum(x, x_orig_lo), x_orig_hi)          # honor_original_bounds
            out["status"][orig] = status
            out["iters"][orig] = iters
            out["cost"][orig] = f / dobj
            out["viol"][orig] = ((torch.clamp(sl - c, min=0) + torch.clamp(c - su, min=0)) / dc).amax(1)
            out["dual"][orig] = kkt_residuals(df, c, J, s, lam, vxl, vxu, vsl, vsu, x)[0]
            out["lam"][orig] = lam * dc / dobj[:, None]

        rounds = 0
        for it in range(self.max_iter + 1):
            dual0, prim0, sd0, prods0 = kkt_residuals(df, c, J, s, lam, vxl, vxu, vsl, vsu, x)
            comp0 = complementarity(prods0, sd0, torch.zeros_like(mu))
            E0 = torch.stack([dual0, prim0, comp0]).amax(0)
            viol = (torch.clamp(sl - c, min=0) + torch.clamp(c - su, min=0)) / dc                           # unscaled row violation (relaxed bounds)
            vmax = viol.amax(1)
            # IPOPT's test (scaled error <= tol, unscaled violation <= constr_viol_tol) switches an instance to the
            # feasibility polish; it is done when the constraints hold to polish_viol_tol as well -- and the test still holds there:
            # a polished iterate whose scaled error grew past tol (the polish moves x with the multipliers frozen) leaves the
            # polish and takes Newton steps again (csrc/cplb_solver_core.hpp, phase_round_begin)
            converged = (status < 0) & (E0 <= self.tol) & (vmax <= self.constr_viol_tol)
            unpolish = ~converged & polish & (vmax <= self.polish_viol_tol)     # ... and its Newton steps start undamped
            delta_lm = torch.where(unpolish, torch.zeros_like(delta_lm), delta_lm)
            polish = polish & ~unpolish | converged
            done_now = (status < 0) & polish & (vmax <= self.polish_viol_tol)
            status = torch.where(done_now, torch.full_like(status, SUCCESS), status)
            nonfinite = (status < 0) & ~(torch.isfinite(E0))
            status = torch.where(nonfinite, torch.full_like(status, INVALID_NUMBER), status)
            active = status < 0
            if self.verbose:
                i0 = 0
                print(f"it {it:3d} active {int(active.sum()):5d} | inst0: f {float(f[i0] / dobj[i0]):.6e} prim {float(prim0[i0]):.2e} dual {float(dual0[i0]):.2e} "
                      f"comp {float(comp0[i0]):.2e} mu {float(mu[i0]):.1e}")
            n_active = int(active.sum())
            if n_active == 0 or it == self.max_iter:
                break
            if self.compact and N >= self.compact_min and 2 * n_active <= N:
                # Lock-step rounds cost the same whether an instance is still iterating or not: once half of the working set
                # has finished, the finished ones are written out and dropped (instances are independent, so the others'
                # iterates do not change).
                flush()
                keep = torch.nonzero(active).flatten()
                (x, s, lam, vxl, vxu, vsl, vsu, mu, status, iters, delta_last, delta_lm, polish, f, df, c, J, dc, dobj, sl, su,
                 cu_s, cl_s, orig, dual0, prim0, sd0, prods0, active) = (
                    t[keep] for t in (x, s, lam, vxl, vxu, vsl, vsu, mu, status, iters, delta_last, delta_lm, polish, f, df, c, J,
                                      dc, dobj, sl, su, cu_s, cl_s, orig, dual0, prim0, sd0, prods0, active))
                N = n_active
                if per_instance is not None:
                    per_instance = {k: torch.as_tensor(v, device=dev)[keep] for k, v in per_instance.items()}
                    kw1 = {"per_instance": per_instance}
                    kwh = repeat_params(nf + 1)
                    kw_rep.clear()
                    kw_rep[1] = kw1
            rounds += 1
            iters += active.to(torch.int64)

            # monotone barrier update (Waechter & Biegler eq. 7): shrink mu while the barrier problem is solved to kappa_eps * mu
            dp0 = torch.maximum(dual0, prim0)
            for _ in range(4):
                Emu = torch.maximum(dp0, complementarity(prods0, sd0, mu))
                shrink = active & (Emu <= 10.0 * mu) & (mu > self.tol / 10.0)
                mu = torch.where(shrink, torch.clamp(torch.minimum(0.2 * mu, mu ** 1.5), min=self.tol / 10.0), mu)
            tau = torch.clamp(1.0 - mu, min=0.99)

            # ---- primal-dual Newton step with the slacks eliminated --------------------------------------------
            W = lagrangian_hessian(x, df, J, lam)
            gxl, gxu, gsl, gsu = gaps(x, s)
            mu_c = mu[:, None]
            sig_x = vxl / gxl * x_lo_f + vxu / gxu * x_hi_f
            sig_s = vsl / gsl * s_lo_f + vsu / gsu * s_hi_f
            r_x = (df + torch.einsum("nij,ni->nj", J, lam) - mu_c / gxl * x_lo_f + mu_c / gxu * x_hi_f) * free_f
            r_s = (-lam - mu_c / gsl * s_lo_f + mu_c / gsu * s_hi_f) * ineq_f
            h = c - s
            D = torch.where(ineq, 1.0 / sig_s.clamp(min=1e-300), torch.zeros_like(sig_s))                   # (N, m)
            Jf = J * free_f                                                                                # zero the fixed columns
            H0 = W + torch.diag_embed(sig_x * free_f + (1.0 - free_f))
            delta_c = 1e-8 * mu ** 0.25
            rhs = torch.cat([-r_x, -h - D * r_s], dim=1)
            Kbase = torch.zeros(N, n + m, n + m, dtype=f64, device=dev)
            Kbase[:, :n, n:] = Jf.transpose(1, 2)
            Kbase[:, n:, :n] = Jf
            Kbase[:, n:, n:] = -torch.diag_embed(D + delta_c[:, None])
            # inertia-free regularisation (Chiang & Zavala 2016): raise delta_w until the step sees positive curvature
            delta = delta_lm.clone()
            need = active.clone()
            dx = torch.zeros(N, n, dtype=f64, device=dev)
            dlam = torch.zeros(N, m, dtype=f64, device=dev)
            ds = torch.zeros(N, m, dtype=f64, device=dev)
            quad = torch.zeros(N, dtype=f64, device=dev)
            for _reg in range(14):
                H = H0 + torch.diag_embed(delta[:, None] * free_f.expand(N, n))
                K = Kbase.clone()
                K[:, :n, :n] = H
                okK = torch.isfinite(K).all(2).all(1) & torch.isfinite(rhs).all(1)
                K = torch.where(okK[:, None, None], K, eyeK)
                LU_t, piv_t = torch.linalg.lu_factor(K)
                sol = torch.linalg.lu_solve(LU_t, piv_t, torch.where(okK[:, None], rhs, torch.zeros_like(rhs))[:, :, None])[:, :, 0]
                if _reg == 0:
                    LU, piv = LU_t, piv_t
                else:
                    LU = torch.where(need[:, None, None], LU_t, LU)
                    piv = torch.where(need[:, None], piv_t, piv)
                dx_t, dlam_t = sol[:, :n] * free_f, sol[:, n:]
                ds_t = (D * (dlam_t - r_s)) * ineq_f
                quad_t = torch.einsum("ni,nij,nj->n", dx_t, H, dx_t) + (sig_s * ds_t * ds_t).sum(1)
                good = torch.isfinite(sol).all(1) & (quad_t >= 1e-8 * ((dx_t * dx_t).sum(1) + (ds_t * ds_t).sum(1)))
                last = _reg == 13
                take = need & (good | last)
                dx = torch.where(take[:, None], dx_t, dx)
                dlam = torch.where(take[:, None], dlam_t, dlam)
                ds = torch.where(take[:, None], ds_t, ds)
                quad = torch.where(take, quad_t, quad)
                delta_last = torch.where(take, delta, delta_last)
                need = need & ~take
                if not bool(need.any()):
                    break
                delta = torch.where(need, torch.clamp(delta * 8.0, min=1e-4), delta)
            bad_step = ~(torch.isfinite(dx).all(1) & torch.isfinite(dlam).all(1))
            dx = torch.where(bad_step[:, None], torch.zeros_like(dx), dx)
            dlam = torch.where(bad_step[:, None], torch.zeros_like(dlam), dlam)
            ds = torch.where(bad_step[:, None], torch.zeros_like(ds), ds)
            dvxl = (mu_c / gxl - vxl - vxl / gxl * dx) * x_lo_f
            dvxu = (mu_c / gxu - vxu + vxu / gxu * dx) * x_hi_f
            dvsl = (mu_c / gsl - vsl - vsl / gsl * ds) * s_lo_f
            dvsu = (mu_c / gsu - vsu + vsu / gsu * ds) * s_hi_f

            def max_step(val, dval, mask_f):
                # largest a in (0,1] with val + a*dval >= (1 - tau) * val where the gap shrinks
                a = torch.where((dval < 0) & (mask_f > 0), -tau[:, None] * val / dval, big)
                return a.amin(1)

            a_p = torch.stack([max_step(gxl, dx, x_lo_f), max_step(gxu, -dx, x_hi_f),
                               max_step(gsl, ds, s_lo_f), max_step(gsu, -ds, s_hi_f)]).amin(0).clamp(max=1.0)
            a_d = torch.stack([max_step(vxl, dvxl, x_lo_f), max_step(vxu, dvxu, x_hi_f),
                               max_step(vsl, dvsl, s_lo_f), max_step(vsu, dvsu, s_hi_f)]).amin(0).clamp(max=1.0)

            # ---- l1 merit line search on the primal step, second-order correction on the first trial ---------------
            phi0 = barrier(f, x, s, mu)
            h1 = h.abs().sum(1)
            gphi_x = (df - mu_c / gxl * x_lo_f + mu_c / gxu * x_hi_f) * free_f
            gphi_s = (-mu_c / gsl * s_lo_f + mu_c / gsu * s_hi_f) * ineq_f
            dphi = (gphi_x * dx).sum(1) + (gphi_s * ds).sum(1)
            nu_need = (dphi + 0.5 * quad.clamp(min=0)) / (0.9 * h1.clamp(min=1e-300))
            nu = torch.maximum(nu_need.clamp(min=0.0), (lam + dlam).abs().amax(1)) * 1.1 + 1e-3
            Dm = dphi - nu * h1
            merit0 = phi0 + nu * h1
            pol = active & polish
            if bool(pol.any()):
                # feasibility polish: minimum-norm Newton step, x only (multipliers stay), on the equality rows and on the
                # inequality rows that sit beyond their ORIGINAL bound (pulled back onto it; the relaxed bound is the test)
                over = ineq & s_hi & (c > cu_s)
                under = ineq & s_lo & (c < cl_s)
                act_f = (is_eq | over | under).to(f64)
                r_p = torch.where(over, c - cu_s, torch.where(under, c - cl_s, (c - sl) * eq_f))
                Je = Jf * act_f[:, :, None]
                M = Je @ Je.transpose(1, 2) + torch.diag_embed((1.0 - act_f) + 1e-14)
                M = torch.where(torch.isfinite(M).all(2).all(1)[:, None, None], M, torch.eye(m, dtype=f64, device=dev))
                y = torch.linalg.solve(M, r_p[:, :, None])
                dx_p = -(Je.transpose(1, 2) @ y)[:, :, 0] * free_f
                dx_p = torch.where(torch.isfinite(dx_p).all(1)[:, None], dx_p, torch.zeros_like(dx_p))
                a_pp = torch.stack([max_step(gxl, dx_p, x_lo_f), max_step(gxu, -dx_p, x_hi_f)]).amin(0).clamp(max=1.0)
                dx = torch.where(pol[:, None], dx_p, dx)
                ds = torch.where(pol[:, None], torch.zeros_like(ds), ds)
                dlam = torch.where(pol[:, None], torch.zeros_like(dlam), dlam)
                a_p = torch.where(pol, a_pp, a_p)
                a_d = torch.where(pol, torch.zeros_like(a_d), a_d)
            R0 = polish_residual(c)
            alpha = torch.where(active, a_p, torch.zeros_like(a_p))
            tiny = (dx.abs() / (1.0 + x.abs())).amax(1) < 1e-13          # tiny_step_tol: below rounding the merit test is noise
            accepted = ~active
            x_new, s_new = x, s
            dlam_used = dlam

            def try_points(X, S_lin, AL):
                """Merit test of K candidate points per instance in ONE widened evaluation: X (N, K, n), S_lin (N, K, m) the
                linearly stepped slacks, AL (N, K) the step lengths -> ok (N, K), slacks (N, K, m), row values (N, K, m)."""
                K = X.shape[1]
                ft, ct = trial_eval(X.reshape(N * K, n), K)
                ft, ct = dobj[:, None] * ft.view(N, K), dc[:, None, :] * ct.view(N, K, m)
                keep = (mu / nu)[:, None, None]
                st = torch.where(s_hi & ~s_lo, torch.minimum(ct, su[:, None, :] - keep), S_lin)      # slack reset (Nocedal & Wright 2006, §19.3): the row value itself, mu/nu inside its bound
                st = torch.where(s_lo & ~s_hi, torch.maximum(ct, sl[:, None, :] + keep), st)
                gxl = torch.where(x_lo, X - xl, one)
                gxu = torch.where(x_hi, xu - X, one)
                gsl = torch.where(s_lo, st - sl[:, None, :], one)
                gsu = torch.where(s_hi, su[:, None, :] - st, one)
                lb = (torch.log(gxl) * x_lo_f + torch.log(gxu) * x_hi_f).sum(2) + (torch.log(gsl) * s_lo_f + torch.log(gsu) * s_hi_f).sum(2)
                mt = (ft - mu[:, None] * lb) + nu[:, None] * (ct - st).abs().sum(2)
                ok = torch.isfinite(mt) & (mt <= (merit0 + 10.0 * 2.2e-16 * merit0.abs())[:, None] + 1e-4 * AL * Dm[:, None])
                # polishing instances: the slack of a strictly satisfied inequality row is the row value; accept when the
                # polish residual shrinks
                inside = (~s_lo | (ct > sl[:, None, :])) & (~s_hi | (ct < su[:, None, :]))
                st_p = torch.where(ineq & inside, ct, s[:, None, :])
                exc = torch.clamp(ct - cu_s[:, None, :], min=0.0) * s_hi_f + torch.clamp(cl_s[:, None, :] - ct, min=0.0) * s_lo_f
                R_t = torch.maximum(((ct - sl[:, None, :]) * eq_f).abs().amax(2), exc.amax(2))
                ok_p = torch.isfinite(ct).all(2) & (R_t < R0[:, None])
                st = torch.where(pol[:, None, None], st_p, st)
                ok = torch.where(pol[:, None], ok_p, ok)
                return ok, st, ct

            # Candidates alpha0 * 2^-k are tried four at a time (one widened launch instead of four round trips); the first
            # acceptable one in the order full step, second-order correction, 1/2, 1/4, ... is taken, as a sequential
            # backtracking search would.
            KC = 4
            scale = 0.5 ** torch.arange(KC, device=dev, dtype=f64)
            base = alpha.clone()                                  # alpha0 * 2^-(4 g) of the current group
            tried = 0
            _ls = 0
            while tried < self.max_backtracks:
                AL = base[:, None] * scale[None, :]
                X = x[:, None, :] + AL[:, :, None] * dx[:, None, :]
                ok, st, ct = try_points(X, s[:, None, :] + AL[:, :, None] * ds[:, None, :], AL)
                ok = ok | (tiny[:, None] & torch.isfinite(ct).all(2))
                if tried + KC > self.max_backtracks:
                    ok[:, self.max_backtracks - tried:] = False
                if tried == 0:
                    first_ok = ok[:, 0]
                    take = first_ok & ~accepted
                    x_new = torch.where(take[:, None], X[:, 0], x_new)
                    s_new = torch.where(take[:, None], st[:, 0], s_new)
                    accepted = accepted | first_ok
                    if not bool(accepted.all()):
                        # second-order correction (Waechter & Biegler 2006, §2.4): same matrix, constraint residual of the
                        # rejected trial point added to the right-hand side -- removes the Maratos effect on the bilinear
                        # moment rows and the friction cones
                        h_soc = alpha[:, None] * h + (ct[:, 0] - (s + alpha[:, None] * ds))
                        rhs_c = torch.cat([-r_x, -h_soc - D * r_s], dim=1)
                        sol_c = torch.linalg.lu_solve(LU, piv, torch.where(okK[:, None], rhs_c, torch.zeros_like(rhs_c))[:, :, None])[:, :, 0]
                        dx_c, dlam_c = sol_c[:, :n] * free_f, sol_c[:, n:]
                        ds_c = (D * (dlam_c - r_s)) * ineq_f
                        fin_c = torch.isfinite(sol_c).all(1)
                        a_c = torch.stack([max_step(gxl, dx_c, x_lo_f), max_step(gxu, -dx_c, x_hi_f),
                                           max_step(gsl, ds_c, s_lo_f), max_step(gsu, -ds_c, s_hi_f)]).amin(0).clamp(max=1.0)
                        xc = torch.where(fin_c[:, None], x + a_c[:, None] * dx_c, x)
                        okc, stc, _ = try_points(xc[:, None, :], (s + a_c[:, None] * ds_c)[:, None, :], alpha[:, None])
                        takec = okc[:, 0] & fin_c & ~accepted & ~pol
                        x_new = torch.where(takec[:, None], xc, x_new)
                        s_new = torch.where(takec[:, None], stc[:, 0], s_new)
                        dlam_used = torch.where(takec[:, None], dlam_c, dlam_used)
                        accepted = accepted | takec
                # the first acceptable candidate of this group (for the first group: among 1/2, 1/4, 1/8)
                okg = ok.clone()
                if tried == 0:
                    okg[:, 0] = False
                any_ok = okg.any(1)
                kfirst = torch.argmax(okg.to(torch.int8), dim=1)
                take = any_ok & ~accepted
                idx = kfirst[:, None, None]
                x_new = torch.where(take[:, None], torch.gather(X, 1, idx.expand(N, 1, n))[:, 0], x_new)
                s_new = torch.where(take[:, None], torch.gather(st, 1, idx.expand(N, 1, m))[:, 0], s_new)
                alpha = torch.where(take, torch.gather(AL, 1, kfirst[:, None])[:, 0], alpha)
                accepted = accepted | any_ok
                tried += KC
                _ls = tried
                if bool(accepted.all()):
                    break
                base = base * scale[-1] * 0.5
            alpha = torch.where(accepted, alpha, a_p * 0.5 ** self.max_backtracks)
            dlam = dlam_used
            # Levenberg-Marquardt damping of the next step: a search that had to backtrack asks for a shorter step next
            # time, a full step relaxes the damping again (directions the cost is flat in -- ForceWeight 0 -- otherwise
            # produce Newton steps of hundreds of newtons that the nonlinear friction and moment rows reject)
            n_back = torch.log2((a_p / alpha.clamp(min=1e-300)).clamp(min=1.0)).round()
            n_back = torch.where(pol, torch.ones_like(n_back), n_back)
            delta_lm = torch.where(active & (n_back >= 2), torch.clamp(delta_last * 8.0, min=1e-6),
                                   torch.where(active & (n_back >= 1), torch.clamp(delta_last * 2.0, min=1e-6),
                                               torch.where(active, delta_last / 4.0, delta_last)))
            delta_lm = torch.where(delta_lm < 1e-12, torch.zeros_like(delta_lm), delta_lm).clamp(max=1.0)
            failed = ~accepted           # search exhausted: take the last (tiny) step
            if bool(failed.any()):
                x_new = torch.where(failed[:, None], x + alpha[:, None] * dx, x_new)
                s_new = torch.where(failed[:, None], s + alpha[:, None] * ds, s_new)
            if self.verbose:
                print(f"      a_p {float(a_p[0]):.2e} a_d {float(a_d[0]):.2e} alpha {float(alpha[0]):.2e} ls {_ls} nu {float(nu[0]):.2e} delta {float(delta_last[0]):.1e} "
                      f"|dx| {float(dx[0].abs().max()):.2e} |ds| {float(ds[0].abs().max()):.2e} Dm {float(Dm[0]):.2e} failed {bool(failed[0])}")
            alpha = torch.where(active, alpha, torch.zeros_like(alpha))
            a_dual = torch.where(active, a_d, torch.zeros_like(a_d))

            lam = lam + alpha[:, None] * dlam
            vxl = vxl + a_dual[:, None] * dvxl
            vxu = vxu + a_dual[:, None] * dvxu
            vsl = vsl + a_dual[:, None] * dvsl
            vsu = vsu + a_dual[:, None] * dvsu
            x, s = x_new, s_new
            f, df, c, J = scaled(*full_eval(x))
            # kappa_sigma safeguard (Waechter & Biegler eq. 16)
            gxl, gxu, gsl, gsu = gaps(x, s)
            ks = 1e10
            vxl = torch.minimum(torch.maximum(vxl, mu_c / (ks * gxl)), ks * mu_c / gxl) * x_lo_f
            vxu = torch.minimum(torch.maximum(vxu, mu_c / (ks * gxu)), ks * mu_c / gxu) * x_hi_f
            vsl = torch.minimum(torch.maximum(vsl, mu_c / (ks * gsl)), ks * mu_c / gsl) * s_lo_f
            vsu = torch.minimum(torch.maximum(vsu, mu_c / (ks * gsu)), ks * mu_c / gsu) * s_hi_f

        status = torch.where(status < 0, torch.full_like(status, MAX_ITER), status)
        flush()
        return SolveResult(x=out["x"], status=out["status"], iterations=out["iters"], cost=out["cost"], constr_viol=out["viol"],
                           dual_inf=out["dual"], rounds=rounds, evaluations=evaluations, instance_evaluations=instance_evals,
                           lam=out["lam"])


def default_start(problem, N=1, device=None):
    """A finite starting point for every instance.  The reference starts IPOPT at x = 0 (Variable3D.cpp:8-10), where the
    friction-cone Jacobian is 0/0 (SURVEY Q3) and a superquadric centred near the origin has a vanishing gradient; a
    solver that checks its derivatives needs something else: the CoM at the middle of its bounds (clipped to +-1), the
    contact positions spread towards alternating corners of theirs (80 % of the half range in x and y), normals (0,0,1)
    and the weight shared by the contacts with a tangential component so that no tangential-force norm vanishes."""
    lb, ub = problem.GetBoundsOnOptimizationVariables()
    n = problem.n
    nc = (n - 3) // 9
    lo, hi = np.maximum(lb, -1.0), np.minimum(ub, 1.0)
    mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
    x = mid.copy()
    corners = [(1.0, 1.0), (-1.0, 1.0), (-1.0, -1.0), (1.0, -1.0)]
    for k in range(nc):
        b = 3 + 9 * k
        sx, sy = corners[k % 4]
        shrink = 0.8 / (1 + k // 4)
        x[b:b + 3] = np.clip([1.0 + 0.5 * k, -1.0 + 0.25 * k, 981.0 / nc], lb[b:b + 3], ub[b:b + 3])
        x[b + 3] = mid[b + 3] + sx * shrink * half[b + 3]
        x[b + 4] = mid[b + 4] + sy * shrink * half[b + 4]
        x[b + 6:b + 9] = np.clip([0.0, 0.0, 1.0], lb[b + 6:b + 9], ub[b + 6:b + 9])
    x = np.tile(x, (N, 1))
    return torch.as_tensor(x, device=device)
