"""An optimality certificate for the results of the native solve round, computed outside the solver.

The solve (cplb_solve_device, and its CPU replay) returns x, the constraint multipliers lam, cost, constr_viol and dual_inf.
`certify` takes the problem's C oracle (one per instance for a per-instance sweep), the solver options, the starts x0 and those
outputs, evaluates g, the Jacobian, the cost and its gradient with the oracle AT THE RETURNED x, and measures, per instance:

* x      -- inside the original variable bounds, exactly (honor_original_bounds clips to them).
* cost   -- the oracle's cost at the returned x, bit for bit without pow() upstream (Ground, no environment), 1e-12 relative
            otherwise.  The solve reports the values of its final iterate, which is x unless the clipping moved an entry back onto
            its bound (include/cpl_batched.h).  A free entry lying exactly on an original bound may have been clipped by up to
            delta_j = bound_relax_factor * max(|bound|, 1); there the cost may differ by what moving that entry back by delta_j
            can change: the cost is a separable convex quadratic, so per entry at most max(|df_j| delta_j, f(x + delta_j e_j) - f(x))
            (convexity bounds the change on the segment by its first-order lower bound and its end point), plus 4 eps |f|.
* constr_viol -- max over rows of (cl_r - g)+ + (g - cu_r)+, with cl_r, cu_r the bounds the solver works with: equality rows
            exact, inequality rows relaxed by bound_relax_factor * max(|bound|, 1) (its slack bounds sl / su are these, scaled by
            dc).  The solver forms it as ((dc cl_r - dc g)+ + ...) / dc: within 4 eps max(|g|, |bounds|) (three roundings).  After
            clipping: within twice the first-order change sum_j |J_rj| delta_j of a row as well, and at most constr_viol_tol
            (what the convergence test guaranteed); otherwise at most polish_viol_tol (what SUCCEEDED requires).
* stationarity -- IPOPT's scaled dual infeasibility, with the pieces the solver does not return reconstructed or bounded.

Scaled measure (Waechter & Biegler 2006, sections 3.8 and 2.1; IPOPT's gradient-based scaling).  The solver works on
    min dobj f(x)   s.t.   dc_r g_r(x) = s_r,  sl_r <= s_r <= su_r,  xl <= x <= xu   (xl, xu relaxed)
with dobj = min(1, nlp_scaling_max_gradient / max_j |df_j(xs)|) and dc_r = min(1, nlp_scaling_max_gradient / max_j |J_rj(xs)|),
both at the projected start xs (bound_push / bound_frac, fixed variables at their value), maxima over the free columns.  The test
recomputes them from x0 with the same rule (`scaling`).  Its multipliers are lam_s = lam * dobj / dc (lam is returned unscaled,
IPOPT's sign convention L = f + lam^T g: lam_r >= 0 when the upper bound of row r is active, <= 0 when the lower one is).  The
scaled residuals of a free variable j and of an inequality row r are
    dobj (df_j + sum_r J_rj lam_r) - zl_j + zu_j      and      lam_s_r - vu_r + vl_r     (the slack stationarity)
and the convergence test asks their maximum divided by
    s_d = max(100, (sum |lam_s| + sum z + sum v) / (3m + 2n)) / 100
to be <= tol, with every gap * bound multiplier / s_d <= tol and the violation <= constr_viol_tol; a feasibility polish with the
multipliers frozen follows.  dual_inf is that maximum at the final iterate.

The bound multipliers z, v are not returned.  For each variable the certificate takes the most favourable z >= 0 that
complementarity allows, gap * z <= tol s_d: z in [-tol s_d / gap_u, tol s_d / gap_l], an open side where there is no bound, where
the gap is 0, or where the entry may have been clipped (the measured gap was then anywhere in (0, delta_j]).  The gap is to the
relaxed bound at the returned x.  For inequality rows the slack is not returned either: the row value stands in for it, and the
gap is the row's distance to its relaxed bound minus tol (the primal test bounds |dc g - s| <= tol), so a row counts as possibly
active unless it is inactive by more than that; a multiplier of the wrong sign on an active row, or a large one on an inactive
row, is left over.  s_d is computed from lam alone (sum |lam_s|; z, v >= 0 only make the true s_d larger), so the bar tol s_d is
never above the solver's own.

Tolerances of the stationarity checks, all from tol (SUCCEEDED means the scaled error is <= tol at the returned iterate):
    residual left over  <=  tol s_d + 16 eps (dobj |df_j| + sum_r |dc_r J_rj lam_s_r|)      (per column; per row 16 eps |lam_s_r|)
    dual_inf            <=  tol
    dual_inf            >=  (least residual left over with the widest z the solver can hold) / s_d_hi     (unclipped x only)
The test forms the residual exactly (Fraction arithmetic on the oracle's fp64 values); the solver's fp64 sum has at most 9 terms
here (the longest Jacobian column has 6 entries, plus the gradient and the two bound terms), each product and addition rounded
once with error <= eps/2 times the magnitudes summed, and lam = lam_s dc / dobj is two roundings from the solver's lam_s: 16
covers both with room for the scaling products dc J and dobj df.  For the lower bound, s_d_hi bounds the solver's s_d from above:
every residual and every gap * multiplier is <= tol s_d there, so a bounded component's multipliers sum to at most
|value| + tol s_d + 2 tol s_d / half span (their difference is the value up to the residual; the smaller one sits at a gap of at
least half the span), which gives s_d <= max(1, P / (K - tol Q)) with P, Q those sums and K = 100 (3m + 2n); with budget
tol s_d_hi the certificate's z interval contains every z the solver can hold, so what is left beyond it (less rounding) the solver
measured too.  After clipping the residual at x is not the one the solver measured, and only the upper check applies.

Degenerate multipliers.  Where LICQ fails -- the moment rows of a one-contact problem, whose Jacobian rows are linearly dependent
at the solution -- the multipliers are not unique and can be huge (1e9 has been seen on the `simple` problem).  s_d then grows
with them, and the unscaled residual df + J^T lam on the CoM columns can be O(10) while the scaled measure is far below tol:
that is IPOPT's convergence test doing what it is defined to do (s_d exists exactly so that large multipliers do not make the
test unreachable), not a wrong result.  The certificate judges the scaled measure for the same reason.
"""
from __future__ import annotations

from fractions import Fraction

import numpy as np

EPS = 2.0 ** -52
INF_BOUND = 1e19
ROUNDING_TERMS = 16


def _push_inside(v, lo, hi, has_lo, has_hi, k1, k2):
    span = np.where(has_lo & has_hi, hi - lo, np.inf)
    pl = np.minimum(k1 * np.maximum(np.abs(lo), 1.0), k2 * span)
    pu = np.minimum(k1 * np.maximum(np.abs(hi), 1.0), k2 * span)
    v = np.where(has_lo, np.maximum(v, lo + pl), v)
    return np.where(has_hi, np.minimum(v, hi - pu), v)


class Shape:
    """The problem-level data of a solve: bounds (original and relaxed) and the Jacobian structure."""

    def __init__(self, o, opt):
        self.n, self.m, self.nnz = o.n, o.m, o.nnz
        self.iRow, self.jCol = (np.asarray(a, dtype=np.int64) for a in o.structure())
        self.xlo, self.xhi = (np.asarray(a, dtype=np.float64) for a in o.var_bounds())
        self.cl, self.cu = (np.asarray(a, dtype=np.float64) for a in o.con_bounds())
        relax = opt.bound_relax_factor
        self.fixed = self.xlo == self.xhi
        self.xl = np.where(self.fixed, self.xlo, self.xlo - relax * np.maximum(np.abs(self.xlo), 1.0))
        self.xu = np.where(self.fixed, self.xhi, self.xhi + relax * np.maximum(np.abs(self.xhi), 1.0))
        self.x_lo = ~self.fixed & (self.xl > -INF_BOUND)
        self.x_hi = ~self.fixed & (self.xu < INF_BOUND)
        self.is_eq = self.cl == self.cu
        self.cl_r = np.where(self.is_eq, self.cl, self.cl - relax * np.maximum(np.abs(self.cl), 1.0))
        self.cu_r = np.where(self.is_eq, self.cu, self.cu + relax * np.maximum(np.abs(self.cu), 1.0))
        self.s_lo = ~self.is_eq & (self.cl > -INF_BOUND)
        self.s_hi = ~self.is_eq & (self.cu < INF_BOUND)
        self.cols = [np.nonzero(self.jCol == j)[0] for j in range(self.n)]


def scaling(o, S, opt, x0):
    """dobj and dc (m,) of one instance, from its start x0 with the solver's rule (module docstring)."""
    x = np.where(S.fixed, S.xl, x0)
    x = _push_inside(x, S.xl, S.xu, S.x_lo, S.x_hi, opt.bound_push, opt.bound_frac)
    ev = o.eval(x)
    free = ~S.fixed
    gmax = float(np.max(np.abs(ev["grad"][free]), initial=0.0))
    rowmax = np.zeros(S.m)
    slots = free[S.jCol]
    np.maximum.at(rowmax, S.iRow[slots], np.abs(ev["jac"][slots]))
    mg = opt.nlp_scaling_max_gradient
    return min(mg / max(gmax, 1e-300), 1.0), np.minimum(mg / np.maximum(rowmax, 1e-300), 1.0)


def _dist(v, lo, hi):
    """distance of v from the interval [lo, hi] (ends may be infinite)"""
    return max(lo - v, v - hi, 0.0)


def certify_instance(o, S, opt, x0, x, lam, cost, constr_viol, dual_inf):
    """Measures of one instance (see the module docstring)."""
    ev = o.eval(x)
    g, jac, f, grad = ev["g"], ev["jac"], float(ev["cost"]), ev["grad"]
    dobj, dc = scaling(o, S, opt, x0)
    lam_s = lam * dobj / dc
    sd = max(100.0, float(np.abs(lam_s).sum()) / (3 * S.m + 2 * S.n)) / 100.0
    budget = opt.tol * sd
    # entries honor_original_bounds may have clipped: free entries exactly on an original bound.  The iterate the solver measured
    # lies between that bound and the relaxed one, delta_j = bound_relax_factor * max(|bound|, 1) away at most.
    at_lo, at_hi = ~S.fixed & (x == S.xlo), ~S.fixed & (x == S.xhi)
    clipped = np.nonzero(at_lo | at_hi)[0]
    delta = np.where(at_lo, S.xlo - S.xl, 0.0) + np.where(at_hi, S.xu - S.xhi, 0.0)
    cost_slack = 0.0
    for j in clipped:   # the cost is a separable convex quadratic: |f(x + t e_j) - f(x)| <= max(|df_j| delta_j, f(x + delta_j e_j) - f(x))
        xe = x.copy()
        xe[j] = S.xl[j] if at_lo[j] else S.xu[j]
        cost_slack += max(abs(grad[j]) * delta[j], float(o.eval(xe, want=("cost",))["cost"]) - f)
    fl, fd = Fraction(dobj), [Fraction(float(v)) for v in lam]
    # (what, scaled value the bound multipliers must cancel, magnitude summed into it, gap of the side whose multiplier enters with
    # a + sign, gap of the other side, half span, bounded at all)
    items = []
    for j in range(S.n):                       # free variables: dobj (df + J^T lam) - zl + zu
        if S.fixed[j]:
            continue
        r, mag = Fraction(float(grad[j])), dobj * abs(grad[j])
        for e in S.cols[j]:
            r += Fraction(float(jac[e])) * fd[S.iRow[e]]
            mag += abs(dc[S.iRow[e]] * jac[e] * lam_s[S.iRow[e]])
        gl = (0.0 if at_lo[j] else x[j] - S.xl[j]) if S.x_lo[j] else np.inf   # clipped: the measured gap was anywhere in (0, delta_j]
        gu = (0.0 if at_hi[j] else S.xu[j] - x[j]) if S.x_hi[j] else np.inf
        items.append((f"variable {j}", float(fl * r), mag, gl, gu, 0.5 * (S.xu[j] - S.xl[j]), S.x_lo[j] or S.x_hi[j]))
    cs = dc * g
    for r in np.nonzero(~S.is_eq)[0]:          # inequality rows: lam_s = vu - vl, each v complementarity-bounded
        gl = cs[r] - dc[r] * S.cl_r[r] - opt.tol if S.s_lo[r] else np.inf
        gu = dc[r] * S.cu_r[r] - cs[r] - opt.tol if S.s_hi[r] else np.inf
        # (lam_s = vu - vl: the upper side's multiplier is the positive one, so the gaps enter the other way round)
        items.append((f"row {r} (sign / complementarity of lam)", float(lam_s[r]), abs(lam_s[r]), gu, gl,
                      0.5 * dc[r] * (S.cu_r[r] - S.cl_r[r]), True))

    def left_over(budget):
        """max over items of (what no complementary bound multiplier can cancel) - rounding; the item; max of what is left"""
        worst, excess, dual = None, -np.inf, 0.0
        for what, v, mag, gl, gu, _, _ in items:
            left = _dist(v, -budget / gu if gu > 0 else -np.inf, budget / gl if gl > 0 else np.inf)
            dual = max(dual, left)
            if left - ROUNDING_TERMS * EPS * mag > excess:
                excess, worst = left - ROUNDING_TERMS * EPS * mag, what
        return excess, worst, dual

    excess, worst, dual = left_over(budget)
    excess -= budget
    # Upper bound of the solver's s_d (its bound multipliers are not returned): at a SUCCEEDED iterate every residual is <= tol s_d
    # and every gap * multiplier <= tol s_d, so per bounded component  zl + zu <= |value| + tol s_d + 2 tol s_d / half span
    # (|zl - zu| is the value up to the residual; the smaller of the two sits at a gap >= half the span).  Summed:
    # S <= P + tol s_d Q, and s_d = max(1, S / K) <= max(1, P / (K - tol Q)), K = 100 (3m + 2n).
    P = float(np.abs(lam_s).sum()) + sum(abs(v) + ROUNDING_TERMS * EPS * mag for _, v, mag, _, _, _, bounded in items if bounded)
    Q = sum(1.0 + (2.0 / h if np.isfinite(h) else 0.0) for _, _, _, _, _, h, bounded in items if bounded)
    K = 100.0 * (3 * S.m + 2 * S.n)
    sd_hi = max(1.0, P / (K - opt.tol * Q)) if K > opt.tol * Q else np.inf
    low = max(left_over(opt.tol * sd_hi)[0], 0.0) / sd_hi   # the least scaled residual the solver can have measured
    viol_shift = np.zeros(S.m)   # first-order change of every row over the clipped entries
    np.add.at(viol_shift, S.iRow, np.abs(jac) * delta[S.jCol])
    viol_rows = np.maximum(S.cl_r - g, 0.0) + np.maximum(g - S.cu_r, 0.0)
    scale = np.maximum(np.abs(g), np.where(np.abs(S.cl_r) < INF_BOUND, np.abs(S.cl_r), 0.0))
    scale = np.maximum(scale, np.where(np.abs(S.cu_r) < INF_BOUND, np.abs(S.cu_r), 0.0))
    return dict(cost=f, viol=float(viol_rows.max(initial=0.0)), viol_slack=4 * EPS * float(scale.max(initial=0.0)), sd=sd, clipped=clipped,
                cost_slack=cost_slack + (4 * EPS * abs(f) if len(clipped) else 0.0), viol_shift=2.0 * float(viol_shift.max(initial=0.0)),
                dual=dual / sd, dual_low=low, g_scale=float(scale.max(initial=0.0)), excess=excess, worst=worst, lam_s_max=float(np.abs(lam_s).max(initial=0.0)))


def certify(oracles, opt, x0, out, which=None):
    """Certificate of the instances `which` (default: all) of a solve.  oracles: one oracle (shared parameters) or a list with
    one per instance; opt: the solver options (cplb_solver_options fields); x0: (N, n) starts; out: dict of NumPy arrays x, lam,
    status, cost, constr_viol, dual_inf.  Returns {instance: measures}."""
    one = not isinstance(oracles, (list, tuple))
    S = Shape(oracles if one else oracles[0], opt)
    which = range(len(out["status"])) if which is None else which
    return {int(i): certify_instance(oracles if one else oracles[i], S, opt, np.asarray(x0[i], dtype=np.float64), out["x"][i], out["lam"][i],
                                     float(out["cost"][i]), float(out["constr_viol"][i]), float(out["dual_inf"][i])) | {"shape": S}
            for i in which}


def assert_certified(oracles, opt, x0, out, which=None, pow_upstream=False, what=""):
    """certify, then every check of the module docstring on every instance in `which` (SUCCEEDED instances only)."""
    which = np.arange(len(out["status"])) if which is None else np.asarray(which)
    assert (np.asarray(out["status"])[which] == 0).all(), f"{what}: certify SUCCEEDED instances only"
    rep = certify(oracles, opt, x0, out, which)
    for i, c in rep.items():
        S, x = c["shape"], out["x"][i]
        tag = f"{what}: instance {i}"
        # pow() upstream: the evaluator's rows are the oracle's to 1e-12 relative, with 1 as the floor of the scale (the parity bar
        # of tests/helpers.py::assert_parity), so the violation the solver measured may differ from the oracle's by that much more
        viol_slack = c["viol_slack"] + (1e-12 * max(c["g_scale"], 1.0) if pow_upstream else 0.0)
        assert ((x >= S.xlo) & (x <= S.xhi)).all(), f"{tag}: x outside the original variable bounds"
        if len(c["clipped"]):   # cost and constr_viol are the unclipped iterate's (include/cpl_batched.h)
            assert abs(c["cost"] - out["cost"][i]) <= c["cost_slack"] + (1e-12 * abs(c["cost"]) if pow_upstream else 0.0), \
                f"{tag}: cost {out['cost'][i]!r}, oracle at the clipped x {c['cost']!r}, more than the clipping explains"
            assert abs(c["viol"] - out["constr_viol"][i]) <= c["viol_shift"] + viol_slack, \
                f"{tag}: constr_viol {out['constr_viol'][i]!r}, violation at the clipped x {c['viol']!r}"
            assert c["viol"] <= opt.constr_viol_tol, f"{tag}: SUCCEEDED with a violation {c['viol']:.3e} at the clipped x"
        else:
            if pow_upstream:
                assert abs(c["cost"] - out["cost"][i]) <= 1e-12 * abs(c["cost"]), f"{tag}: cost {out['cost'][i]!r}, oracle at x {c['cost']!r}"
            else:
                assert np.float64(c["cost"]).view(np.int64) == np.float64(out["cost"][i]).view(np.int64), \
                    f"{tag}: cost {out['cost'][i]!r} is not the oracle's cost at x, {c['cost']!r}"
            assert abs(c["viol"] - out["constr_viol"][i]) <= viol_slack, \
                f"{tag}: constr_viol {out['constr_viol'][i]!r}, violation of the relaxed bounds at x {c['viol']!r}"
            assert c["viol"] <= opt.polish_viol_tol + c["viol_slack"], f"{tag}: SUCCEEDED with a violation {c['viol']:.3e} at x"
        assert 0.0 <= out["dual_inf"][i] <= opt.tol, f"{tag}: SUCCEEDED with dual_inf {out['dual_inf'][i]!r} above tol {opt.tol:g}"
        if not len(c["clipped"]):   # (after clipping the residual at x is not the one the solver measured)
            assert out["dual_inf"][i] >= c["dual_low"], \
                f"{tag}: dual_inf {out['dual_inf'][i]:.3e} is below the least residual the certificate finds, {c['dual_low']:.3e}"
        assert c["excess"] <= 0.0, (f"{tag}: scaled stationarity residual left at {c['worst']} beyond every complementary bound "
                                    f"multiplier: {c['dual']:.3e} (x s_d = {c['sd']:.3e}) against tol {opt.tol:.1e}, dual_inf "
                                    f"{out['dual_inf'][i]:.3e}")
    return rep
