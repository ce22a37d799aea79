"""Shared test plumbing: the named configurations, product/oracle pairs with identical parameters,
and the parity comparison (bit-exact where no pow() is upstream, <= 1e-12 relative elsewhere)."""
from __future__ import annotations

import os

import numpy as np

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic
from oracle import cpl_oracle_py as orc

RTOL = 1e-12  # north_star: "within 1e-12 relative (fp64)"

NAMES_PERMUTED = ["r_foot", "l_foot", "r_hand", "l_hand"]  # vector order != sorted order (SURVEY H3)

CASES = {
    # name: (contact names, env kind, batch generator)
    "ground4": (synthetic.NAMES4, "ground", lambda N: synthetic.ground_batch(N, 4, 1002)),
    "superquadric4": (synthetic.NAMES4, "superquadric", lambda N: synthetic.superquadric_batch(N, 4, 1003)),
    "ground8": (synthetic.NAMES8, "ground", lambda N: synthetic.ground_batch(N, 8, 1004)),
    "noenv4": (NAMES_PERMUTED, "none", lambda N: synthetic.ground_batch(N, 4, 77)),
    "ground1": (["contact1"], "ground", lambda N: synthetic.ground_batch(N, 1, 5)),
    "superquadric3": (["c", "a", "b"], "superquadric", lambda N: synthetic.superquadric_batch(N, 3, 9)),
    "ground5": (["e", "d", "c", "b", "a"], "ground", lambda N: synthetic.ground_batch(N, 5, 11)),
    "noenv2": (["right", "left"], "none", lambda N: synthetic.ground_batch(N, 2, 12)),
    "noenv8": (synthetic.NAMES8, "none", lambda N: synthetic.ground_batch(N, 8, 13)),
    "superquadric8": (synthetic.NAMES8, "superquadric", lambda N: synthetic.superquadric_batch(N, 8, 15)),
    "ground12": (["k%02d" % (11 - i) for i in range(12)], "ground", lambda N: synthetic.ground_batch(N, 12, 17)),
    # CPLB_MAX_CONTACTS: 32 warps per CTA in the component-major kernel, one warp per CTA in the instance-major one
    "superquadric32": (["k%02d" % ((7 * i) % 32) for i in range(32)], "superquadric", lambda N: synthetic.superquadric_batch(N, 32, 19)),
    # fractional curvatures: every pow() of the reference is a real pow() on the GPU too (no integer fast path);
    # contacts on the positive side of the centre only (pow(negative, fractional) is NaN -- also covered, see below)
    "superquadric4_fracP": (synthetic.NAMES4, "superquadric", lambda N: _positive_side(synthetic.superquadric_batch(N, 4, 23)),
                            {"sq": dict(C=[0.0, 0.0, 1.0], R=[0.3, 0.35, 2.0], P=[2.5, 3.75, 10.0])}),
    "superquadric4_fracP_nan": (synthetic.NAMES4, "superquadric", lambda N: synthetic.superquadric_batch(N, 4, 29),
                                {"sq": dict(C=[0.0, 0.0, 1.0], R=[0.3, 0.35, 2.0], P=[2.5, 4.0, 3.0])}),
    "superquadric4_P2": (synthetic.NAMES4, "superquadric", lambda N: synthetic.superquadric_batch(N, 4, 31),
                         {"sq": dict(C=[0.1, -0.1, 0.9], R=[0.5, 0.4, 0.6], P=[2.0, 4.0, 7.0])}),
    "superquadric4_P63": (synthetic.NAMES4, "superquadric", lambda N: synthetic.superquadric_batch(N, 4, 37),
                          {"sq": dict(C=[0.0, 0.0, 1.0], R=[0.3, 0.3, 0.4], P=[63.0, 40.0, 17.0])}),
}


def _positive_side(x):
    """Mirror every contact position to p >= C (C = (0,0,1)) so that fractional powers stay real."""
    x = x.copy()
    nc = (x.shape[1] - 3) // 9
    C = np.array([0.0, 0.0, 1.0])
    for k in range(nc):
        sl = slice(3 + 9 * k + 3, 3 + 9 * k + 6)
        x[:, sl] = C + np.abs(x[:, sl] - C)
    return x


class OracleProblem:
    """Gives the oracle the same setter names as BatchedCplProblem so one routine configures both."""

    def __init__(self, names, env_name, mass):
        kind = {"none": orc.ENV_NONE, "ground": orc.ENV_GROUND, "superquadric": orc.ENV_SUPERQUADRIC}[env_name]
        self.o = orc.Oracle(names, kind, mass)
        self.names = list(names)

    def SetGroundZ(self, z): self.o.set_ground_z(z)
    def SetParameters(self, C, R, P): self.o.set_superquadric(C, R, P)
    def SetMu(self, mu): self.o.set_mu(mu)
    def SetManipulationWrench(self, w): self.o.set_wrench(w)
    def SetForceThreshold(self, nm, t): self.o.set_force_threshold(nm, t)
    def SetCoMRef(self, r): self.o.set_com_ref(r)
    def SetCoMWeight(self, w): self.o.set_com_weight(w)
    def SetPosRef(self, nm, r): self.o.set_pos_ref(nm, r)
    def SetForceRef(self, nm, r): self.o.set_force_ref(nm, r)
    def SetPosWeight(self, w): self.o.set_pos_weight(w)
    def SetForceWeight(self, w): self.o.set_force_weight(w)
    def SetContactPosWeight(self, nm, w): self.o.set_contact_pos_weight(nm, w)
    def SetContactForceWeight(self, nm, w): self.o.set_contact_force_weight(nm, w)
    def SetPosBounds(self, nm, lb, ub): self.o.set_var_bounds(orc.BLOCK_P, nm, lb, ub)
    def SetForceBounds(self, nm, lb, ub): self.o.set_var_bounds(orc.BLOCK_F, nm, lb, ub)
    def SetNormalBounds(self, nm, lb, ub): self.o.set_var_bounds(orc.BLOCK_N, nm, lb, ub)


def configure(problem, env, names, env_name, rich=True, extra=None):
    """Same non-default parameters on either side.  `env` is the cpl.Ground/Superquadric object for the
    product, or the OracleProblem itself for the oracle."""
    if env_name == "ground":
        env.SetGroundZ(synthetic.TESTBASIC["ground_z"])
    elif env_name == "superquadric":
        sq = (extra or {}).get("sq", synthetic.SUPERQUADRIC)
        env.SetParameters(sq["C"], sq["R"], sq["P"])
    (env if env is not None else problem).SetMu(0.5)
    problem.SetManipulationWrench(synthetic.TESTBASIC["wrench"])
    problem.SetCoMWeight(2.0)
    if rich:  # exercise every per-contact parameter with distinct values
        problem.SetCoMRef([0.05, -0.02, 0.9])
        for k, nm in enumerate(names):
            problem.SetForceThreshold(nm, 10.0 + 3.0 * k)
            problem.SetPosRef(nm, [0.1 * k, -0.05 * k, 0.02 * k])
            problem.SetForceRef(nm, [1.0 + k, 2.0 - k, 100.0 + 10.0 * k])
            problem.SetContactPosWeight(nm, 0.5 + 0.25 * k)
            problem.SetContactForceWeight(nm, 0.001 * (k + 1))


def set_oracle_instance(o, per_instance, i):
    """Give oracle `o` the parameters of instance i of a per-instance dict (keys: _cabi.INSTANCE_PARAMS names, instance-major
    NumPy arrays): the oracle then plays that instance's CplProblem."""
    shared = {"mass": o.set_mass, "wrench": o.set_wrench, "mu": o.set_mu, "ground_z": o.set_ground_z, "com_ref": o.set_com_ref,
              "com_weight": o.set_com_weight}
    per_contact = {"force_threshold": o.set_force_threshold, "pos_ref": o.set_pos_ref, "force_ref": o.set_force_ref,
                   "pos_weight": o.set_contact_pos_weight, "force_weight": o.set_contact_force_weight}
    stride = {name: per for name, _, per in _cabi.INSTANCE_PARAMS}
    for name, arr in per_instance.items():
        row = arr[i]
        if name in shared:
            shared[name](row)
        elif name in per_contact:
            s = stride[name]
            for k, nm in enumerate(o.names):
                per_contact[name](nm, row[k] if s == 1 else row[s * k:s * k + s])
        else:
            raise ValueError(f"set_oracle_instance does not handle per-instance parameter '{name}'")


def make_pair(case, mass=100.0, rich=True):
    names, env_name, gen = CASES[case][:3]
    extra = CASES[case][3] if len(CASES[case]) > 3 else None
    env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, mass, env)
    if os.environ.get("CPLB_TEST_IM_KERNEL"):  # development aid: run the whole suite with one instance-major kernel forced
        prob.SetInstanceMajorKernel(os.environ["CPLB_TEST_IM_KERNEL"])
    configure(prob, env, names, env_name, rich, extra)
    op = OracleProblem(names, env_name, mass)
    configure(op, op if env_name != "none" else None, names, env_name, rich, extra)
    return prob, op.o, gen


def pow_downstream_masks(o):
    """Boolean masks (over g rows / jac slots) of the outputs that have a pow() upstream: only the
    EnvironmentConstraint / EnvironmentNormal rows of a Superquadric problem."""
    gm = np.zeros(o.m, dtype=bool)
    jm = np.zeros(o.nnz, dtype=bool)
    if o.env_kind == orc.ENV_SUPERQUADRIC:
        iRow, jCol = o.structure()
        for j in range(o.nc):
            rows = 6 + 6 * j + np.arange(4)
            gm[rows] = True
            jm |= np.isin(iRow, rows)
        # the identity entries of EnvironmentNormal's n-block are constants
        perm = o.sorted_order()
        for j in range(o.nc):
            ncol = 3 + 9 * int(perm[j]) + 6
            jm &= ~(np.isin(iRow, 6 + 6 * j + 1 + np.arange(3)) & (jCol >= ncol) & (jCol < ncol + 3))
    return gm, jm


Q5_FACTOR = 32  # multiple of eps * amplification * |exact entry| granted to the three diagonal normal-Jacobian entries (see below)
ALLOWANCE = {"entries": 0, "pow_entries": 0, "worst_vs_plain_bar": 0.0}  # running tally over every assert_parity call of the session


def expanded_square_bound(o, x):
    """SURVEY Q5: the diagonal entries of the superquadric normal Jacobian end in
    Q = C_u^2 W_u + C_v^2 W_v + p_u^2 W_u + p_v^2 W_v - 2 C_u p_u W_u - 2 C_v p_v W_v  (= (p_u-C_u)^2 W_u + (p_v-C_v)^2 W_v),
    summed term by term in fp64 (Superquadric.cpp:99-100,153-154,207-208).  The reference's own value therefore
    carries an ABSOLUTE rounding error of a few eps * sum|terms| * |everything Q is multiplied by|
    = eps * amp * |exact entry|, amp = sum|terms| / |Q|; near p = C (amp >> 1) it is mostly noise and no evaluation
    can agree with it to better than that.  Returns (N, nnz) absolute bounds 64 * eps * amp * |exact entry| for those
    three entries per contact (exact entry from the closed form h_a (g_u^2 + g_v^2) / |g|^3) and 0 elsewhere."""
    N = x.shape[0]
    bound = np.zeros((N, o.nnz))
    if o.env_kind != orc.ENV_SUPERQUADRIC:
        return bound
    C, R, P = o.sq
    iRow, jCol = o.structure()
    perm = o.sorted_order()
    with np.errstate(all="ignore"):
        for j in range(o.nc):
            k = int(perm[j])
            p = x[:, 3 + 9 * k + 3:3 + 9 * k + 6]
            d = p - C
            ad = np.abs(d)
            g = (P / R ** P) * ad ** (P - 1)
            h = (P / R ** P) * (P - 1) * ad ** (P - 2)
            s = (g ** 2).sum(axis=1)
            for a in range(3):
                u, v = (1 if a == 0 else 0), (1 if a == 2 else 2)
                Wu = P[v] ** 2 * ad[:, v] ** (2 * P[v]) * R[u] ** (2 * P[u])
                Wv = P[u] ** 2 * ad[:, u] ** (2 * P[u]) * R[v] ** (2 * P[v])
                num = (np.abs(C[u]) + np.abs(p[:, u])) ** 2 * Wu + (np.abs(C[v]) + np.abs(p[:, v])) ** 2 * Wv
                den = d[:, u] ** 2 * Wu + d[:, v] ** 2 * Wv
                exact = h[:, a] * (g[:, u] ** 2 + g[:, v] ** 2) / (s * np.sqrt(s))
                slot = np.nonzero((iRow == 6 + 6 * j + 1 + a) & (jCol == 3 + 9 * k + 3 + a))[0]
                assert slot.size == 1
                bnd = Q5_FACTOR * 1.12e-16 * (num / den) * exact
                bound[:, slot[0]] = np.where(np.isfinite(bnd), bnd, 0.0)
    return bound


def same_bits(a, b):
    """Bit-identical, with NaNs matched by position (payload bits ignored)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    if not (na == nb).all():
        return False
    return bool((a.view(np.int64)[~na] == b.view(np.int64)[~nb]).all())


def assert_parity(got, want, o, what, x=None, allowance=True):
    """got/want: dicts with instance-major arrays g (N,m), jac (N,nnz), cost (N,), grad (N,n).  Returns the number of entries
    that passed only through the expanded-square allowance (SURVEY Q5; 0 when x is None or allowance=False: plain 1e-12 bar)."""
    gm, jm = pow_downstream_masks(o)
    used = 0
    for key in ("g", "jac", "cost", "grad"):
        if want.get(key) is None or got.get(key) is None:
            continue
        a, b = np.asarray(got[key]), np.asarray(want[key])
        assert a.shape == b.shape, (what, key, a.shape, b.shape)
        mask = {"g": gm, "jac": jm}.get(key)
        if mask is None or not mask.any():
            assert same_bits(a, b), f"{what}: {key} is not bit-identical to the oracle"
            continue
        assert same_bits(a[:, ~mask], b[:, ~mask]), f"{what}: pow-free part of {key} is not bit-identical"
        aa, bb = a[:, mask], b[:, mask]
        assert (np.isnan(aa) == np.isnan(bb)).all(), f"{what}: NaN positions differ in {key}"
        assert (np.isinf(aa) == np.isinf(bb)).all() and (aa[np.isinf(aa)] == bb[np.isinf(bb)]).all()
        fin = np.isfinite(bb)
        scale = np.abs(bb)
        if key == "g":
            # EnvironmentConstraint value is a sum of O(>=1) terms minus 1; the normal rows are n - n_env with
            # |n_env| <= 1: relative-to-result is meaningless under cancellation, so the floor is the term scale
            scale = np.maximum(scale, 1.0)
        scale = np.where(scale > 0.0, scale, 1.0)  # an exact 0.0 in the oracle: absolute 1e-12
        # the bar is 1e-12 relative; where the reference's own expanded-square sum cancels the bar is the reference's
        # own rounding noise there (expanded_square_bound) -- the best any evaluation that is not bit-identical can do
        err = np.abs(aa - bb)
        tol = RTOL * scale
        plain = (err / tol)[fin]
        ALLOWANCE["pow_entries"] += int(plain.size)
        if plain.size:
            ALLOWANCE["worst_vs_plain_bar"] = max(ALLOWANCE["worst_vs_plain_bar"], float(plain.max()))
        if key == "jac" and x is not None and allowance:
            tol = np.maximum(tol, expanded_square_bound(o, x)[:, mask])
            n_used = int((plain > 1.0).sum())   # entries beyond the plain bar: they pass, if at all, through the allowance
            used += n_used
            ALLOWANCE["entries"] += n_used
        ratio = (err / tol)[fin]
        worst = float(ratio.max()) if ratio.size else 0.0
        err = err / scale
        assert worst <= 1.0, (f"{what}: {key} differs from the oracle by {float(err[fin].max()):.3e} relative "
                              f"({worst:.2f}x the tolerance)")
    return used


def to_instance_major(arr, layout):
    a = np.asarray(arr)
    return a.T if (layout == cpl.COMPONENT_MAJOR and a.ndim == 2) else a


class OracleEvalProblem(OracleProblem):
    """The oracle behind the evaluation surface a solver drives (`n, m, nnz, eval, GetJacobianStructure,
    GetBoundsOn*`): lets the lock-step solve driver run the identical loop on the CPU reference restatement."""

    def __init__(self, names, env_name, mass, nthreads=1):
        super().__init__(names, env_name, mass)
        self.n, self.m, self.nnz = self.o.n, self.o.m, self.o.nnz
        self.nthreads = nthreads
        self.calls = 0

    def GetJacobianStructure(self):
        return self.o.structure()

    def GetBoundsOnOptimizationVariables(self):
        return self.o.var_bounds()

    def GetBoundsOnConstraints(self):
        return self.o.con_bounds()

    def eval(self, x, g=True, jac=True, cost=False, grad=False):
        import torch

        want = tuple(k for k, w in (("g", g), ("jac", jac), ("cost", cost), ("grad", grad)) if w)
        self.calls += 1
        out = self.o.eval_batch(x.detach().cpu().numpy(), want=want, nthreads=self.nthreads)
        return {k: (None if out[k] is None else torch.as_tensor(out[k])) for k in ("g", "jac", "cost", "grad")}
