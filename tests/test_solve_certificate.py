"""The native solve round's results certified independently of the solver: CPU half, on the CPU replay.

tests/solve_certificate.py evaluates the returned x with the C oracle and checks what the solver claims about it: x inside the
original bounds, cost and constr_viol being the values at x, and IPOPT's scaled stationarity -- grad f + J^T lam formed in exact
arithmetic, judged with the solver's own scaling and s_d -- including the sign of every inequality multiplier.  The replay
(tests/native/solver_replay.cpp: csrc/cplb_solver_core.hpp on the host, the oracle behind the evaluations) is bit-identical to
the GPU solve on Ground and no-environment problems, so what is certified here holds for the GPU's results too; the GPU half is
tests/test_gpu_solve_certificate.py.  A second replay entry takes one oracle per instance, for per-instance parameter sweeps.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200.lockstep_solver import SUCCESS
from helpers import OracleEvalProblem, set_oracle_instance
from solve_certificate import assert_certified, certify
from test_solve import MASS, MASSES, NAMES, SETUPS, starts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "centroidalplanner_b200", "csrc")
ORACLE = os.path.join(ROOT, "oracle")
OUT = ("x", "lam", "status", "iterations", "cost", "constr_viol", "dual_inf")
NAMES8 = ["l_foot_a", "l_foot_b", "r_foot_a", "r_foot_b", "l_hand_a", "l_hand_b", "r_hand_a", "r_hand_b"][::-1]


def setup_ground8(problem, env):  # test_solve.py::test_native_round_on_an_eight_contact_problem
    env.SetGroundZ(0.1)
    env.SetMu(0.5)
    problem.SetCoMWeight(2.0)
    problem.SetForceWeight(0.0)
    for nm in NAMES8:
        problem.SetPosBounds(nm, [-0.3, -0.3, 0.0], [0.3, 0.3, 1.0])
    problem.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])


def setup_none(problem, env):
    """No environment, contact positions free inside a box and below the CoM, normals fixed upwards: the no-environment problem of
    the per-instance sweeps (positions, hence pos_ref, take part; com_planner's are fixed)."""
    problem.SetMu(0.5)
    problem.SetCoMWeight(2.0)
    for nm in NAMES:
        problem.SetNormalBounds(nm, [0, 0, 1.0], [0, 0, 1.0])
        problem.SetPosBounds(nm, [-0.3, -0.3, 0.0], [0.3, 0.3, 0.2])
    problem.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])


CASES = dict(SETUPS)
CASES["ground8"] = (NAMES8, "ground", setup_ground8)    # a 129 x 129 KKT matrix
CASES["none"] = (NAMES, "none", setup_none)
REPLAYED = ["simple", "ground", "com_planner", "example_planner", "example_com_planner", "ground8"]   # no pow() upstream


def oracle_side(case, force_weight=None):
    names, env_name, setup = CASES[case]
    op = OracleEvalProblem(names, env_name, MASSES.get(case, MASS))
    setup(op, op)
    if force_weight is not None:
        op.SetForceWeight(force_weight)
    return op


def product_side(case, force_weight=None):
    names, env_name, setup = CASES[case]
    env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, MASSES.get(case, MASS), env)
    setup(prob, env)
    if force_weight is not None:
        prob.SetForceWeight(force_weight)
    return prob


def sweep(case, N, seed, cost_only=False):
    """Per-instance parameters for every field of cplb_instance_params (or only the six cost fields), different per instance and
    large enough to move the optimum: CoM reference within +-0.05 of (0, 0, 0.9), contact position references spread over and
    beyond the position box (active bounds), force references around the weight share, every weight > 0."""
    nc = len(CASES[case][0])
    rng = np.random.default_rng(seed)
    p = dict(com_ref=np.array([0.0, 0.0, 0.9]) + rng.uniform(-0.05, 0.05, (N, 3)), com_weight=rng.uniform(1.0, 3.0, N),
             pos_ref=np.stack([rng.uniform(-0.4, 0.4, (N, nc)), rng.uniform(-0.4, 0.4, (N, nc)), rng.uniform(0.0, 0.2, (N, nc))], axis=2),
             force_ref=np.stack([rng.uniform(-30.0, 30.0, (N, nc)), rng.uniform(-30.0, 30.0, (N, nc)), rng.uniform(150.0, 350.0, (N, nc))], axis=2),
             pos_weight=rng.uniform(0.5, 2.0, (N, nc)), force_weight=rng.uniform(1e-4, 1e-2, (N, nc)))
    if not cost_only:
        p.update(mass=rng.uniform(80.0, 120.0, N), mu=rng.uniform(0.45, 0.8, N), force_threshold=rng.uniform(5.0, 30.0, (N, nc)),
                 wrench=np.array([100.0, 0, 0, 0, 0, 100.0]) + rng.normal(0.0, 10.0, (N, 6)) * np.array([1, 1, 1, 0.2, 0.2, 1.0]),
                 ground_z=rng.uniform(0.05, 0.15, N))
    return {k: np.ascontiguousarray(v.reshape(N, -1) if v.ndim > 2 else v) for k, v in p.items()}


def instance_oracles(case, per_instance):
    """One oracle per instance, each playing its instance's CplProblem."""
    N = len(next(iter(per_instance.values())))
    ops = []
    for i in range(N):
        op = oracle_side(case)
        set_oracle_instance(op.o, per_instance, i)
        ops.append(op)
    return ops


def _cxx():
    return shutil.which("g++") or "g++"


@pytest.fixture(scope="module")
def replay_lib(tmp_path_factory):
    """solver_replay.cpp as a shared library linked against the oracle library the ctypes wrapper loads."""
    subprocess.check_call(["make", "-C", ORACLE, "libcpl_oracle.so"], stdout=subprocess.DEVNULL)
    so = str(tmp_path_factory.mktemp("replay") / "libsolver_replay.so")
    subprocess.check_call([_cxx(), "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", ORACLE, "-I", os.path.join(ROOT, "include"),
                           "-I", CSRC, os.path.join(NATIVE, "solver_replay.cpp"), "-o", so, "-L", ORACLE, "-lcpl_oracle",
                           f"-Wl,-rpath,{ORACLE}", "-lpthread"])
    lib = C.CDLL(so)
    for f in (lib.cplb_replay_solve, lib.cplb_replay_solve_per_instance):
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p] + [C.c_void_p] * 8 + [C.c_int]
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def replay(lib, oracles, x0, solver):
    """The CPU replay of `solver` (a NativeInteriorPoint: its options) from the starts x0: on one oracle problem, or with a list
    of oracle problems one per instance (cplb_replay_solve_per_instance)."""
    x0 = np.ascontiguousarray(np.asarray(x0.cpu() if hasattr(x0, "cpu") else x0, dtype=np.float64))
    N = x0.shape[0]
    one = not isinstance(oracles, (list, tuple))
    op = oracles if one else oracles[0]
    out = dict(x=np.empty((N, op.n)), lam=np.empty((N, op.m)), status=np.empty(N, np.int32), iterations=np.empty(N, np.int32),
               cost=np.empty(N), constr_viol=np.empty(N), dual_inf=np.empty(N))
    stats = np.zeros(4, np.int64)
    if one:
        fn, handle = lib.cplb_replay_solve, C.c_void_p(op.o._h)
    else:
        handles = (C.c_void_p * N)(*[p.o._h for p in oracles])
        fn, handle = lib.cplb_replay_solve_per_instance, C.cast(handles, C.c_void_p)
    rc = fn(handle, N, _ptr(x0), C.cast(C.byref(solver.options), C.c_void_p), *[_ptr(out[k]) for k in OUT], _ptr(stats), os.cpu_count() or 1)
    assert rc == 0
    out["status"] = out["status"].astype(np.int64)
    out["iterations"] = out["iterations"].astype(np.int64)
    out.update(rounds=int(stats[0]), evaluations=int(stats[1]), instance_evaluations=int(stats[2]), tail_instances=int(stats[3]))
    return out


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype.kind != "f":
        return bool(np.array_equal(a, b))
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all() and (a.view(np.int64)[~na] == b.view(np.int64)[~nb]).all())


def oracles_of(ops):
    return [p.o for p in ops] if isinstance(ops, (list, tuple)) else ops.o


# ---- the certificate on the replay ---------------------------------------------------------------------------------------------
# At tol 1e-8 the set-ups with a zero force weight and several contacts on the ground or at fixed positions (ground, ground8,
# com_planner, example_com_planner) have a continuum of minimisers along which the scaled error does not fall to 1e-8 within
# max_iter from every start (the line search has no restoration phase): 0, 0, 21 and 61 of 64 starts succeed.  There the 1e-8
# sweep adds the force weight that makes the minimiser unique (as test_solve.py's driver comparisons do), so that every start
# succeeds and is certified; simple and example_planner are certified at 1e-8 as they are.
NEEDS_FORCE_WEIGHT_AT_1E8 = {"ground", "ground8", "com_planner", "example_com_planner"}


@pytest.mark.parametrize("tol", [1e-3, 1e-8])
@pytest.mark.parametrize("case", REPLAYED)
def test_replayed_solutions_are_certified_kkt_points(case, tol, replay_lib):
    op = oracle_side(case, force_weight=1e-4 if tol < 1e-3 and case in NEEDS_FORCE_WEIGHT_AT_1E8 else None)
    N = 64
    x0 = starts(op, N, seed=7)
    s = cpl.NativeInteriorPoint(tol=tol, tail_instances=0)
    r = replay(replay_lib, op, x0, s)
    assert (r["status"] == SUCCESS).all(), (r["status"].tolist(), r["iterations"].tolist())
    assert_certified(op.o, s.options, x0.numpy(), r, what=f"{case}, tol {tol:g}")


def test_degenerate_multipliers_pass_the_scaled_measure_only(replay_lib):
    """One contact: the six statics rows in x, F and p are linearly dependent at the solution (LICQ fails), the moment-row
    multipliers are not unique and come out near 1e9.  The unscaled residual grad f + J^T lam on the CoM columns is then O(10) --
    but s_d, which exists so that large multipliers do not make the test unreachable, is ~1e4, and the scaled residual is below
    tol.  That is IPOPT's convergence test as defined, not a wrong result: the certificate must pass it."""
    op = oracle_side("simple")
    x0 = starts(op, 16, seed=7)
    s = cpl.NativeInteriorPoint(tail_instances=0)
    r = replay(replay_lib, op, x0, s)
    rep = assert_certified(op.o, s.options, x0.numpy(), r, what="simple")
    assert max(c["lam_s_max"] for c in rep.values()) > 1e6 and max(c["sd"] for c in rep.values()) > 100.0


def test_certificate_rejects_wrong_multipliers_and_values(replay_lib):
    """The checker itself: the replay's results with a negated lam, lam without its row scaling dc, lam scaled by 1.01, the cost of
    a neighbouring point, a constr_viol that is off, a dual_inf above tol (which must not lift the bar: lam x 1.5 with dual_inf 1e6
    is refused too) or a dual_inf below the residual the certificate finds are each refused."""
    op = oracle_side("ground")
    x0 = starts(op, 8, seed=7)
    s = cpl.NativeInteriorPoint(tail_instances=0)
    r = replay(replay_lib, op, x0, s)
    assert_certified(op.o, s.options, x0.numpy(), r)
    from solve_certificate import Shape, scaling
    S = Shape(op.o, s.options)
    dc = np.array([scaling(op.o, S, s.options, x0[i].numpy())[1] for i in range(8)])
    assert (dc < 1.0).any()
    bad = {"negated lam": dict(r, lam=-r["lam"]), "lam without dc": dict(r, lam=r["lam"] / dc), "lam x 1.01": dict(r, lam=r["lam"] * 1.01),
           "cost of another point": dict(r, cost=np.nextafter(r["cost"], np.inf)),
           "constr_viol off": dict(r, constr_viol=r["constr_viol"] + 1e-6),
           "lam x 1.5 with dual_inf 1e6": dict(r, lam=r["lam"] * 1.5, dual_inf=np.full_like(r["dual_inf"], 1e6)),
           "dual_inf above tol": dict(r, dual_inf=r["dual_inf"] + s.options.tol), "dual_inf zero": dict(r, dual_inf=0.0 * r["dual_inf"])}
    for what, out in bad.items():
        with pytest.raises(AssertionError):
            assert_certified(op.o, s.options, x0.numpy(), out, what=what)


def test_replay_agrees_with_scipy_slsqp_on_a_nondegenerate_problem(replay_lib):
    """With a force weight the minimiser is unique: the replay of the native round (tol 1e-8) and SciPy's SLSQP on the same oracle
    callbacks, from the same starts, must find the same optimal cost and the same x.  The cost is stationary at the minimiser, so
    it agrees to about the square of the distance between the two points: 1e-8 relative.  x agrees to 1e-3: both stopping rules
    allow a residual of ~1e-8 in a problem whose weakest curvature is the force weight 1e-4 against forces of O(100)."""
    from scipy.optimize import minimize

    op = oracle_side("ground", force_weight=1e-4)
    x0 = starts(op, 4, seed=7)
    s = cpl.NativeInteriorPoint(tol=1e-8, tail_instances=0)
    r = replay(replay_lib, op, x0, s)
    assert (r["status"] == SUCCESS).all()
    assert_certified(op.o, s.options, x0.numpy(), r, what="ground, force weight 1e-4")
    iRow, jCol = op.GetJacobianStructure()
    lb, ub = op.GetBoundsOnOptimizationVariables()
    cl, cu = op.GetBoundsOnConstraints()
    eq = cl == cu

    def dense(x):
        J = np.zeros((op.m, op.n))
        J[iRow, jCol] = op.o.eval(x)["jac"]
        return J

    cons = [{"type": "eq", "fun": lambda x: op.o.eval(x)["g"][eq] - cl[eq], "jac": lambda x: dense(x)[eq]},
            {"type": "ineq", "fun": lambda x: cu[~eq] - op.o.eval(x)["g"][~eq], "jac": lambda x: -dense(x)[~eq]}]
    for i in range(len(x0)):
        q = minimize(lambda x: op.o.eval(x)["cost"], x0[i].numpy(), jac=lambda x: op.o.eval(x)["grad"], bounds=list(zip(lb, ub)),
                     constraints=cons, method="SLSQP", options={"maxiter": 500, "ftol": 1e-12})
        assert q.status == 0, q.message
        assert abs(r["cost"][i] - q.fun) <= 1e-8 * abs(q.fun), (i, r["cost"][i], q.fun)
        assert np.abs(r["x"][i] - q.x).max() <= 1e-3, (i, np.abs(r["x"][i] - q.x).max())


# ---- the per-instance replay ---------------------------------------------------------------------------------------------------
def test_per_instance_replay_with_shared_values_is_the_shared_replay(replay_lib):
    """One oracle per instance, all with the shared parameters: the same bits as the single-oracle replay, in the lock-step rounds
    and in the tail."""
    op = oracle_side("ground")
    x0 = starts(op, 24, seed=5)
    ops = [oracle_side("ground") for _ in range(24)]
    for tail in (0, 10):
        s = cpl.NativeInteriorPoint(tail_instances=tail)
        a, b = replay(replay_lib, op, x0, s), replay(replay_lib, ops, x0, s)
        for k in OUT:
            assert same_bits(a[k], b[k]), (tail, k)


@pytest.mark.parametrize("cost_only", [False, True], ids=["all_fields", "cost_fields"])
@pytest.mark.parametrize("case", ["ground", "none"])
def test_per_instance_replay_is_certified(case, cost_only, replay_lib):
    """A sweep in which every instance is its own planning problem, replayed with one oracle per instance: every instance is a KKT
    point of ITS problem (certified with its own oracle), and not of the shared one; the tail gives the same bits."""
    N = 48
    per = sweep(case, N, seed=11, cost_only=cost_only)
    ops = instance_oracles(case, per)
    x0 = starts(ops[0], N, seed=3)
    s = cpl.NativeInteriorPoint(tail_instances=0)
    r = replay(replay_lib, ops, x0, s)
    assert (r["status"] == SUCCESS).all(), (r["status"].tolist(), r["iterations"].tolist())
    assert_certified(oracles_of(ops), s.options, x0.numpy(), r, what=f"{case} sweep")
    t = replay(replay_lib, ops, x0, cpl.NativeInteriorPoint(tail_instances=20))
    for k in OUT:
        assert same_bits(t[k], r[k]), k
    # the parameters moved the optimum: judged with the shared problem's oracle, the cost at x is not the reported one
    shared = certify(oracle_side(case).o, s.options, x0.numpy(), r)
    assert sum(c["cost"] != r["cost"][i] for i, c in shared.items()) >= N // 2
