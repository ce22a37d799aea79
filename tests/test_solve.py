"""The reference's own test suite (tests/TestBasic.cpp) replayed through the lock-step solve driver.

The reference's four tests build a planner, call Solve() (IPOPT) and assert post-solve invariants.  IPOPT is absent from
this image; `centroidalplanner_b200.lockstep_solver.LockStepInteriorPoint` is the stand-in (the same interior-point
scheme, batched over instances, every callback round one batched evaluation).  Each test below is one TEST_F with its
parameters and its EXPECT lines, asserted for EVERY instance of a small batch of different starting points:

  * CPU (`not gpu`): the evaluator behind the driver is the oracle -- pins the driver and the assertions themselves;
  * GPU (`-m gpu`): the evaluator is the CUDA path through the C ABI, x never leaves the device.  For Ground and
    no-environment problems every output of the CUDA path is bit-identical to the oracle's, so with the linear algebra on
    the same device the two solves must walk the SAME iterates bit for bit (`test_gpu_solve_trajectory_is_the_oracle_s`).

The two scenarios of the reference's Python example (examples/python/test.py: a two-contact planner with every default, a
CoMPlanner with two lifting contacts and a CoM reference) run through the same machinery; the example asserts nothing, so
they are held to TestBasic's equilibrium and friction lines.

Where the reference asserts a strict `<= 0.0` on a quantity an interior-point method only drives to its bound within the
bound relaxation (IPOPT bound_relax_factor = 1e-8), the tolerance is written out.
"""
import numpy as np
import pytest
import torch

import centroidalplanner_b200 as cpl
from centroidalplanner_b200.lockstep_solver import SUCCESS, LockStepInteriorPoint, default_start
from helpers import OracleEvalProblem

G = -9.81
MASS = 100.0
NAMES = ["contact1", "contact2", "contact3", "contact4"]
MASSES = {"example_planner": 20.0}
RELAX = 1e-8  # IPOPT bound_relax_factor


def starts(problem, N, seed, device=None):
    """Instance 0 starts at default_start, the others at perturbations of it."""
    x0 = default_start(problem, N)
    rng = np.random.default_rng(seed)
    x0[1:] += torch.as_tensor(rng.normal(0.0, 0.05, tuple(x0[1:].shape)))
    return x0 if device is None else x0.to(device)


# ---- the four TEST_F setups, applied to anything with the CplProblem setter names --------------------------------
def setup_simple(problem, env):                     # TestBasic.cpp:27-61
    env.SetGroundZ(0.1)
    return dict(ground_z=0.1)


def setup_ground(problem, env):                     # TestBasic.cpp:64-136
    env.SetGroundZ(0.1)
    env.SetMu(0.5)
    problem.SetCoMWeight(2.0)
    problem.SetForceWeight(0.0)
    for nm in NAMES:
        problem.SetPosBounds(nm, [-0.3, -0.3, 0.0], [0.3, 0.3, 1.0])
    problem.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])
    return dict(ground_z=0.1, mu=0.5, wrench=np.array([100.0, 0, 0, 0, 0, 100.0]))


def setup_superquadric(problem, env):               # TestBasic.cpp:139-222
    env.SetMu(0.5)
    env.SetParameters([0.0, 0.0, 1.0], [0.3, 0.3, 10.0], [10.0, 10.0, 10.0])
    problem.SetForceWeight(0.0)
    for nm in NAMES:
        problem.SetPosBounds(nm, [-0.5, -0.5, 0.5], [0.5, 0.5, 1.5])
    problem.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])
    return dict(mu=0.5, wrench=np.array([100.0, 0, 0, 0, 0, 100.0]), C=np.array([0, 0, 1.0]), R=np.array([0.3, 0.3, 10.0]),
                P=np.array([10.0, 10, 10]), p_lb=np.array([-0.5, -0.5, 0.5]), p_ub=np.array([0.5, 0.5, 1.5]))


def setup_com_planner(problem, env):                # TestBasic.cpp:225-292 with the CoMPlanner bookkeeping (src/CoMPlanner.cpp)
    problem.SetPosWeight(0.0)                       # CoMPlanner.cpp:10-11
    problem.SetForceWeight(0.0)
    problem.SetMu(0.5)
    pts = {"contact1": [1.0, 1.0, 0.0], "contact2": [-1.0, 1.0, 0.0], "contact3": [-1.0, -1.0, 0.0], "contact4": [1.0, -1.0, 0.0]}
    for nm in NAMES:
        problem.SetNormalBounds(nm, [0, 0, 1.0], [0, 0, 1.0])   # SetContactNormal
        problem.SetPosBounds(nm, pts[nm], pts[nm])               # SetContactPosition
    problem.SetForceBounds("contact4", [0, 0, 0], [0, 0, 0])     # SetLiftingContact: zero force, threshold 0
    problem.SetForceThreshold("contact4", 0.0)
    for nm in NAMES[:3]:
        problem.SetForceThreshold(nm, 20.0)                     # CentroidalPlanner.cpp:340: not forwarded to contact4
    return dict(mu=0.5, wrench=np.zeros(6))


def setup_example_planner(problem, env):           # examples/python/test.py:7-18: two contacts, mass 20, everything else default
    env.SetGroundZ(0.1)
    return dict(ground_z=0.1, mu=0.5, wrench=np.zeros(6), mass=20.0)   # mu default: Environment.h:46


def setup_example_com_planner(problem, env):       # examples/python/test.py:21-42: two of four contacts lifting, CoM reference set
    problem.SetPosWeight(0.0)
    problem.SetForceWeight(0.0)
    problem.SetMu(0.5)
    problem.SetCoMRef([0.2, 0.2, 1.0])
    pts = {"c_1": [1.0, 1.0, 0.0], "c_2": [-1.0, 1.0, 0.0], "c_3": [1.0, -1.0, 0.0], "c_4": [-1.0, -1.0, 0.0]}
    for nm, p in pts.items():
        problem.SetNormalBounds(nm, [0, 0, 1.0], [0, 0, 1.0])
        problem.SetPosBounds(nm, p, p)
    for nm in ("c_3", "c_4"):                      # SetLiftingContact
        problem.SetForceBounds(nm, [0, 0, 0], [0, 0, 0])
        problem.SetForceThreshold(nm, 0.0)
    return dict(mu=0.5, wrench=np.zeros(6))


SETUPS = {"simple": (["contact1"], "ground", setup_simple), "ground": (NAMES, "ground", setup_ground),
          "superquadric": (NAMES, "superquadric", setup_superquadric), "com_planner": (NAMES, "none", setup_com_planner),
          "example_planner": (["micio", "miao"], "ground", setup_example_planner),
          "example_com_planner": (["c_1", "c_2", "c_3", "c_4"], "none", setup_example_com_planner)}


def oracle_problem(case):
    names, env_name, setup = SETUPS[case]
    op = OracleEvalProblem(names, env_name, MASSES.get(case, MASS))
    return op, names, setup(op, op)


def product_problem(case):
    names, env_name, setup = SETUPS[case]
    env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, MASSES.get(case, MASS), env)
    return prob, names, setup(prob, env)


def solution_maps(problem_names, x):
    """CplProblem::GetSolution for every instance: list of (com, {name: (F, p, n)}) in sorted-name order."""
    out = []
    order = sorted(range(len(problem_names)), key=lambda k: problem_names[k])
    for xi in np.asarray(x):
        out.append((xi[0:3], {problem_names[k]: (xi[3 + 9 * k:6 + 9 * k], xi[6 + 9 * k:9 + 9 * k], xi[9 + 9 * k:12 + 9 * k]) for k in order}))
    return out


def solve_and_check(case, problem, names, par, x0, solver_cls=None):
    """Every instance must succeed, except on the superquadric problem: a |x|^10 surface with the contact normals tied to its
    gradient is where the stand-in's l1 line search (no restoration phase) can run out of iterations from an unlucky start --
    there the default start must succeed and at least 90 % of the perturbed ones; every success must pass every EXPECT."""
    res = (solver_cls or LockStepInteriorPoint)(max_iter=1000 if case == "superquadric" else 500).Solve(problem, x0)
    ok = (res.status == SUCCESS).cpu().numpy()
    report = (res.status.tolist(), res.iterations.tolist())
    if case == "superquadric":
        assert ok[0] and ok.mean() >= 0.9, report
    else:
        assert ok.all(), report
    check_expectations(case, names, par, res.x.cpu().numpy()[ok])
    return res


def check_expectations(case, names, par, x):
    """The EXPECT_* lines of the corresponding TEST_F, for every instance."""
    for com, cmap in solution_maps(names, x):
        F_sum, T_sum = np.zeros(3), np.zeros(3)
        for F, p, n in cmap.values():
            F_sum += F
            T_sum += np.cross(p - com, F)
            if case in ("simple", "ground", "example_planner"):
                assert abs(p[2] - par["ground_z"]) < 1e-6            # :53,119
                assert abs(np.linalg.norm(n) - 1.0) < 1e-6           # :54,120
                assert abs(n[2] - 1.0) < 1e-6                        # :55,121
            if case == "superquadric":
                sq = (((p - par["C"]) / par["R"]) ** par["P"]).sum()
                assert abs(sq - 1.0) < 1e-4                          # :196
                assert abs(np.linalg.norm(n) - 1.0) < 1e-6           # :197
                assert (p - par["p_lb"] >= 0.0).all() and (p - par["p_ub"] <= 0.0).all()   # :206-211
            if case != "simple":
                mu = par["mu"]
                assert -F.dot(n) <= RELAX                            # :127,203,279 (strict in the reference)
                assert np.linalg.norm(F - n.dot(F) * n) - mu * F.dot(n) <= RELAX   # :128,204,280
        if case == "simple":
            assert abs(F_sum[2] - (-MASS * G)) < 1e-6                # :59
            continue
        w = par["wrench"]
        mass = par.get("mass", MASS)
        tol_t = 1e-5 if case == "ground" else 1e-4
        assert abs(F_sum[0] - w[0]) < 1e-6 and abs(F_sum[1] - w[1]) < 1e-6   # :131-132
        assert abs(F_sum[2] - (-mass * G + w[2])) < 1e-6             # :133
        assert np.abs(T_sum - w[3:6]).max() < tol_t                  # :134-136


@pytest.mark.parametrize("case", list(SETUPS))
def test_testbasic_through_the_oracle(case):
    op, names, par = oracle_problem(case)
    x0 = starts(op, 4, seed=7)
    res = solve_and_check(case, op, names, par, x0)
    assert res.evaluations == op.calls                               # one oracle batch per evaluator call


def test_solver_agrees_with_scipy_slsqp_on_a_nondegenerate_problem():
    """With a force weight the minimiser is unique: the driver (tol 1e-8) and SciPy's SLSQP on the same oracle callbacks
    must find the same optimal cost."""
    from scipy.optimize import minimize

    op, names, _ = oracle_problem("ground")
    op.SetForceWeight(1e-4)
    x0 = default_start(op, 1)
    res = LockStepInteriorPoint(tol=1e-8).Solve(op, x0)
    assert res.ok() and int(res.iterations[0]) < 60
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
    r = minimize(lambda x: op.o.eval(x)["cost"], x0[0].numpy(), jac=lambda x: op.o.eval(x)["grad"], bounds=list(zip(lb, ub)),
                 constraints=cons, method="SLSQP", options={"maxiter": 500, "ftol": 1e-12})
    assert r.status == 0
    assert abs(float(res.cost[0]) - r.fun) < 1e-6 * abs(r.fun)


def test_dropping_finished_instances_does_not_change_the_others():
    """Working-set compaction (finished instances leave the lock-step batch) is invisible in the results: instances are
    independent, so every iterate, iteration count and solution is bit-identical with and without it."""
    op, _, _ = oracle_problem("ground")
    x0 = starts(op, 12, seed=7)
    a = LockStepInteriorPoint(compact=False).Solve(op, x0)
    b = LockStepInteriorPoint(compact_min=2).Solve(op, x0)
    assert a.ok() and b.ok() and a.rounds == b.rounds
    assert (a.iterations == b.iterations).all()
    assert (a.x.numpy().view(np.int64) == b.x.numpy().view(np.int64)).all()
    assert b.instance_evaluations < a.instance_evaluations


def test_start_at_zero_is_reported_as_invalid_number():
    """x = 0 is the reference's start (Variable3D.cpp:8-10); the friction Jacobian there is 0/0 (SURVEY Q3) and the driver
    says so instead of iterating on NaNs."""
    from centroidalplanner_b200.lockstep_solver import INVALID_NUMBER

    op, _, _ = oracle_problem("ground")
    res = LockStepInteriorPoint(max_iter=5).Solve(op, torch.zeros(1, op.n, dtype=torch.float64))
    assert int(res.status[0]) == INVALID_NUMBER


# ---- GPU: the CUDA evaluator behind the same driver ---------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SETUPS))
def test_testbasic_through_the_cuda_path(case, cuda_device):
    prob, names, par = product_problem(case)
    x0 = starts(prob, 64, seed=7, device=cuda_device)
    before = prob.launch_count()
    res = solve_and_check(case, prob, names, par, x0)
    assert prob.launch_count() - before == res.evaluations           # every evaluator call of the solve was one kernel launch


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ground", "com_planner"])
def test_gpu_solve_trajectory_is_the_oracle_s(case, cuda_device):
    """Host-path evaluations (cplb_eval_host, CUDA kernels) and oracle evaluations under the same CPU linear algebra:
    bit-identical evaluator outputs => bit-identical iterates, iteration counts and solutions."""
    prob, names, _ = product_problem(case)
    op, _, _ = oracle_problem(case)
    x0 = starts(op, 8, seed=11)
    a = LockStepInteriorPoint().Solve(prob, x0)          # CPU tensors -> cplb_eval_host
    b = LockStepInteriorPoint().Solve(op, x0)
    assert a.rounds == b.rounds and a.evaluations == b.evaluations
    assert (a.iterations == b.iterations).all() and (a.status == b.status).all()
    assert (a.x.numpy().view(np.int64) == b.x.numpy().view(np.int64)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["native", "torch"])
def test_com_planner_facade_solve(driver, cuda_device):
    """TEST_F(TestBasic, testCoMPlanner) (tests/TestBasic.cpp:225-292) call for call through the facade mirror; Solve() runs the
    native solve round by default, any other driver on request."""
    planner = cpl.BatchedCoMPlanner(NAMES, MASS)
    planner.SetMu(0.5)
    assert planner.GetMu() == 0.5
    planner.SetContactPosition("contact1", [1.0, 1.0, 0.0])
    planner.SetContactPosition("contact2", [-1.0, 1.0, 0.0])
    planner.SetContactPosition("contact3", [-1.0, -1.0, 0.0])
    planner.SetContactPosition("contact4", [1.0, -1.0, 0.0])
    planner.SetLiftingContact("contact4")
    assert planner.GetLiftingContacts() == ["contact4"]
    for c in NAMES:
        planner.SetForceThreshold(c, 20.0)
    sols = planner.Solve() if driver == "native" else planner.Solve(solver=LockStepInteriorPoint())
    assert planner.last_solve.ok()
    assert (getattr(planner.last_solve, "tail_instances", 0) == 1) == (driver == "native")   # one instance: straight into the tail
    sol = sols[0]
    assert list(sol["contact_values_map"]) == sorted(NAMES)
    F_sum, T_sum = np.zeros(3), np.zeros(3)
    for v in sol["contact_values_map"].values():
        F, p, n = v["force_value"], v["position_value"], v["normal_value"]
        F_sum += F
        T_sum += np.cross(p - sol["com_sol"], F)
        assert -F.dot(n) <= RELAX
        assert np.linalg.norm(F - n.dot(F) * n) - 0.5 * F.dot(n) <= RELAX
    assert np.abs(F_sum - [0.0, 0.0, -MASS * G]).max() < 1e-6
    assert np.abs(T_sum).max() < 1e-4
    assert np.abs(sol["contact_values_map"]["contact4"]["force_value"]).max() == 0.0   # lifting contact carries nothing


@pytest.mark.gpu
def test_instances_that_are_different_problems(cuda_device):
    """INTEGRATION §4b through the solve driver: every instance has its own manipulation wrench and robot mass (per-instance
    parameter arrays forwarded to every evaluation, including the widened Hessian-difference launches); each solution must
    balance ITS wrench and weight (the equilibrium lines of TEST_F testGroundEnv, tests/TestBasic.cpp:131-136)."""
    prob, names, par = product_problem("ground")
    N = 48
    rng = np.random.default_rng(5)
    wrench = np.tile(par["wrench"], (N, 1)) + rng.normal(0.0, 20.0, (N, 6)) * np.array([1, 1, 1, 0.2, 0.2, 1.0])
    mass = rng.uniform(60.0, 140.0, N)
    per_instance = {"wrench": torch.as_tensor(wrench, device=cuda_device), "mass": torch.as_tensor(mass, device=cuda_device)}
    x0 = starts(prob, N, seed=3, device=cuda_device)
    res = LockStepInteriorPoint(compact_min=8).Solve(prob, x0, per_instance=per_instance)   # the parameter arrays are compacted too
    assert (res.status == SUCCESS).all(), (res.status.tolist(), res.iterations.tolist())
    for i, (com, cmap) in enumerate(solution_maps(names, res.x.cpu().numpy())):
        F_sum, T_sum = np.zeros(3), np.zeros(3)
        for F, p, n in cmap.values():
            F_sum += F
            T_sum += np.cross(p - com, F)
            assert abs(p[2] - par["ground_z"]) < 1e-6 and abs(n[2] - 1.0) < 1e-6
            assert -F.dot(n) <= RELAX and np.linalg.norm(F - n.dot(F) * n) - par["mu"] * F.dot(n) <= RELAX
        assert np.abs(F_sum - (wrench[i, :3] - mass[i] * np.array([0.0, 0.0, G]))).max() < 1e-6
        assert np.abs(T_sum - wrench[i, 3:]).max() < 1e-5


# ---- the native solve round (cplb_solve_device: csrc/cplb_solver.cu, csrc/cplb_solver_core.hpp) ----------------------------------
def test_native_solve_round_on_the_cpu_with_the_oracle(tmp_path):
    """tests/native/solver_host_check.cpp runs the SAME per-instance code the GPU runs one CTA per instance (cplb_solver_core.hpp)
    one thread per instance with the oracle behind the batched evaluations: the reference's three four-contact TEST_Fs and
    testSimpleProblem from 64 perturbed starts each; every EXPECT line on every solved instance."""
    import os
    import shutil
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "solver_host_check")
    subprocess.check_call(["make", "-C", os.path.join(root, "oracle"), "libcpl_oracle.so"], stdout=subprocess.DEVNULL)
    subprocess.check_call([shutil.which("g++") or "g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(root, "oracle"),
                           "-I", os.path.join(root, "centroidalplanner_b200", "csrc"), os.path.join(root, "tests", "native", "solver_host_check.cpp"),
                           "-o", exe, "-L", os.path.join(root, "oracle"), "-lcpl_oracle", f"-Wl,-rpath,{os.path.join(root, 'oracle')}", "-lpthread"])
    summary = {}
    for which, n in (("ground", 64), ("complanner", 64), ("simple", 64), ("ground8", 12)):   # ground8: 8 contacts, a 129 x 129 KKT matrix
        r = subprocess.run([exe, which, str(n)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0 and "-> 0 failures" in r.stdout, r.stdout + r.stderr
        summary[which] = r.stdout.strip().splitlines()[-1]
    # the tail (tail_iteration: an instance on its own through all its remaining iterations) taking over at 16 running instances
    # and from the first round: same instances evaluated, same iteration counts, same residuals as the lock-step rounds
    import re

    def key(line):
        return re.search(r"\((\d+) instance evaluations\), max iterations (\d+), worst statics residual (\S+)", line).groups()

    for tail in ("16", "1000"):
        r = subprocess.run([exe, "ground", "64"], capture_output=True, text=True, timeout=600, env=dict(os.environ, SOLVER_TAIL=tail))
        assert r.returncode == 0 and "-> 0 failures" in r.stdout, r.stdout + r.stderr
        assert key(r.stdout.strip().splitlines()[-1]) == key(summary["ground"]), (r.stdout, summary["ground"])
    r = subprocess.run([exe, "superquadric", "24"], capture_output=True, text=True, timeout=900)
    last = r.stdout.strip().splitlines()[-1]
    assert int(last.split("->")[1].split()[0]) <= 2, r.stdout     # an unlucky start may run out of iterations (see solve_and_check)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SETUPS))
def test_testbasic_through_the_native_solve_round(case, cuda_device):
    """The reference's TEST_Fs through cplb_solve_device: 256 starts per problem, every EXPECT line on every instance."""
    prob, names, par = product_problem(case)
    x0 = starts(prob, 256, seed=7, device=cuda_device)
    before = prob.launch_count()
    import functools

    # lock-step rounds to the end (tail_instances=0): a round per iteration of the slowest instance
    res = solve_and_check(case, prob, names, par, x0, solver_cls=functools.partial(cpl.NativeInteriorPoint, tail_instances=0))
    assert res.evaluations == 1 + 4 * res.rounds and prob.launch_count() > before
    assert res.instance_evaluations > 0 and int(res.iterations.max()) == res.rounds and res.tail_instances == 0
    # The tail (one CTA carries an instance through all its remaining iterations, evaluations inline) runs the same arithmetic in
    # the same order: whether it takes over from the first round (default: 256 instances fit the GPU at once), late (once 40 are
    # left) or never, every instance must end at the same bits after the same number of iterations.
    max_iter = 1000 if case == "superquadric" else 500
    for tail, expect_all in ((-1, True), (40, False)):
        alt = cpl.NativeInteriorPoint(max_iter=max_iter, tail_instances=tail).Solve(prob, x0)
        assert torch.equal(alt.status, res.status) and torch.equal(alt.iterations, res.iterations), (case, tail)
        assert torch.equal(alt.x.view(torch.int64), res.x.view(torch.int64)), (case, tail)
        assert torch.equal(alt.lam.view(torch.int64), res.lam.view(torch.int64)) and torch.equal(alt.cost.view(torch.int64), res.cost.view(torch.int64))
        assert alt.instance_evaluations == res.instance_evaluations, (case, tail)
        if expect_all:
            assert alt.tail_instances > 0 and (alt.rounds == 0) == (alt.tail_instances == 256)
        else:
            assert alt.rounds <= res.rounds and alt.tail_instances <= 40     # (all may converge in the same round: no tail then)
            assert (alt.rounds < res.rounds) == (alt.tail_instances > 0)


@pytest.mark.gpu
def test_native_round_is_deterministic(cuda_device):
    """Finished instances leave the working set in the order their CTAs get there (an atomic counter), so the slot an instance
    occupies differs from run to run; what is computed for it must not: two solves of the same 3,000 starts end at the same bits."""
    prob, names, par = product_problem("ground")
    x0 = starts(prob, 3000, seed=17, device=cuda_device)
    a = cpl.NativeInteriorPoint().Solve(prob, x0)
    b = cpl.NativeInteriorPoint().Solve(prob, x0)
    assert a.rounds > 0 and a.tail_instances > 0 and a.ok()
    assert torch.equal(a.iterations, b.iterations) and torch.equal(a.status, b.status)
    assert torch.equal(a.x.view(torch.int64), b.x.view(torch.int64)) and torch.equal(a.lam.view(torch.int64), b.lam.view(torch.int64))


@pytest.mark.gpu
def test_native_round_on_an_eight_contact_problem(cuda_device):
    """Config 4's shape through cplb_solve_device: 8 contacts (n = 75, m = 54: a 129 x 129 KKT matrix, 133 KB of shared memory; the
    dense Jacobian and the Hessian live in global memory).  TestBasic's ground set-up on eight contacts; every solved instance must
    be in static equilibrium on the ground with every force inside its cone."""
    names = ["l_foot_a", "l_foot_b", "r_foot_a", "r_foot_b", "l_hand_a", "l_hand_b", "r_hand_a", "r_hand_b"][::-1]
    env = cpl.Ground()
    env.SetGroundZ(0.1)
    env.SetMu(0.5)
    prob = cpl.BatchedCplProblem(names, MASS, env)
    prob.SetCoMWeight(2.0)
    prob.SetForceWeight(0.0)
    for nm in names:
        prob.SetPosBounds(nm, [-0.3, -0.3, 0.0], [0.3, 0.3, 1.0])
    wrench = np.array([100.0, 0, 0, 0, 0, 100.0])
    prob.SetManipulationWrench(list(wrench))
    x0 = starts(prob, 40, seed=11, device=cuda_device)
    res = cpl.NativeInteriorPoint().Solve(prob, x0)
    ok = (res.status == SUCCESS).cpu().numpy()
    assert ok[0] and ok.mean() >= 0.9, (res.status.tolist(), res.iterations.tolist())
    for com, cmap in np.asarray(solution_maps(names, res.x.cpu().numpy()[ok]), dtype=object):
        F_sum, T_sum = np.zeros(3), np.zeros(3)
        for F, p, n in cmap.values():
            F_sum += F
            T_sum += np.cross(p - com, F)
            assert abs(p[2] - 0.1) < 1e-6 and abs(n[2] - 1.0) < 1e-6
            assert -F.dot(n) <= RELAX and np.linalg.norm(F - n.dot(F) * n) - 0.5 * F.dot(n) <= RELAX
        assert np.abs(F_sum - (wrench[:3] - MASS * np.array([0.0, 0.0, G]))).max() < 1e-6
        assert np.abs(T_sum - wrench[3:]).max() < 1e-4
    lock = cpl.NativeInteriorPoint(tail_instances=0).Solve(prob, x0)
    assert torch.equal(lock.x.view(torch.int64), res.x.view(torch.int64)) and torch.equal(lock.iterations, res.iterations)


@pytest.mark.gpu
def test_native_round_with_per_instance_parameters(cuda_device):
    """A sweep: every instance solves ITS planning problem (own manipulation wrench and mass) through cplb_solve_device, and must
    balance its own wrench and weight (the equilibrium lines of TEST_F testGroundEnv, tests/TestBasic.cpp:131-136).  Lock-step
    rounds (the parameter arrays are gathered into working-set order every round), the tail (reads them by instance) and a mix
    must end at the same bits."""
    prob, names, par = product_problem("ground")
    N = 300
    rng = np.random.default_rng(5)
    wrench = np.tile(par["wrench"], (N, 1)) + rng.normal(0.0, 20.0, (N, 6)) * np.array([1, 1, 1, 0.2, 0.2, 1.0])
    mass = rng.uniform(60.0, 140.0, N)
    mu = rng.uniform(0.4, 0.8, N)
    per_instance = {"wrench": torch.as_tensor(wrench, device=cuda_device), "mass": torch.as_tensor(mass, device=cuda_device),
                    "mu": torch.as_tensor(mu, device=cuda_device)}
    x0 = starts(prob, N, seed=3, device=cuda_device)
    res = cpl.NativeInteriorPoint(tail_instances=0).Solve(prob, x0, per_instance=per_instance)
    ok = (res.status == SUCCESS).cpu().numpy()
    # (random wrenches and friction coefficients: the stand-in's line search, which has no restoration phase, may run out of
    # iterations on a few of them; every instance it reports as solved must pass every line)
    assert ok.mean() >= 0.95, (res.status.tolist(), res.iterations.tolist())
    for i, (com, cmap) in enumerate(solution_maps(names, res.x.cpu().numpy())):
        if not ok[i]:
            continue
        F_sum, T_sum = np.zeros(3), np.zeros(3)
        for F, p, n in cmap.values():
            F_sum += F
            T_sum += np.cross(p - com, F)
            assert abs(p[2] - par["ground_z"]) < 1e-6 and abs(n[2] - 1.0) < 1e-6
            assert -F.dot(n) <= RELAX and np.linalg.norm(F - n.dot(F) * n) - mu[i] * F.dot(n) <= RELAX
        assert np.abs(F_sum - (wrench[i, :3] - mass[i] * np.array([0.0, 0.0, G]))).max() < 1e-6
        assert np.abs(T_sum - wrench[i, 3:]).max() < 1e-5
    for tail in (-1, 100):
        alt = cpl.NativeInteriorPoint(tail_instances=tail).Solve(prob, x0, per_instance=per_instance)
        assert torch.equal(alt.status, res.status) and torch.equal(alt.iterations, res.iterations), tail
        assert torch.equal(alt.x.view(torch.int64), res.x.view(torch.int64)), tail
        # (-1: the tail takes over once the running instances fit the GPU at once -- from the first round if all N do)
        assert 0 < alt.tail_instances <= (N if tail < 0 else tail) and (alt.rounds == 0) == (alt.tail_instances == N)
    # the shared-parameter solve of the same starts is a different problem: the sweep really used the arrays
    shared = cpl.NativeInteriorPoint().Solve(prob, x0)
    assert not torch.equal(shared.x, res.x)
    with pytest.raises(ValueError, match="elements"):
        cpl.NativeInteriorPoint().Solve(prob, x0, per_instance={"mass": per_instance["mass"][:10].contiguous()})


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ground", "com_planner", "example_planner"])
def test_native_round_and_the_previous_driver_find_the_same_solutions(case, cuda_device):
    """Same algorithm, different linear algebra (own pivoted LU in shared memory vs cuBLAS): both drivers must succeed from the
    same starts and, where the minimiser is unique (a force weight makes it so), agree on the optimal cost."""
    prob, names, par = product_problem(case)
    prob.SetForceWeight(1e-4)
    x0 = starts(prob, 32, seed=5, device=cuda_device)
    a = cpl.NativeInteriorPoint(tol=1e-8).Solve(prob, x0)
    b = LockStepInteriorPoint(tol=1e-8).Solve(prob, x0)
    # The native round is deterministic.  The torch driver is not (cuBLAS' batched LU, index_add atomics): at this tolerance about
    # one run in ten leaves an instance or two of the CoMPlanner problem short of the iteration cap, so it only has to solve most.
    okb = b.status == SUCCESS
    assert a.ok() and float(okb.double().mean()) >= 0.9, (a.status.tolist(), b.status.tolist())
    assert float(((a.cost - b.cost).abs() / b.cost.abs().clamp(min=1e-12))[okb].max()) < 1e-6
    assert float(a.constr_viol.max()) <= 1e-8 and float(b.constr_viol[okb].max()) <= 1e-8


@pytest.mark.gpu
def test_native_round_reports_the_zero_start_as_invalid_number_and_checks_its_arguments(cuda_device):
    from centroidalplanner_b200.lockstep_solver import INVALID_NUMBER

    prob, _, _ = product_problem("ground")
    res = cpl.NativeInteriorPoint(max_iter=5).Solve(prob, torch.zeros(3, prob.n, dtype=torch.float64, device=cuda_device))
    assert res.status.tolist() == [INVALID_NUMBER] * 3 and res.rounds == 0
    # through the ABI with every result buffer pre-filled with a sentinel: a rejected start reports 0 iterations and NaN
    # residuals (include/cpl_batched.h), whatever the caller's buffers held
    import ctypes as C
    from centroidalplanner_b200 import _cabi
    from centroidalplanner_b200.problem import _check

    N, f64, i32 = 3, torch.float64, torch.int32
    x0 = torch.zeros(N, prob.n, dtype=f64, device=cuda_device)
    buf = dict(x=torch.full((N, prob.n), 7.0, dtype=f64, device=cuda_device), status=torch.full((N,), 77, dtype=i32, device=cuda_device),
               iters=torch.full((N,), 77, dtype=i32, device=cuda_device), cost=torch.full((N,), 7.0, dtype=f64, device=cuda_device),
               viol=torch.full((N,), 7.0, dtype=f64, device=cuda_device), dual=torch.full((N,), 7.0, dtype=f64, device=cuda_device),
               lam=torch.full((N, prob.m), 7.0, dtype=f64, device=cuda_device))
    out = _cabi.SolveOutputs(*(buf[k].data_ptr() for k in ("x", "status", "iters", "cost", "viol", "dual", "lam")), None, None, None, None)
    opts = cpl.NativeInteriorPoint(max_iter=5).options
    _check(prob._lib.cplb_solve_device(prob._h, N, x0.data_ptr(), None, C.byref(opts), C.byref(out),
                                       C.c_void_p(torch.cuda.current_stream(cuda_device).cuda_stream)))
    torch.cuda.synchronize(cuda_device)
    assert buf["status"].tolist() == [INVALID_NUMBER] * N and buf["iters"].tolist() == [0] * N
    assert torch.isnan(buf["viol"]).all() and torch.isnan(buf["dual"]).all()
    assert not (buf["x"] == 7.0).any() and not (buf["cost"] == 7.0).any() and not (buf["lam"] == 7.0).any()
    with pytest.raises(ValueError, match="device-resident"):
        cpl.NativeInteriorPoint().Solve(prob, torch.zeros(3, prob.n, dtype=torch.float64))
    with pytest.raises(ValueError):
        cpl.NativeInteriorPoint(tol=-1.0).Solve(prob, torch.zeros(3, prob.n, dtype=torch.float64, device=cuda_device))
    sh = cpl.BatchedCplProblem(NAMES, MASS, cpl.Ground(), devices=[0, 0])
    with pytest.raises(ValueError, match="single-device"):
        cpl.NativeInteriorPoint().Solve(sh, torch.zeros(3, sh.n, dtype=torch.float64, device=cuda_device))
