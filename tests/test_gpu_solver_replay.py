"""The native solve round (cplb_solve_device) pinned bit for bit against its CPU replay.

csrc/cplb_solver_core.hpp is the per-instance code of the solve on both sides: one CTA per instance on the GPU, one host thread
per instance in the replay (tests/native/solver_host_engine.hpp, called through tests/native/solver_replay.cpp) with the C oracle
behind the evaluations.  For Ground and no-environment problems every evaluator output is bit-identical to the oracle's; the
first-warp folds replay the GPU's butterfly on the host (warp_fold) and the logarithm / fractional powers of the barrier are
written with IEEE operations only (log_hd, sqrt).  So from the same starts a GPU solve and its replay must end at the same bits:
status, iterations, x, lam, cost, constr_viol and dual_inf, in every mode of the round (lock-step to the end, the tail from the
first round, a mix), and truncated after k iterations.  A wrong pivot, a slot mix-up in the KKT assembly, a barrier or
regularisation update that is off or a line search that takes the wrong candidate all show up here even where the solve still
converges.

Superquadric problems are excluded on purpose: pow() is upstream in their evaluator, whose outputs are only <= 1e-12 equal to the
oracle's, so the replay cannot match them bit for bit.
"""
from __future__ import annotations

import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

import centroidalplanner_b200 as cpl
from centroidalplanner_b200.lockstep_solver import INVALID_NUMBER, MAX_ITER, SUCCESS
from helpers import OracleEvalProblem
from test_solve import MASS, MASSES, SETUPS, starts

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NATIVE = os.path.join(ROOT, "tests", "native")
CSRC = os.path.join(ROOT, "centroidalplanner_b200", "csrc")
ORACLE = os.path.join(ROOT, "oracle")
FIELDS = ("status", "iterations", "x", "lam", "cost", "constr_viol", "dual_inf")

NAMES8 = ["l_foot_a", "l_foot_b", "r_foot_a", "r_foot_b", "l_hand_a", "l_hand_b", "r_hand_a", "r_hand_b"][::-1]


def setup_ground8(problem, env):  # test_solve.py::test_native_round_on_an_eight_contact_problem
    env.SetGroundZ(0.1)
    env.SetMu(0.5)
    problem.SetCoMWeight(2.0)
    problem.SetForceWeight(0.0)
    for nm in NAMES8:
        problem.SetPosBounds(nm, [-0.3, -0.3, 0.0], [0.3, 0.3, 1.0])
    problem.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])


CASES = {k: SETUPS[k] for k in ("simple", "ground", "com_planner", "example_planner", "example_com_planner")}
CASES["ground8"] = (NAMES8, "ground", setup_ground8)   # a 129 x 129 KKT matrix, the dense matrices in global memory
STARTS = {"ground8": 48}                               # 256 elsewhere


def oracle_side(case):
    names, env_name, setup = CASES[case]
    op = OracleEvalProblem(names, env_name, MASSES.get(case, MASS))
    setup(op, op)
    return op


def product_side(case):
    names, env_name, setup = CASES[case]
    env = {"none": None, "ground": cpl.Ground}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, MASSES.get(case, MASS), env)
    setup(prob, env)
    return prob


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
    lib.cplb_replay_solve.restype = C.c_int
    lib.cplb_replay_solve.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p] + [C.c_void_p] * 8 + [C.c_int]
    return lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def replay(lib, op, x0, solver):
    """The CPU replay of `solver` (a NativeInteriorPoint: its options) on the oracle problem op from the starts x0."""
    x0 = np.ascontiguousarray(np.asarray(x0.cpu() if torch.is_tensor(x0) else x0, dtype=np.float64))
    N = x0.shape[0]
    out = dict(x=np.empty((N, op.n)), lam=np.empty((N, op.m)), status=np.empty(N, np.int32), iterations=np.empty(N, np.int32),
               cost=np.empty(N), constr_viol=np.empty(N), dual_inf=np.empty(N))
    stats = np.zeros(4, np.int64)
    rc = lib.cplb_replay_solve(C.c_void_p(op.o._h), N, _ptr(x0), C.cast(C.byref(solver.options), C.c_void_p), _ptr(out["x"]), _ptr(out["lam"]),
                               _ptr(out["status"]), _ptr(out["iterations"]), _ptr(out["cost"]), _ptr(out["constr_viol"]),
                               _ptr(out["dual_inf"]), _ptr(stats), os.cpu_count() or 1)
    assert rc == 0
    out["status"] = out["status"].astype(np.int64)
    out["iterations"] = out["iterations"].astype(np.int64)
    out.update(rounds=int(stats[0]), evaluations=int(stats[1]), instance_evaluations=int(stats[2]), tail_instances=int(stats[3]))
    return out


def gpu_fields(res):
    return {k: getattr(res, k).cpu().numpy() for k in FIELDS}


def same_bits(a, b):
    """Bit-identical, NaNs matched by position (payloads may differ between devices)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype.kind != "f":
        return bool((a == b).all())
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all() and (a.view(np.int64)[~na] == b.view(np.int64)[~nb]).all())


def differing_instances(got, want):
    bad = np.zeros(len(want["status"]), dtype=bool)
    for k in FIELDS:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        a2, b2 = a.reshape(len(bad), -1), b.reshape(len(bad), -1)
        if a.dtype.kind == "f":
            na, nb = np.isnan(a2), np.isnan(b2)
            diff = (na != nb) | (~na & ~nb & (a2.view(np.int64) != b2.view(np.int64)))
        else:
            diff = a2 != b2
        bad |= diff.any(axis=1)
    return np.nonzero(bad)[0]


def first_parting_iteration(lib, prob, op, x0, i, kw):
    """Bisects max_iter for the first k at which the GPU and the replay of instance i differ (the GPU solve of the whole batch,
    the replay of instance i alone: an instance's result does not depend on its batch)."""
    def differs(k):
        s = cpl.NativeInteriorPoint(**dict(kw, max_iter=k))
        g = {f: v[i:i + 1] for f, v in gpu_fields(s.Solve(prob, x0)).items()}
        return len(differing_instances(g, replay(lib, op, x0[i:i + 1], s))) > 0
    lo, hi = 0, kw.get("max_iter", 500)   # invariant: no difference at lo (checked), a difference at hi
    if differs(0):
        return 0
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if differs(mid) else (mid, hi)
    return hi


def assert_same_solve(lib, prob, op, x0, got, want, kw, what):
    bad = differing_instances(got, want)
    if len(bad) == 0:
        return
    i = int(bad[0])
    fields = [k for k in FIELDS if not same_bits(np.asarray(got[k])[i], np.asarray(want[k])[i])]
    k = first_parting_iteration(lib, prob, op, x0, i, kw)
    pytest.fail(f"{what}: {len(bad)} instances differ from the CPU replay; first instance {i} (fields {fields}), "
                f"which parts from the replay at iteration {k} (max_iter bisection)")


# ---- CPU: the shared logarithm ---------------------------------------------------------------------------------------------
def log_inputs():
    rng = np.random.default_rng(2026)
    xs = [np.array([1.0, 0.5, 2.0, np.sqrt(2.0), np.sqrt(0.5), 5e-324, 2.2250738585072014e-308, 2.225073858507201e-308,
                    1.7976931348623157e308, 1e-300, 1e300, np.e, 10.0])]
    p2 = np.ldexp(1.0, np.arange(-1074, 1024))                                 # exact powers of two and their neighbours
    xs += [p2, np.nextafter(p2, 0.0)[1:], np.nextafter(p2, np.inf)]
    k = np.arange(1, 20001, dtype=np.float64)                                 # 1 +- k eps
    xs += [1.0 + k * 2.0 ** -52, 1.0 - k * 2.0 ** -53]
    per = 450                                                                 # every binade, subnormals included
    e = np.repeat(np.arange(-1074, 1024), per)
    xs.append(np.ldexp(1.0 + rng.random(e.size), e))
    xs.append(rng.integers(1, 2 ** 52, 20000).astype(np.uint64).view(np.float64))   # subnormal bit patterns
    xs.append(np.exp(rng.uniform(-40.0, 10.0, 40000)))                         # gap, mu and slack magnitudes
    x = np.concatenate(xs)
    return x[np.isfinite(x) & (x > 0)]


@pytest.fixture(scope="module")
def log_hd(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("log") / "liblog_hd.so")
    subprocess.check_call([_cxx(), "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", CSRC, os.path.join(NATIVE, "log_hd_shim.cpp"),
                           "-o", so])
    lib = C.CDLL(so)
    lib.cplb_log_hd_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]

    def f(x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        y = np.empty_like(x)
        lib.cplb_log_hd_batch(_ptr(x), _ptr(y), x.size)
        return y
    return f


def test_shared_log_is_within_one_ulp_of_the_true_value(log_hd):
    """log_hd against mpmath at 50 digits on ~10^6 points: every binade from the subnormals to 1e308, exact powers of two and
    their neighbours, 1 +- k eps.  At most 1 ulp of the true value everywhere."""
    mpmath = pytest.importorskip("mpmath")
    x = log_inputs()
    assert x.size >= 1_000_000
    y = log_hd(x)
    mpmath.mp.dps = 50
    hi = np.empty_like(x)
    lo = np.empty_like(x)
    for t, v in enumerate(x.tolist()):
        L = mpmath.log(mpmath.mpf(v))
        h = float(L)
        hi[t] = h
        lo[t] = float(L - h)
    exact0 = hi == 0.0
    assert (x[exact0] == 1.0).all() and (y[exact0] == 0.0).all() and not np.signbit(y[exact0]).any()   # log(1) = +0 exactly
    m, ex = np.frexp(np.where(exact0, 1.0, hi))
    ulp = np.ldexp(1.0, ex - 53)
    ulp = np.where((np.abs(m) == 0.5) & (lo * hi < 0), ulp / 2, ulp)         # true value just below a power of two
    err = np.abs((y - hi) - lo) / ulp                                         # y - hi is exact (they are ulps apart)
    err[exact0] = 0.0
    worst = int(np.argmax(err))
    assert err.max() <= 1.0, f"log_hd({x[worst]!r}) = {y[worst]!r}, {err[worst]:.3f} ulp from the true value"


def test_shared_log_special_values(log_hd):
    y = log_hd(np.array([0.0, -0.0, -1.0, -5e-324, -np.inf, np.inf, np.nan, 1.0]))
    assert y[0] == -np.inf and y[1] == -np.inf
    assert np.isnan(y[2:5]).all() and y[5] == np.inf and np.isnan(y[6]) and y[7] == 0.0 and not np.signbit(y[7])


def test_the_cpu_replay_runs_and_solves(replay_lib):
    """The CPU half on its own: the replay of the ground problem solves every start (TestBasic's lines are checked by
    test_solve.py::test_native_solve_round_on_the_cpu_with_the_oracle), and rejected starts report the documented outputs."""
    op = oracle_side("ground")
    x0 = starts(op, 16, seed=7)
    x0[3] = 0.0
    x0[9, 4] = float("nan")
    r = replay(replay_lib, op, x0, cpl.NativeInteriorPoint(tail_instances=0))
    rejected = np.zeros(16, dtype=bool)
    rejected[[3, 9]] = True
    assert (r["status"][~rejected] == SUCCESS).all() and (r["status"][rejected] == INVALID_NUMBER).all()
    assert (r["iterations"][rejected] == 0).all() and np.isnan(r["constr_viol"][rejected]).all() and np.isnan(r["dual_inf"][rejected]).all()
    assert r["rounds"] == r["iterations"].max() and r["evaluations"] == 1 + 4 * r["rounds"]


# ---- GPU: device and host builds of the same elementary functions -------------------------------------------------------------
@pytest.mark.gpu
def test_shared_log_and_sqrt_forms_give_the_same_bits_on_the_gpu(cuda_device, tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    exe = str(tmp_path / "log_hd_check")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-fmad=false", "-std=c++17", "-Xcompiler", "-ffp-contract=off",
                           "-I", CSRC, os.path.join(NATIVE, "log_hd_check.cu"), "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("mismatches 0") == 3, r.stdout


# ---- GPU: the solve against its replay ----------------------------------------------------------------------------------------
def test_oracle_and_product_problems_have_the_same_shape():
    """Guard on set-up drift: the replay's problem (the oracle) and the GPU's (the product) have the same bounds and structure."""
    for case in CASES:
        op, prob = oracle_side(case), product_side(case)
        assert (op.n, op.m, op.nnz) == (prob.n, prob.m, prob.nnz), case
        for a, b in zip(op.GetJacobianStructure(), prob.GetJacobianStructure()):
            assert np.array_equal(np.asarray(a), np.asarray(b)), case
        for a, b in zip(op.GetBoundsOnOptimizationVariables() + op.GetBoundsOnConstraints(),
                        prob.GetBoundsOnOptimizationVariables() + prob.GetBoundsOnConstraints()):
            assert same_bits(np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)), case


MODES = {"lockstep": 0, "tail": -1, "mixed": 40}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_gpu_solve_is_its_cpu_replay_bit_for_bit(case, replay_lib, cuda_device):
    op, prob = oracle_side(case), product_side(case)
    N = STARTS.get(case, 256)
    x0 = starts(op, N, seed=7)
    want = replay(replay_lib, op, x0, cpl.NativeInteriorPoint(tail_instances=0))
    assert (want["status"] == SUCCESS).mean() >= 0.9, want["status"]
    xg = x0.to(cuda_device)
    for mode, tail in MODES.items():
        kw = dict(tail_instances=tail)
        res = cpl.NativeInteriorPoint(**kw).Solve(prob, xg)
        assert_same_solve(replay_lib, prob, op, xg, gpu_fields(res), want, kw, f"{case}, {mode}")
        if mode == "lockstep":
            assert (res.rounds, res.evaluations, res.instance_evaluations) == (want["rounds"], want["evaluations"], want["instance_evaluations"])


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ground", "com_planner", "example_planner", "ground8"])
def test_truncated_gpu_solves_are_their_cpu_replay(case, replay_lib, cuda_device):
    """A solve stopped after k iterations returns the k-th iterate with status MaxIter (unless it converged first): every field
    equal to the replay's there too, in the lock-step rounds and in the tail."""
    op, prob = oracle_side(case), product_side(case)
    x0 = starts(op, 64 if case != "ground8" else 24, seed=13)
    xg = x0.to(cuda_device)
    for k in (1, 2, 3, 5, 10):
        want = replay(replay_lib, op, x0, cpl.NativeInteriorPoint(max_iter=k, tail_instances=0))
        assert ((want["status"] == MAX_ITER) | (want["status"] == SUCCESS)).all() and (want["iterations"] <= k).all()
        assert (want["status"] == MAX_ITER).any()
        for mode in ("lockstep", "tail"):
            kw = dict(max_iter=k, tail_instances=MODES[mode])
            got = gpu_fields(cpl.NativeInteriorPoint(**kw).Solve(prob, xg))
            assert_same_solve(replay_lib, prob, op, xg, got, want, kw, f"{case}, max_iter {k}, {mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["lockstep", "tail"])
def test_rejected_starts_do_not_touch_the_rest_of_the_batch(mode, replay_lib, cuda_device):
    """Every seventh start is zero (0/0 in the friction Jacobian) or holds a NaN: those report INVALID_NUMBER after 0 iterations
    with NaN residuals; every other instance equals the replay of the valid starts alone."""
    op, prob = oracle_side("ground"), product_side("ground")
    N = 128
    x0 = starts(op, N, seed=19)
    rejected = np.arange(N) % 7 == 3
    for t, i in enumerate(np.nonzero(rejected)[0]):
        if t % 2:
            x0[i] = 0.0
        else:
            x0[i, (5 * t) % op.n] = float("nan")
    kw = dict(tail_instances=MODES[mode])
    res = cpl.NativeInteriorPoint(**kw).Solve(prob, x0.to(cuda_device))
    got = gpu_fields(res)
    assert (got["status"][rejected] == INVALID_NUMBER).all() and (got["iterations"][rejected] == 0).all()
    assert np.isnan(got["constr_viol"][rejected]).all() and np.isnan(got["dual_inf"][rejected]).all()
    valid = np.nonzero(~rejected)[0]
    want = replay(replay_lib, op, x0[valid], cpl.NativeInteriorPoint(**kw))
    assert_same_solve(replay_lib, prob, op, x0[valid].to(cuda_device), {k: v[valid] for k, v in got.items()}, want, kw, f"valid starts, {mode}")


# ---- GPU: the shape limit of the solve ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("env_name", ["ground", "none"])
def test_solve_refuses_shapes_beyond_the_shared_memory_of_a_cta(env_name, cuda_device):
    """One instance's KKT system lives in one CTA's shared memory.  The largest contact count that fits solves; one more is
    refused up front with a message naming the count and the limit."""
    def problem(k):
        env = cpl.Ground() if env_name == "ground" else None
        if env is not None:
            env.SetGroundZ(0.1)
        return cpl.BatchedCplProblem(["c%02d" % c for c in range(k)], MASS, env)

    big = problem(32)
    with pytest.raises(ValueError, match="32 contacts") as e:
        cpl.NativeInteriorPoint(max_iter=3).Solve(big, starts(big, 2, seed=1, device=cuda_device))
    limit = int(re.search(r"at most (\d+) contacts", str(e.value)).group(1))
    assert limit == {"ground": 10, "none": 13}[env_name]          # include/cpl_batched.h, next to cplb_solve_device
    ok = problem(limit)
    res = cpl.NativeInteriorPoint(max_iter=3).Solve(ok, starts(ok, 4, seed=1, device=cuda_device))
    assert ((res.status == SUCCESS) | (res.status == MAX_ITER)).all() and (res.iterations > 0).all()
    over = problem(limit + 1)
    with pytest.raises(ValueError, match=f"{limit + 1} contacts.*at most {limit} contacts"):
        cpl.NativeInteriorPoint(max_iter=3).Solve(over, starts(over, 4, seed=1, device=cuda_device))
