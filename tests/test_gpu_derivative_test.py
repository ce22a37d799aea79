"""The batched first-order derivative test (cplb_derivative_test_device, csrc/cplb_derivtest.cu) on the GPU.

The reference turns on IPOPT's `derivative_test first-order` before every solve (src/CentroidalPlanner.cpp:26).  The product's
counterpart is pinned here bit for bit, all seven outputs:
  * against a CPU replay -- NumPy over the C oracle: the oracle evaluates the widened rows x + h_j e_j, and the rule of
    include/cpl_batched.h is written with the same IEEE operations (the library is built with -fmad=false).  Ground and
    no-environment problems only: pow() is upstream in the Superquadric evaluator, which is not bit-identical to the oracle.
  * against the widened batched path -- x widened to N (n + 1) rows in torch, one cplb_eval_device of g + cost, the differences
    and the comparison in torch.  The fused kernel evaluates with eval_points, whose bits are the batched kernels', so this holds
    in every environment and at every contact count (16 and 32 contacts: several column chunks per instance).
Expected counts always come from one of these references, never from a hand-picked threshold: forward differences at h = 1e-8
lose about eps |f| / h, and with default weights the cost is large enough that small gradient entries are flagged honestly.
"""
from __future__ import annotations

import numpy as np
import pytest
import torch

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic
from helpers import configure, make_pair
from oracle import cpl_oracle_py as orc
from test_gpu_solver_replay import CASES, oracle_side, product_side, same_bits
from test_solve import starts

pytestmark = pytest.mark.gpu

KEYS = ("num_wrong", "num_wrong_outside", "max_rel_error", "worst_row", "worst_col", "jac_fd", "grad_fd")


def _reduce(rel, wrong_outside_mask, n, tol):
    """rel (N, n + m n) in entry order -> the five per-instance outputs."""
    N = rel.shape[0]
    wrong = ~(rel <= tol)
    key = np.where(np.isnan(rel), np.inf, rel)
    worst = np.argmax(key, axis=1)                    # the first entry with the largest key
    return dict(num_wrong=wrong.sum(axis=1).astype(np.int32),
                num_wrong_outside=(wrong[:, n:] & wrong_outside_mask).sum(axis=1).astype(np.int32),
                max_rel_error=rel[np.arange(N), worst],
                worst_row=np.where(worst < n, -1, (worst - n) // n).astype(np.int32),
                worst_col=np.where(worst < n, worst, (worst - n) % n).astype(np.int32))


def replay(o, x, perturbation=1e-8, tol=1e-4):
    """The derivative test of one oracle problem at the rows of x (N, n), in NumPy."""
    x = np.ascontiguousarray(np.asarray(x, dtype=np.float64))
    N, n = x.shape
    m = o.m
    iRow, jCol = o.structure()
    with np.errstate(all="ignore"):
        ax = np.abs(x)
        h = perturbation * np.where(ax > 1.0, ax, 1.0)
        X = np.repeat(x[:, None, :], n, axis=1)
        cols = np.arange(n)
        X[:, cols, cols] = x + h
        base = o.eval_batch(x, nthreads=8)
        pert = o.eval_batch(X.reshape(N * n, n), want=("g", "cost"), nthreads=8)
        gp, fp = pert["g"].reshape(N, n, m), pert["cost"].reshape(N, n)
        grad_fd = (fp - base["cost"][:, None]) / h
        jfd = ((gp - base["g"][:, None, :]) / h[:, :, None]).transpose(0, 2, 1)        # (N, m, n)
        dense = np.zeros((N, m, n))
        dense[:, iRow, jCol] = base["jac"]
        ag, aj = np.abs(base["grad"]), np.abs(dense)
        rel_g = np.abs(grad_fd - base["grad"]) / np.where(ag > 1.0, ag, 1.0)
        rel_j = np.abs(jfd - dense) / np.where(aj > 1.0, aj, 1.0)
    outside = np.ones((m, n), dtype=bool)
    outside[iRow, jCol] = False
    out = _reduce(np.concatenate([rel_g, rel_j.reshape(N, m * n)], axis=1), outside.reshape(-1), n, tol)
    out.update(jac_fd=np.ascontiguousarray(jfd[:, iRow, jCol]), grad_fd=grad_fd)
    return out


def widened(prob, x, per_instance=None, perturbation=1e-8, tol=1e-4):
    """The unfused alternative on the GPU: x widened to N (n + 1) rows, one batched evaluation of g + cost, and the differences
    and the comparison in torch (the same IEEE operations as the kernel)."""
    N, n = x.shape
    m = prob.m
    iRow, jCol = (torch.as_tensor(a, device=x.device, dtype=torch.int64) for a in prob.GetJacobianStructure())
    ax = x.abs()
    h = perturbation * torch.where(ax > 1.0, ax, torch.ones_like(ax))
    X = x[:, None, :].repeat(1, n + 1, 1)
    cols = torch.arange(n, device=x.device)
    X[:, 1 + cols, cols] = x + h
    wide_pi = None if per_instance is None else {k: v.repeat_interleave(n + 1, dim=0).contiguous() for k, v in per_instance.items()}
    ev = prob.eval(X.reshape(N * (n + 1), n), g=True, jac=False, cost=True, per_instance=wide_pi)
    g, f = ev["g"].reshape(N, n + 1, m), ev["cost"].reshape(N, n + 1)
    ex = prob.eval(x, g=False, jac=True, cost=False, grad=True, per_instance=per_instance)
    grad_fd = (f[:, 1:] - f[:, :1]) / h
    jfd = ((g[:, 1:, :] - g[:, :1, :]) / h[:, :, None]).transpose(1, 2)
    dense = torch.zeros(N, m, n, dtype=torch.float64, device=x.device)
    dense[:, iRow, jCol] = ex["jac"]
    ag, aj = ex["grad"].abs(), dense.abs()
    rel_g = (grad_fd - ex["grad"]).abs() / torch.where(ag > 1.0, ag, torch.ones_like(ag))
    rel_j = (jfd - dense).abs() / torch.where(aj > 1.0, aj, torch.ones_like(aj))
    rel = torch.cat([rel_g, rel_j.reshape(N, m * n)], dim=1)
    wrong = ~(rel <= tol)
    outside = torch.ones(m, n, dtype=torch.bool, device=x.device)
    outside[iRow, jCol] = False
    worst = torch.where(rel.isnan(), torch.full_like(rel, float("inf")), rel).argmax(dim=1)
    return dict(num_wrong=wrong.sum(dim=1).to(torch.int32), num_wrong_outside=(wrong[:, n:] & outside.reshape(-1)).sum(dim=1).to(torch.int32),
                max_rel_error=rel.gather(1, worst[:, None])[:, 0],
                worst_row=torch.where(worst < n, -1, torch.div(worst - n, n, rounding_mode="floor")).to(torch.int32),
                worst_col=torch.where(worst < n, worst, (worst - n) % n).to(torch.int32),
                jac_fd=jfd[:, iRow, jCol].contiguous(), grad_fd=grad_fd)


def as_numpy(rep):
    get = rep.__getitem__ if isinstance(rep, dict) else (lambda k: getattr(rep, k))
    return {k: get(k).cpu().numpy() if torch.is_tensor(get(k)) else np.asarray(get(k)) for k in KEYS}


def assert_same(got, want, what):
    for k in KEYS:
        a, b = np.asarray(got[k]), np.asarray(want[k])
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        if not same_bits(a, b):
            bad = np.nonzero(~((a == b) | (np.isnan(a) & np.isnan(b))).reshape(len(a), -1).all(axis=1))[0] if a.dtype.kind == "f" \
                else np.nonzero((a != b).reshape(len(a), -1).any(axis=1))[0]
            i = int(bad[0]) if len(bad) else 0
            raise AssertionError(f"{what}: {k} differs first at instance {i}: got {a[i]!r}, want {b[i]!r}")


@pytest.mark.parametrize("case", sorted(CASES))
def test_bit_for_bit_against_the_cpu_replay(case, cuda_device):
    """The test-solve cases (1, 2, 4 and 8 contacts, sorted order != vector order, no environment), seeded starts around the
    default start: all seven outputs equal the NumPy-over-oracle replay."""
    prob, op = product_side(case), oracle_side(case)
    x0 = starts(prob, 48, seed=11, device=cuda_device)
    got = as_numpy(prob.DerivativeTest(x0))
    want = replay(op.o, x0.cpu().numpy())
    assert_same(got, want, case)
    assert got["jac_fd"].shape == (48, prob.nnz) and got["grad_fd"].shape == (48, prob.n)


def _all_per_instance(names, N, rng, device):
    nc = len(names)
    arrs = dict(mass=rng.uniform(60.0, 140.0, N), wrench=rng.normal(0.0, 20.0, (N, 6)), mu=rng.uniform(0.3, 0.9, N),
                force_threshold=rng.uniform(0.0, 30.0, (N, nc)), ground_z=rng.uniform(-0.1, 0.2, N), com_ref=rng.normal(0.0, 0.3, (N, 3)),
                com_weight=rng.uniform(0.5, 3.0, N), pos_ref=rng.normal(0.0, 0.3, (N, 3 * nc)), force_ref=rng.normal(0.0, 50.0, (N, 3 * nc)),
                pos_weight=rng.uniform(0.0, 2.0, (N, nc)), force_weight=rng.uniform(0.0, 0.01, (N, nc)))
    return arrs, {k: torch.as_tensor(np.ascontiguousarray(v), device=device) for k, v in arrs.items()}


def test_per_instance_arrays_against_one_oracle_per_instance(cuda_device):
    """64 instances, every field of cplb_instance_params given per instance: each instance is replayed by its own oracle, configured
    through its setters."""
    case = "ground"
    names = CASES[case][0]
    prob = product_side(case)
    N = 64
    arrs, pi = _all_per_instance(names, N, np.random.default_rng(21), cuda_device)
    x0 = starts(prob, N, seed=12, device=cuda_device)
    got = as_numpy(prob.DerivativeTest(x0, per_instance=pi))
    xs = x0.cpu().numpy()
    rows = []
    for i in range(N):
        op = oracle_side(case)
        o = op.o
        o.set_mass(arrs["mass"][i])
        o.set_wrench(arrs["wrench"][i])
        o.set_mu(arrs["mu"][i])
        o.set_ground_z(arrs["ground_z"][i])
        o.set_com_ref(arrs["com_ref"][i])
        o.set_com_weight(arrs["com_weight"][i])
        for k, nm in enumerate(names):
            o.set_force_threshold(nm, arrs["force_threshold"][i, k])
            o.set_pos_ref(nm, arrs["pos_ref"][i, 3 * k:3 * k + 3])
            o.set_force_ref(nm, arrs["force_ref"][i, 3 * k:3 * k + 3])
            o.set_contact_pos_weight(nm, arrs["pos_weight"][i, k])
            o.set_contact_force_weight(nm, arrs["force_weight"][i, k])
        rows.append(replay(o, xs[i:i + 1]))
    want = {k: np.concatenate([r[k] for r in rows]) for k in KEYS}
    assert_same(got, want, "per-instance")
    # the arrays were used: the shared-parameter test of the same points differs
    shared = as_numpy(prob.DerivativeTest(x0))
    assert not same_bits(shared["grad_fd"], got["grad_fd"])


def _big_case(nc, env_name, seed):
    names = ["k%02d" % ((7 * i) % nc) for i in range(nc)]
    env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, 100.0, env)
    configure(prob, env, names, env_name)
    gen = synthetic.superquadric_batch if env_name == "superquadric" else synthetic.ground_batch
    return prob, lambda N: gen(N, nc, seed)


@pytest.mark.parametrize("case", ["ground1", "ground4", "noenv4", "superquadric4", "ground8", "superquadric8", "superquadric4_fracP",
                                  "ground16", "noenv32", "superquadric32"])
def test_bit_for_bit_against_the_widened_batched_path(case, cuda_device):
    """Every environment, Superquadric included, up to 32 contacts (the solver stops at 10 / 13): the fused kernel's outputs are the
    widened path's, bit for bit."""
    if case == "ground16":
        prob, gen = _big_case(16, "ground", 41)
    elif case == "noenv32":
        prob, gen = _big_case(32, "none", 43)
    else:
        prob, _, gen = make_pair(case)
    N = 64 if prob.n < 200 else 16
    x = torch.as_tensor(gen(N), device=cuda_device)
    got = as_numpy(prob.DerivativeTest(x))
    want = as_numpy(widened(prob, x))
    assert_same(got, want, case)
    # per-instance parameters take the same path on both sides
    _, pi = _all_per_instance(prob.contact_names, N, np.random.default_rng(5), cuda_device)
    if prob._env_kind != _cabi.ENV_GROUND:
        del pi["ground_z"]
    assert_same(as_numpy(prob.DerivativeTest(x, per_instance=pi)), as_numpy(widened(prob, x, per_instance=pi)), case + " per-instance")


def _kink_point(F, n=(0.0, 0.0, 1.0)):
    return np.array([[0.0, 0.0, 1.0, *F, 0.0, 0.0, 0.0, *n]])


def test_detection_at_the_friction_cone_kink(cuda_device):
    """F = (1e-9, 0, 100), n = (0, 0, 1): the tangential-force norm of FrictionCone (FrictionCone.cpp:85-87) has a kink at zero
    tangential force, and the forward difference across it is wrong: the F_y entry of the contact's second FrictionCone row is
    flagged (difference ~0.9, exact 0).  The normal's tangential entries of that row cross the same kink scaled by F.n = 100, so the
    worst entry is the n_y one of that row.  The replay agrees on all seven outputs."""
    prob = cpl.BatchedCplProblem(["contact1"], 100.0, cpl.Ground())
    o = orc.Oracle(["contact1"], orc.ENV_GROUND, 100.0)
    x = _kink_point((1e-9, 0.0, 100.0))
    xd = torch.as_tensor(x, device=cuda_device)
    got = as_numpy(prob.DerivativeTest(xd))
    assert_same(got, replay(o, x), "kink")
    cone = prob.GetContactRow("contact1") + 4                  # the two FrictionCone rows follow the four environment rows
    Fy = prob.GetBlockColumn(cpl.BLOCK_FORCE, "contact1") + 1
    ny = prob.GetBlockColumn(cpl.BLOCK_NORMAL, "contact1") + 1
    iRow, jCol = prob.GetJacobianStructure()
    exact = prob.eval(xd, g=False, jac=True)["jac"].cpu().numpy()[0]
    slot = int(np.nonzero((iRow == cone + 1) & (jCol == Fy))[0][0])
    assert abs(got["jac_fd"][0, slot] - exact[slot]) / max(1.0, abs(exact[slot])) > 1e-4   # flagged
    assert (got["worst_row"][0], got["worst_col"][0]) == (cone + 1, ny)
    assert got["num_wrong"][0] >= 2 and got["num_wrong_outside"][0] == 0 and got["max_rel_error"][0] > 1.0


def test_detection_at_zero_tangential_force(cuda_device):
    """F_t = 0 exactly: the Jacobian holds NaN there (0/0, the documented quirk, SURVEY Q3); the NaN entry counts as wrong and
    max_rel_error is NaN."""
    prob = cpl.BatchedCplProblem(["contact1"], 100.0, cpl.Ground())
    o = orc.Oracle(["contact1"], orc.ENV_GROUND, 100.0)
    x = _kink_point((0.0, 0.0, 100.0))
    got = as_numpy(prob.DerivativeTest(torch.as_tensor(x, device=cuda_device)))
    want = replay(o, x)
    assert_same(got, want, "F_t = 0")
    assert np.isnan(got["max_rel_error"][0]) and got["num_wrong"][0] >= 1
    ex = prob.eval(torch.as_tensor(x, device=cuda_device), g=False, jac=True)["jac"].cpu().numpy()
    iRow, jCol = prob.GetJacobianStructure()
    first_nan = np.nonzero(np.isnan(ex[0]))[0]
    assert first_nan.size
    # the worst entry is the first NaN in the entry order (gradient first, then the dense Jacobian row by row)
    entries = sorted(int(iRow[s]) * prob.n + int(jCol[s]) for s in first_nan)
    assert got["worst_row"][0] * prob.n + got["worst_col"][0] == entries[0]


def test_planner_facade_runs_the_test_before_an_untouched_solve(cuda_device):
    """Solve(derivative_test=True) fills last_derivative_test (the report of DerivativeTest at x0) and the solve's x, status and
    iterations are bit-identical to those of derivative_test=False."""
    names = ["contact1", "contact2", "contact3", "contact4"]
    env = cpl.Ground()
    env.SetGroundZ(0.1)
    env.SetMu(0.5)
    pl = cpl.BatchedCentroidalPlanner(names, 100.0, env)
    pl.SetManipulationWrench([100.0, 0, 0, 0, 0, 100.0])
    prob = pl.GetCplProblem()
    x0 = starts(prob, 32, seed=4, device=cuda_device)
    pl.Solve(x0)
    plain = pl.last_solve
    assert not hasattr(pl, "last_derivative_test")
    pl.Solve(x0, derivative_test=True)
    checked = pl.last_solve
    for k in ("x", "status", "iterations"):
        assert torch.equal(getattr(plain, k).view(torch.int64) if k == "x" else getattr(plain, k),
                           getattr(checked, k).view(torch.int64) if k == "x" else getattr(checked, k)), k
    assert_same(as_numpy(pl.last_derivative_test), as_numpy(prob.DerivativeTest(x0)), "facade")


def test_pybind_and_ctypes_return_the_same_bits(cuda_device):
    # the module is imported under one name in the whole session, as the other pybind tests import it: a second name would load
    # the same extension twice, and pybind11 refuses to register its types again
    import os
    import sys

    sys.path.insert(0, os.path.dirname(cpl.__file__))
    import pycplb

    names = ["r_foot", "l_foot", "r_hand", "l_hand"]
    env = cpl.Ground()
    env.SetGroundZ(0.05)
    env.SetMu(0.6)
    prob = cpl.BatchedCplProblem(names, 80.0, env)
    penv = pycplb.Ground()
    penv.SetGroundZ(0.05)
    penv.SetMu(0.6)
    pp = pycplb.BatchedProblem(names, 80.0, penv, 0)
    x = torch.as_tensor(synthetic.ground_batch(100, 4, 3), device=cuda_device)
    want = as_numpy(prob.DerivativeTest(x, tol=1e-5))
    N = x.shape[0]
    out = dict(num_wrong=torch.empty(N, dtype=torch.int32, device=cuda_device), num_wrong_outside=torch.empty(N, dtype=torch.int32, device=cuda_device),
               max_rel_error=torch.empty(N, dtype=torch.float64, device=cuda_device), worst_row=torch.empty(N, dtype=torch.int32, device=cuda_device),
               worst_col=torch.empty(N, dtype=torch.int32, device=cuda_device), jac_fd=torch.empty(N, pp.nnz, dtype=torch.float64, device=cuda_device),
               grad_fd=torch.empty(N, pp.n, dtype=torch.float64, device=cuda_device))
    pp.derivative_test_device(N, x.data_ptr(), **{k: v.data_ptr() for k, v in out.items()}, stream=torch.cuda.current_stream().cuda_stream,
                              tol=1e-5)
    torch.cuda.synchronize()
    assert_same(as_numpy(out), want, "pybind vs ctypes")


def test_call_is_asynchronous_and_streams_do_not_interfere(cuda_device):
    """The call enqueues and returns: with the stream held busy, it comes back before the stream has finished.  Two calls on two
    streams give the same results as two calls in series; each counts one launch."""
    prob, _, gen = make_pair("ground8")
    xa = torch.as_tensor(gen(512), device=cuda_device)
    xb = torch.as_tensor(synthetic.ground_batch(512, 8, 99), device=cuda_device)
    serial_a, serial_b = as_numpy(prob.DerivativeTest(xa)), as_numpy(prob.DerivativeTest(xb))   # (also uploads the structure table)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    launches = prob.launch_count()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(200_000_000)                     # ~0.1 s of spinning on s1
        ra = prob.DerivativeTest(xa)
        returned_before_done = not s1.query()
    with torch.cuda.stream(s2):
        rb = prob.DerivativeTest(xb)
    assert returned_before_done
    torch.cuda.synchronize()
    assert prob.launch_count() == launches + 2
    assert_same(as_numpy(ra), serial_a, "stream 1")
    assert_same(as_numpy(rb), serial_b, "stream 2")

