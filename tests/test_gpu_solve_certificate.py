"""The native solve round's results certified independently of the solver: GPU half.

cplb_solve_device's results (x, lam, cost, constr_viol, dual_inf) are checked with tests/solve_certificate.py -- the C oracle at the
returned x, exact stationarity residual judged by IPOPT's scaled measure, multiplier signs, complementarity -- on every TestBasic
set-up including the Superquadric one (which no replay covers: pow() is upstream there), the 8-contact problem, the lock-step
rounds alone and the tail alone, and a batch large enough to go through many working-set compactions.

Per-instance parameter sweeps (every field of cplb_instance_params, and one with only the six cost fields) are pinned bit for bit
against the per-instance CPU replay (one oracle per instance: tests/native/solver_replay.cpp) in three modes of the round, and each
instance is certified against ITS problem.  A gather that hands an instance another instance's cost parameters for the
difference or line-search points, or a tail that reads a shared value instead of the instance's, still converges -- to the
optimum of the wrong problem; the replay and the certificate both see it.
"""
from __future__ import annotations

import numpy as np
import pytest
import torch

import centroidalplanner_b200 as cpl
from centroidalplanner_b200.lockstep_solver import SUCCESS
from solve_certificate import assert_certified
from test_solve import starts
from test_solve_certificate import (OUT, instance_oracles, oracle_side, oracles_of, product_side, replay, replay_lib,  # noqa: F401
                                    same_bits, sweep)

MODES = {"lockstep": 0, "tail": -1, "mixed": 40}


def gpu_out(res):
    return {k: getattr(res, k).cpu().numpy() for k in OUT}


def on_device(per, dev):
    return {k: torch.as_tensor(v, device=dev).contiguous() for k, v in per.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["simple", "ground", "superquadric", "com_planner", "example_planner", "example_com_planner", "ground8"])
def test_gpu_solutions_are_certified_kkt_points(case, cuda_device):
    """Lock-step rounds to the end and the tail from the first round, each certified on every instance it reports as solved.
    Superquadric: solve_and_check's bar (the default start and >= 90 % of the others succeed), evaluations <= 1e-12 from the
    oracle's, so the cost is compared to 1e-12 relative."""
    op, prob = oracle_side(case), product_side(case)
    N = 48 if case == "ground8" else 256
    sq = case == "superquadric"
    x0 = starts(op, N, seed=7)
    for mode in ("lockstep", "tail"):
        s = cpl.NativeInteriorPoint(max_iter=1000 if sq else 500, tail_instances=MODES[mode])
        res = s.Solve(prob, x0.to(cuda_device))
        out = gpu_out(res)
        ok = out["status"] == SUCCESS
        if sq or case == "ground8":
            assert ok[0] and ok.mean() >= 0.9, (case, mode, out["status"].tolist())
        else:
            assert ok.all(), (case, mode, out["status"].tolist())
        assert (res.tail_instances > 0) == (mode == "tail")
        assert_certified(op.o, s.options, x0.numpy(), out, np.nonzero(ok)[0], pow_upstream=sq, what=f"{case}, {mode}")


@pytest.mark.gpu
def test_gpu_solutions_of_a_large_batch_are_certified(cuda_device):
    """4,096 starts: many lock-step rounds with a shrinking working set (finished instances leave it), then the tail.  Every 32nd
    instance is certified."""
    op, prob = oracle_side("ground"), product_side("ground")
    N = 4096
    x0 = starts(op, N, seed=23)
    s = cpl.NativeInteriorPoint()
    res = s.Solve(prob, x0.to(cuda_device))
    out = gpu_out(res)
    assert (out["status"] == SUCCESS).all()
    assert res.rounds > 0 and 0 < res.tail_instances < N
    assert_certified(op.o, s.options, x0.numpy(), out, np.arange(0, N, 32), what="4096 starts")


def first_parting_iteration(lib, prob, ops, per_dev, x0, i, kw):
    """Bisects max_iter for the first k at which the GPU solve (whole batch) and the replay of instance i alone (its oracle) differ."""
    def differs(k):
        s = cpl.NativeInteriorPoint(**dict(kw, max_iter=k))
        g = {f: v[i:i + 1] for f, v in gpu_out(s.Solve(prob, x0, per_instance=per_dev)).items()}
        w = replay(lib, [ops[i]], x0[i:i + 1], s)
        return not all(same_bits(g[f], w[f]) for f in OUT)
    lo, hi = 0, kw.get("max_iter", 500)
    if differs(0):
        return 0
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (lo, mid) if differs(mid) else (mid, hi)
    return hi


@pytest.mark.gpu
@pytest.mark.parametrize("cost_only", [False, True], ids=["all_fields", "cost_fields"])
@pytest.mark.parametrize("case", ["ground", "none"])
def test_gpu_per_instance_solve_is_its_per_instance_replay_and_certified(case, cost_only, replay_lib, cuda_device):
    """256 instances, each its own planning problem: every field of cplb_instance_params per instance (or only the cost fields).
    The GPU solve -- lock-step rounds to the end (parameters gathered into slot order every round), the tail from the first round
    (read by instance), and a mix -- ends at the replay's bits on every output; every solved instance is a KKT point of its own
    problem."""
    N = 256
    per = sweep(case, N, seed=29 if cost_only else 31, cost_only=cost_only)
    ops = instance_oracles(case, per)
    prob = product_side(case)
    x0 = starts(ops[0], N, seed=3)
    xg, per_dev = x0.to(cuda_device), on_device(per, cuda_device)
    want = replay(replay_lib, ops, x0, cpl.NativeInteriorPoint(tail_instances=0))
    assert (want["status"] == SUCCESS).mean() >= 0.95, want["status"].tolist()
    for mode, tail in MODES.items():
        kw = dict(tail_instances=tail)
        s = cpl.NativeInteriorPoint(**kw)
        got = gpu_out(s.Solve(prob, xg, per_instance=per_dev))
        bad = np.zeros(N, dtype=bool)
        for f in OUT:
            a, b = np.asarray(got[f]).reshape(N, -1), np.asarray(want[f]).reshape(N, -1)
            bad |= np.array([not same_bits(a[i], b[i]) for i in range(N)])
        if bad.any():
            i = int(np.nonzero(bad)[0][0])
            fields = [f for f in OUT if not same_bits(np.asarray(got[f])[i], np.asarray(want[f])[i])]
            k = first_parting_iteration(replay_lib, prob, ops, per_dev, xg, i, kw)
            pytest.fail(f"{case} sweep, {mode}: {int(bad.sum())} instances differ from the per-instance replay; first instance {i} "
                        f"(fields {fields}), which parts from the replay at iteration {k} (max_iter bisection)")
        ok = np.nonzero(got["status"] == SUCCESS)[0]
        if mode == "lockstep":
            assert_certified(oracles_of(ops), s.options, x0.numpy(), got, ok, what=f"{case} sweep, {mode}")
