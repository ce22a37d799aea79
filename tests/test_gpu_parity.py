"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same
seeded inputs.  Bit-exact wherever no pow() is upstream; <= 1e-12 relative elsewhere (north_star)."""
import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import synthetic

from helpers import CASES, assert_parity, make_pair, same_bits, set_oracle_instance, to_instance_major

pytestmark = pytest.mark.gpu

LAYOUTS = [cpl.INSTANCE_MAJOR, cpl.COMPONENT_MAJOR]


def run_device(prob, x_np, layout, device, **want):
    import torch

    xd = torch.from_numpy(np.ascontiguousarray(x_np)).to(device)
    if layout == cpl.COMPONENT_MAJOR:
        xd = xd.t().contiguous()
    out = prob.eval(xd, layout=layout, **want)
    torch.cuda.synchronize()
    return {k: (None if v is None else to_instance_major(v.cpu().numpy(), layout)) for k, v in out.items()}


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", sorted(CASES))
def test_all_outputs_match_oracle(case, layout, cuda_device):
    prob, o, gen = make_pair(case)
    x = gen(1000)
    want = o.eval_batch(x, nthreads=4)
    got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
    assert_parity(got, want, o, f"{case}/layout{layout}", x)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", sorted(CASES))
def test_gpu_matches_reference_golden_vectors(case, layout, cuda_device):
    """tests/golden/ref_vectors.npz: outputs of the reference's own sources (tools/make_golden.py)."""
    import os

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_vectors.npz"))
    prob, o, _ = make_pair(case)
    x = z[f"{case}/x"]
    want = {k: z[f"{case}/{k}"] for k in ("g", "jac", "cost", "grad")}
    got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
    assert_parity(got, want, o, f"golden/{case}/layout{layout}", x)
    r, c = prob.GetJacobianStructure()
    assert np.array_equal(r, z[f"{case}/iRow"]) and np.array_equal(c, z[f"{case}/jCol"])


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("N", [1, 2, 7, 31, 33, 129, 4097])
def test_ragged_batch_sizes(N, layout, cuda_device):
    for case in ("ground4", "superquadric3", "noenv8"):
        prob, o, gen = make_pair(case)
        x = gen(N)
        want = o.eval_batch(x)
        got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
        assert_parity(got, want, o, f"{case}/N{N}/layout{layout}", x)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("want", [dict(g=True, jac=False), dict(g=False, jac=True), dict(g=False, jac=False, cost=True),
                                  dict(g=False, jac=False, grad=True), dict(g=True, jac=True, cost=True, grad=False)])
def test_output_subsets_do_not_touch_other_buffers(want, layout, cuda_device):
    prob, o, gen = make_pair("superquadric4")
    x = gen(513)
    ref = o.eval_batch(x)
    got = run_device(prob, x, layout, cuda_device, **want)
    for k in ("g", "jac", "cost", "grad"):
        if not want.get(k, False):
            assert got[k] is None
            ref[k] = None
    assert_parity(got, ref, o, f"subset{want}/layout{layout}", x)


@pytest.mark.parametrize("G", [1024, 1023])  # 1023: buffers only 8-byte aligned -> the non-bulk (plain load/store) tile path
@pytest.mark.parametrize("N", [1, 5, 8, 33, 1000, 4099])
@pytest.mark.parametrize("case", ["ground4", "superquadric3", "noenv8", "ground12"])
def test_no_write_outside_the_output_slices(case, N, G, cuda_device):
    """Guard bands (compute-sanitizer is closed on this pool): every output buffer sits inside a larger allocation
    filled with a sentinel; after the evaluation the bands before/after -- and, component-major, the pitch padding
    columns ld > N -- must still hold the sentinel, and the payload must equal the oracle."""
    import ctypes as C

    import torch

    from centroidalplanner_b200 import _cabi

    prob, o, gen = make_pair(case)
    x = gen(N)
    want = o.eval_batch(x)
    SENT = -7.25e77
    lib = _cabi.load()
    for layout in LAYOUTS:
        ld = N if layout == cpl.INSTANCE_MAJOR else N + 37
        def make(length):
            count = N * length if layout == cpl.INSTANCE_MAJOR else length * ld
            buf = torch.full((count + 2 * G,), SENT, dtype=torch.float64, device=cuda_device)
            return buf, buf[G:G + count]
        bufs = {k: make(L) for k, L in (("g", o.m), ("jac", o.nnz), ("grad", o.n), ("cost", 1))}
        xfull, xin = make(o.n)
        if layout == cpl.INSTANCE_MAJOR:
            xin.copy_(torch.from_numpy(x).reshape(-1))
        else:
            xin.view(o.n, ld)[:, :N].copy_(torch.from_numpy(np.ascontiguousarray(x.T)))
            bufs["cost"] = make(1)  # cost is always cost[i]
        if layout == cpl.COMPONENT_MAJOR:
            cbuf = torch.full((N + 2 * G,), SENT, dtype=torch.float64, device=cuda_device)
            bufs["cost"] = (cbuf, cbuf[G:G + N])
        args = _cabi.EvalArgs(N, layout, 0, ld, xin.data_ptr(), bufs["g"][1].data_ptr(), bufs["jac"][1].data_ptr(),
                              bufs["cost"][1].data_ptr(), bufs["grad"][1].data_ptr(), None)
        assert lib.cplb_eval_device(prob._h, C.byref(args), None) == 0, lib.cplb_last_error()
        torch.cuda.synchronize()
        got = {}
        for k, L in (("g", o.m), ("jac", o.nnz), ("grad", o.n)):
            full, view = bufs[k]
            assert bool((full[:G] == SENT).all()) and bool((full[-G:] == SENT).all()), f"{case}/{k}: guard band overwritten"
            if layout == cpl.INSTANCE_MAJOR:
                got[k] = view.view(N, L).cpu().numpy()
            else:
                v2 = view.view(L, ld)
                assert bool((v2[:, N:] == SENT).all()), f"{case}/{k}: pitch padding overwritten"
                got[k] = v2[:, :N].t().contiguous().cpu().numpy()
        full, view = bufs["cost"]
        assert bool((full[:G] == SENT).all()) and bool((full[-G:] == SENT).all())
        got["cost"] = view[:N].cpu().numpy()
        assert bool((xfull[:G] == SENT).all()) and bool((xfull[-G:] == SENT).all())
        assert_parity(got, want, o, f"guard/{case}/N{N}/layout{layout}", x)


def test_config1_testbasic_parameter_set(cuda_device):
    """BASELINE.json configs[0] (tests/TestBasic.cpp:64-99, testGroundEnv) with its exact parameters: mass 100, Ground
    z = 0.1, mu = 0.5, W_CoM = 2, W_F = 0, W_p = 1, wrench (100,0,0,0,0,100), p bounds [-0.3,0.3]^2 x [0,1].  IPOPT is
    absent, so the solve itself cannot run; the evaluator is checked on this parameter set at (i) the start point
    x = 0, (ii) the closed-form equilibrium point, (iii) 1,000 random points -- GPU vs oracle, bit for bit."""
    from test_oracle import equilibrium_x

    from helpers import OracleProblem

    names = synthetic.NAMES4
    env = cpl.Ground()
    env.SetGroundZ(synthetic.TESTBASIC["ground_z"])
    env.SetMu(synthetic.TESTBASIC["mu"])
    prob = cpl.BatchedCplProblem(names, synthetic.TESTBASIC["mass"], env)
    synthetic.configure_testbasic(prob, names)
    op = OracleProblem(names, "ground", synthetic.TESTBASIC["mass"])
    op.SetGroundZ(synthetic.TESTBASIC["ground_z"])
    op.SetMu(synthetic.TESTBASIC["mu"])
    synthetic.configure_testbasic(op, names)
    o = op.o
    lb, ub = prob.GetBoundsOnOptimizationVariables()
    for k in range(4):
        assert list(lb[6 + 9 * k:9 + 9 * k]) == [-0.3, -0.3, 0.0] and list(ub[6 + 9 * k:9 + 9 * k]) == [0.3, 0.3, 1.0]
    x = np.concatenate([np.zeros((1, 39)), equilibrium_x()[None, :], synthetic.ground_batch(1000)])
    want = o.eval_batch(x)
    assert np.isnan(want["jac"][0]).sum() == 24            # (i): 0/0 in the six entries of each friction-cone row
    assert list(want["g"][1, :6]) == [-100.0, 0.0, 0.0, 0.0, 0.0, -100.0]   # (ii): balanced except for the manipulation wrench
    for layout in LAYOUTS:
        got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
        assert_parity(got, want, o, f"config1/layout{layout}")


def test_default_start_point_nan_pattern(cuda_device):
    """x = 0 (Variable3D.cpp:8-10): NaN exactly where the reference produces NaN (SURVEY Q3)."""
    for case in ("ground4", "noenv4", "superquadric4"):
        prob, o, _ = make_pair(case)
        x = np.zeros((40, o.n))
        want = o.eval_batch(x)
        assert np.isnan(want["jac"]).any()
        for layout in LAYOUTS:
            got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
            assert_parity(got, want, o, f"{case}/zeros/layout{layout}", x)


def test_equilibrium_point_and_special_values(cuda_device):
    from test_oracle import equilibrium_x

    prob, o, _ = make_pair("ground4", rich=False)
    prob.SetManipulationWrench(np.zeros(6))
    o.set_wrench(np.zeros(6))
    x = np.tile(equilibrium_x(), (64, 1))
    x[1, 3:6] = [0.0, 0.0, -0.0]
    x[2, 0:3] = [1e300, -1e300, 1e-300]      # overflow / underflow are values, not errors
    x[3, 9:12] = [np.inf, 0.0, 1.0]
    x[4, 5] = np.nan
    x[5, 3:6] = [1e-200, -2e-200, 3e-200]    # friction-row divisions outside the fast-division window
    x[6, 3:6] = [1e200, 2e200, -3e200]
    x[7, 3:6] = [4.9e-324, 0.0, 1e-310]      # subnormal forces
    x[8, 9:12] = [1e-170, 1e-170, 1e-170]    # subnormal products
    want = o.eval_batch(x)
    assert np.abs(want["g"][0, :6]).max() <= 1e-12
    for layout in LAYOUTS:
        got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
        assert_parity(got, want, o, f"special/layout{layout}")


def test_superquadric_outside_the_fast_power_window(cuda_device):
    """Contacts absurdly close to / far from the superquadric centre leave the integer-power fast path
    (cplb_device.cuh); zero offsets hit the reference's own 1/(p-C)^2 poles (SURVEY Q3)."""
    prob, o, gen = make_pair("superquadric4")
    x = gen(256)
    C = np.array([0.0, 0.0, 1.0])
    x[0, 6:9] = C + [1e-20, 2e-25, -3e-18]
    x[1, 6:9] = C + [1e15, -1e14, 1e16]
    x[2, 6:9] = C + [0.0, 0.1, 0.2]        # d_x = 0: inf * 0 in the diagonal entries
    x[3, 6:9] = C                          # all three zero
    x[4, 15:18] = C + [1e-3, 1e-2, -1e-2]
    x[5, 15:18] = [np.inf, 0.0, 1.5]
    x[6, 15:18] = [np.nan, 0.2, 1.2]
    x[7, 24:27] = C + [-1e-8, 1e-8, 1e-8]
    want = o.eval_batch(x)
    for layout in LAYOUTS:
        got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
        # rows 0, 1, 7: d so small/large that d^(2P) and the 1/(p-C)^2 factors over/underflow -- the reference itself
        # returns 0/inf/NaN mixtures there; positions of non-finite values must agree, finite values to 1e-12
        assert_parity(got, want, o, f"sq-window/layout{layout}", x)


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", ["ground4", "noenv8", "superquadric4", "superquadric4_fracP"])
def test_other_eigen_reduction_order(case, layout, cuda_device):
    """cplb_set_reduction_order(1): v0+(v1+v2) instead of (v0+v1)+v2 in every Eigen 3-term reduction the reference
    relies on -- the oracle has the same switch, and the two must stay bit-identical (pow-free outputs) in both modes."""
    prob, o, gen = make_pair(case)
    x = gen(2000)
    a = o.eval_batch(x)
    prob.SetReductionOrder(1)
    o.set_reduction_order(1)
    b = o.eval_batch(x)
    assert not np.array_equal(a["g"], b["g"], equal_nan=True)   # the switch changes some last bits ...
    got = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
    assert_parity(got, b, o, f"order1/{case}/layout{layout}", x)  # ... and the GPU follows the oracle
    with pytest.raises(ValueError):
        prob.SetReductionOrder(2)


@pytest.mark.parametrize("layout", LAYOUTS)
def test_inputs_ready_queue_of_independent_batches(layout, cuda_device):
    """CPLB_DEVICE_INPUTS_READY: a queue of independent batches on one stream, each evaluation allowed to read its x
    while the previous kernel is still running.  Results must be those of plain stream order; each batch is written to
    its own outputs, and a final plain-order evaluation that REUSES an output buffer of the queue must still come last."""
    import torch

    prob, o, gen = make_pair("ground4")
    N, Q = 65536, 6
    xs = [torch.from_numpy(gen(N) + 0.001 * q).to(cuda_device) for q in range(Q)]
    xin = [x if layout == cpl.INSTANCE_MAJOR else x.t().contiguous() for x in xs]
    outs = [prob.eval(xi, g=True, jac=True, layout=layout, inputs_ready=True) for xi in xin]      # back to back, one stream
    again = prob.eval(xin[0], g=True, jac=True, layout=layout, out={"g": outs[3]["g"], "jac": outs[3]["jac"]})  # plain order
    torch.cuda.synchronize()
    ref0 = prob.eval(xin[0], g=True, jac=True, layout=layout)
    torch.cuda.synchronize()
    assert torch.equal(again["jac"].view(torch.int64), ref0["jac"].view(torch.int64))               # not clobbered by batch 3
    for q in (1, 2, 4, 5):
        sub = np.arange(0, N, 997)
        want = o.eval_batch(xs[q].cpu().numpy()[sub], want=("g", "jac"))
        got = {k: to_instance_major(outs[q][k].cpu().numpy(), layout)[sub] for k in ("g", "jac")}
        assert_parity(got, want, o, f"ready-queue/{q}/layout{layout}")


def test_parameter_updates_are_seen_by_the_next_launch(cuda_device):
    prob, o, gen = make_pair("ground4")
    x = gen(256)
    prob.SetManipulationWrench([1, 2, 3, 4, 5, 6])
    o.set_wrench([1, 2, 3, 4, 5, 6])
    prob.SetMass(73.5)
    o.set_mass(73.5)
    prob.SetMu(0.9)
    o.set_mu(0.9)
    prob.SetForceThreshold("contact3", 42.0)
    o.set_force_threshold("contact3", 42.0)
    got = run_device(prob, x, cpl.INSTANCE_MAJOR, cuda_device, g=True, jac=True, cost=True, grad=True)
    assert_parity(got, o.eval_batch(x), o, "updated parameters")


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("layout", LAYOUTS)
def test_host_buffer_path_matches_device_path(layout, pinned, cuda_device):
    """cplb_eval_host (H2D, kernel, D2H in chunks on several streams) == cplb_eval_device, bit for bit -- with pinned
    caller buffers (asynchronous copies straight from/to them) and with pageable ones (packed through pinned mirrors)."""
    import torch

    prob, o, gen = make_pair("ground8")
    N = 40000  # > one chunk, ragged last chunk
    x = gen(N)
    xin = x if layout == cpl.INSTANCE_MAJOR else np.ascontiguousarray(x.T)
    out = None
    if pinned:
        shp = (lambda L: (N, L)) if layout == cpl.INSTANCE_MAJOR else (lambda L: (L, N))
        xt = torch.empty(xin.shape, dtype=torch.float64, pin_memory=True)
        xt.copy_(torch.from_numpy(xin))
        xin = xt
        out = {"g": torch.empty(shp(o.m), dtype=torch.float64, pin_memory=True), "jac": torch.empty(shp(o.nnz), dtype=torch.float64, pin_memory=True),
               "cost": torch.empty(N, dtype=torch.float64, pin_memory=True), "grad": torch.empty(shp(o.n), dtype=torch.float64, pin_memory=True)}
    host = prob.eval(xin, g=True, jac=True, cost=True, grad=True, layout=layout, out=out)
    host = {k: to_instance_major(np.asarray(v), layout) for k, v in host.items()}
    dev = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
    for k in ("g", "jac", "cost", "grad"):
        assert same_bits(host[k], dev[k]), k
    sub = np.arange(0, N, 37)
    want = o.eval_batch(x[sub])
    assert_parity({k: host[k][sub] for k in host}, want, o, "host path")


@pytest.mark.parametrize("path", ["device", "host"])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", ["ground4", "noenv8", "superquadric3"])
def test_per_instance_parameters(case, layout, path, cuda_device):
    """cplb_instance_params: every instance carries its own mass, wrench, mu, thresholds, ground height, references and
    weights.  The oracle plays N different CplProblems, one per instance."""
    import torch

    prob, o, gen = make_pair(case)
    N = 300
    nc = o.nc
    x = gen(N)
    rng = np.random.default_rng(42)
    pi = {"mass": rng.uniform(20, 150, N), "wrench": rng.uniform(-50, 50, (N, 6)), "mu": rng.uniform(0.2, 1.2, N),
          "force_threshold": rng.uniform(0, 30, (N, nc)), "com_ref": rng.uniform(-1, 1, (N, 3)), "com_weight": rng.uniform(0, 3, N),
          "pos_ref": rng.uniform(-1, 1, (N, 3 * nc)), "force_ref": rng.uniform(-100, 100, (N, 3 * nc)),
          "pos_weight": rng.uniform(0, 2, (N, nc)), "force_weight": rng.uniform(0, 0.1, (N, nc))}
    if case.startswith("ground"):
        pi["ground_z"] = rng.uniform(-0.2, 0.4, N)
    want = {"g": np.zeros((N, o.m)), "jac": np.zeros((N, o.nnz)), "cost": np.zeros(N), "grad": np.zeros((N, o.n))}
    for i in range(N):
        set_oracle_instance(o, pi, i)
        e = o.eval(x[i])
        for key in want:
            want[key][i] = e[key]
    cm = layout == cpl.COMPONENT_MAJOR
    lay = lambda a: np.ascontiguousarray(a.T) if (cm and a.ndim == 2) else np.ascontiguousarray(a)  # noqa: E731
    if path == "device":
        pid = {k: torch.from_numpy(lay(v)).to(cuda_device) for k, v in pi.items()}
        xd = torch.from_numpy(lay(x)).to(cuda_device)
        out = prob.eval(xd, g=True, jac=True, cost=True, grad=True, layout=layout, per_instance=pid)
        torch.cuda.synchronize()
        got = {k: to_instance_major(v.cpu().numpy(), layout) for k, v in out.items()}
    else:
        out = prob.eval(lay(x), g=True, jac=True, cost=True, grad=True, layout=layout, per_instance={k: lay(v) for k, v in pi.items()})
        got = {k: to_instance_major(v, layout) for k, v in out.items()}
    assert_parity(got, want, o, f"per-instance/{case}/layout{layout}/{path}", x)
    # a subset of the arrays: the others fall back to the shared values (the oracle still holds instance N-1's)
    sub = {"wrench": pi["wrench"], "mu": pi["mu"]}
    if path == "device":
        out = prob.eval(xd, g=True, jac=False, layout=layout, per_instance={k: torch.from_numpy(lay(v)).to(cuda_device) for k, v in sub.items()})
        torch.cuda.synchronize()
        g_sub = to_instance_major(out["g"].cpu().numpy(), layout)
        o2 = make_pair(case)[1]
        for i in (0, N - 1):
            o2.set_wrench(pi["wrench"][i])
            o2.set_mu(pi["mu"][i])
            assert same_bits(g_sub[i][:6], o2.eval(x[i])["g"][:6])


@pytest.mark.parametrize("misaligned", [False, True])
@pytest.mark.parametrize("want", [dict(g=True, jac=True), dict(g=True, jac=False), dict(g=False, jac=True)])
@pytest.mark.parametrize("case,N", [("ground4", 4096), ("ground4", 301), ("ground4", 5), ("ground8", 1023), ("ground1", 777), ("ground12", 130)])
def test_per_instance_constraint_only_evaluations(case, N, want, misaligned, cuda_device):
    """Constraint-only evaluations of Ground problems are the ones whose per-instance parameter slices the instance-major
    kernel stages in shared memory with the x tile (bulk copies; plain copies for ragged tiles and for arrays that are not
    16-byte aligned): every instance, every output, both layouts, against N oracle problems."""
    import torch

    prob, o, gen = make_pair(case)
    nc = o.nc
    x = gen(N)
    rng = np.random.default_rng(N)
    pi = {"mass": rng.uniform(20, 150, N), "wrench": rng.uniform(-50, 50, (N, 6)), "mu": rng.uniform(0.2, 1.2, N),
          "force_threshold": rng.uniform(0, 30, (N, nc)), "ground_z": rng.uniform(-0.2, 0.4, N)}
    ref = {"g": np.zeros((N, o.m)), "jac": np.zeros((N, o.nnz))}
    for i in range(N):
        set_oracle_instance(o, pi, i)
        e = o.eval(x[i], want=("g", "jac"))
        ref["g"][i], ref["jac"][i] = e["g"], e["jac"]

    def dev(a):
        a = np.ascontiguousarray(a)
        if not misaligned:
            return torch.from_numpy(a).to(cuda_device)
        pad = torch.empty(a.size + 1, dtype=torch.float64, device=cuda_device)       # 8 bytes off a 16-byte boundary
        view = pad[1:].view(a.shape)
        view.copy_(torch.from_numpy(a))
        assert view.data_ptr() % 16 == 8
        return view

    for layout in LAYOUTS:
        lay = (lambda a: a.T) if layout == cpl.COMPONENT_MAJOR else (lambda a: a)
        pid = {k: dev(lay(v) if v.ndim == 2 else v) for k, v in pi.items()}
        out = prob.eval(torch.from_numpy(np.ascontiguousarray(lay(x))).to(cuda_device), layout=layout, per_instance=pid, **want)
        torch.cuda.synchronize()
        got = {k: (None if v is None else to_instance_major(v.cpu().numpy(), layout)) for k, v in out.items()}
        assert_parity(got, {k: (ref[k] if want.get(k) else None) for k in ref}, o, f"per-instance-constraints/{case}/{N}/layout{layout}", x)


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("want", [dict(g=True, jac=False), dict(g=False, jac=True), dict(g=False, jac=False, cost=True),
                                  dict(g=False, jac=False, grad=True), dict(g=True, jac=False, cost=True, grad=True)])
def test_host_path_output_subsets(want, layout, pinned, cuda_device):
    """Every subset of outputs through cplb_eval_host: the staging-buffer sections shift with the subset."""
    import torch

    prob, o, gen = make_pair("noenv8")
    N = 20011  # two chunks, ragged
    x = gen(N)
    ref = o.eval_batch(x, nthreads=4)
    xin = x if layout == cpl.INSTANCE_MAJOR else np.ascontiguousarray(x.T)
    out = None
    if pinned:
        shp = (lambda L: (N, L)) if layout == cpl.INSTANCE_MAJOR else (lambda L: (L, N))
        xt = torch.empty(xin.shape, dtype=torch.float64, pin_memory=True)
        xt.copy_(torch.from_numpy(xin))
        xin = xt
        lens = {"g": o.m, "jac": o.nnz, "grad": o.n}
        out = {k: torch.empty((N,) if k == "cost" else shp(lens[k]), dtype=torch.float64, pin_memory=True)
               for k in ("g", "jac", "cost", "grad") if want.get(k, False)}
    got = prob.eval(xin, layout=layout, out=out, **want)
    for k in ("g", "jac", "cost", "grad"):
        if not want.get(k, False):
            assert got[k] is None
        else:
            assert same_bits(to_instance_major(np.asarray(got[k]), layout), ref[k]), k


@pytest.mark.parametrize("layout", LAYOUTS)
def test_concurrent_host_threads_on_their_own_streams(layout, cuda_device):
    """include/cpl_batched.h: evaluation takes x as an argument, so several host threads may evaluate disjoint
    instance ranges of ONE problem on different streams at once (each IPOPT thread with its own slice)."""
    import threading

    import torch

    prob, o, gen = make_pair("ground8")
    N, T = 48000, 6
    x = gen(N)
    xd = torch.from_numpy(x).to(cuda_device)
    ref = run_device(prob, x, layout, cuda_device, g=True, jac=True, cost=True, grad=True)
    bounds = np.linspace(0, N, T + 1).astype(int)
    results, errors = [None] * T, []

    def work(t):
        try:
            st = torch.cuda.Stream(cuda_device)
            lo, hi = int(bounds[t]), int(bounds[t + 1])
            with torch.cuda.stream(st):
                xin = xd[lo:hi].contiguous() if layout == cpl.INSTANCE_MAJOR else xd[lo:hi].t().contiguous()
                for _ in range(5):  # repeated launches interleave across the threads
                    out = prob.eval(xin, g=True, jac=True, cost=True, grad=True, layout=layout, stream=st.cuda_stream)
                st.synchronize()
            results[t] = {k: to_instance_major(v.cpu().numpy(), layout) for k, v in out.items()}
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    th = [threading.Thread(target=work, args=(t,)) for t in range(T)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    for k in ("g", "jac", "cost", "grad"):
        assert same_bits(np.concatenate([r[k] for r in results]), ref[k]), k


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", ["ground4", "superquadric4", "noenv8"])
def test_host_path_can_skip_constant_jacobian_slots(case, layout, cuda_device):
    """CPLB_HOST_JAC_CONSTANTS_PRESENT: constant slots may be skipped (component-major: a sentinel there survives),
    every x-dependent slot is transferred; after FillJacobianConstants the buffer equals the full evaluation."""
    prob, o, gen = make_pair(case)
    N = 20000
    x = gen(N)
    xin = x if layout == cpl.INSTANCE_MAJOR else np.ascontiguousarray(x.T)
    full = prob.eval(xin, g=True, jac=True, layout=layout)
    mask, _ = prob.GetJacobianConstants()
    jac = np.full_like(full["jac"], -9.5)
    part = prob.eval(xin, g=True, jac=True, layout=layout, out={"jac": jac}, jac_constants_present=True)
    a, b = to_instance_major(part["jac"], layout), to_instance_major(full["jac"], layout)
    if layout == cpl.COMPONENT_MAJOR:
        assert (a[:, mask] == -9.5).all()          # whole rows of constant slots are never transferred
    assert same_bits(a[:, ~mask], b[:, ~mask]) and same_bits(part["g"], full["g"])
    prob.FillJacobianConstants(jac, layout=layout)
    assert same_bits(jac, full["jac"])


@pytest.mark.parametrize("case,N", [("ground4", 65536), ("superquadric4", 65536), ("ground8", 1 << 20)])
def test_full_size_configs(case, N, cuda_device):
    """BASELINE.json configs 2-4 at full size.  The oracle checks a strided sample; the two kernels (different
    code paths: thread-per-instance vs warp tiles + bulk copies) must agree bit for bit on every instance;
    and the statics rows obey their closed-form identities for all N."""
    import torch

    prob, o, gen = make_pair(case, rich=False)
    x = gen(N)
    xd = torch.from_numpy(x).to(cuda_device)
    a = prob.eval(xd, g=True, jac=True, layout=cpl.INSTANCE_MAJOR)
    b = prob.eval(xd.t().contiguous(), g=True, jac=True, layout=cpl.COMPONENT_MAJOR)
    torch.cuda.synchronize()
    for k in ("g", "jac"):
        assert torch.equal(a[k].view(torch.int64), b[k].t().contiguous().view(torch.int64)), f"{case}: {k} differs between kernels"
    sub = np.arange(0, N, max(1, N // 2048))
    want = o.eval_batch(x[sub], want=("g", "jac"), nthreads=4)
    got = {"g": a["g"][torch.from_numpy(sub).to(cuda_device)].cpu().numpy(),
           "jac": a["jac"][torch.from_numpy(sub).to(cuda_device)].cpu().numpy()}
    assert_parity(got, want, o, f"{case}/full")  # no x: the plain 1e-12 bar, no expanded-square allowance, on the benchmark configs
    assert assert_parity(got, want, o, f"{case}/full", x[sub]) == 0   # ... and offering the allowance changes nothing: no entry needs it
    # size-independent property: the force-balance Jacobian rows are all 1.0 and row r of g equals
    # Sigma_k F_k[r] - w[r] + m g[r] up to summation-order rounding
    nc = o.nc
    jac = a["jac"]
    assert bool((jac[:, : 3 * nc] == 1.0).all())
    F = xd[:, 3:].reshape(N, nc, 9)[:, :, 0:3].sum(dim=1)
    w = torch.tensor(synthetic.TESTBASIC["wrench"][:3], device=cuda_device, dtype=torch.float64)
    mg = torch.tensor([0.0, 0.0, -981.0], device=cuda_device, dtype=torch.float64)
    assert float((a["g"][:, :3] - (F - w + mg)).abs().max()) <= 1e-9


@pytest.mark.parametrize("layout", LAYOUTS)
def test_asynchronous_host_calls_queue_of_batches(layout, cuda_device):
    """cplb_eval_host_begin / _wait: three batches in flight on two buffer sets (begin k+1, wait k); every batch's outputs
    equal the synchronous call's bit for bit; pageable buffers are refused; an empty call completes at once."""
    import ctypes as C

    from centroidalplanner_b200 import _cabi

    prob, o, gen = make_pair("ground4")
    lib = _cabi.load()
    N = 40000          # three chunks, the last one ragged
    shape = (lambda L: (N, L)) if layout == cpl.INSTANCE_MAJOR else (lambda L: (L, N))

    def pinned(shp):
        ptr = C.c_void_p()
        assert lib.cplb_host_alloc(int(np.prod(shp)) * 8, C.byref(ptr)) == 0
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_double)), shape=(int(np.prod(shp)),)).reshape(shp), ptr

    keep, sets = [], []
    for _ in range(2):
        bufs = {}
        for key, L in (("x", prob.n), ("g", prob.m), ("jac", prob.nnz)):
            bufs[key], ptr = pinned(shape(L))
            keep.append(ptr)
        sets.append(bufs)
    batches = [gen(N) * (1.0 + 0.01 * b) for b in range(3)]
    want = [prob.eval(np.ascontiguousarray(xb if layout == cpl.INSTANCE_MAJOR else xb.T), g=True, jac=True, layout=layout) for xb in batches]
    got, pending = [], None
    for b, xb in enumerate(batches):
        bufs = sets[b % 2]
        bufs["x"][...] = xb if layout == cpl.INSTANCE_MAJOR else xb.T
        bufs["g"][...] = np.nan
        bufs["jac"][...] = np.nan
        ticket, _ = prob.eval_host_begin(bufs["x"], {"g": bufs["g"], "jac": bufs["jac"]}, g=True, jac=True, layout=layout)
        if pending is not None:
            prob.eval_host_wait(pending[0])
            got.append({k: pending[1][k].copy() for k in ("g", "jac")})
        pending = (ticket, bufs)
    prob.eval_host_wait(pending[0])
    got.append({k: pending[1][k].copy() for k in ("g", "jac")})
    for b in range(3):
        assert same_bits(got[b]["g"], want[b]["g"]) and same_bits(got[b]["jac"], want[b]["jac"]), b
    with pytest.raises(ValueError, match="pinned"):
        prob.eval_host_begin(np.zeros(shape(prob.n)), {"g": np.zeros(shape(prob.m))}, g=True, jac=False, layout=layout)
    with pytest.raises(ValueError, match="unknown ticket"):
        prob.eval_host_wait(17)
    for ptr in keep:
        lib.cplb_host_free(ptr)
