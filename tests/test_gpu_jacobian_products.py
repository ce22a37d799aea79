"""The fused Jacobian products (cplb_jacobian_products_device, csrc/cplb_products.cu) and the differentiable evaluation on the GPU.

The bit contract of include/cpl_batched.h is replayed literally: J and the gradient from cplb_eval_device at the same x (or from the
C oracle), then one multiply and one add per structural slot in slot order, written as separate ops (never addcmul, which may
contract to an FMA).  Every product must equal the replay bit for bit, NaN matched by position.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest
import torch

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic
from helpers import configure, make_pair, same_bits, set_oracle_instance

pytestmark = pytest.mark.gpu

F64 = torch.float64


def replay(iRow, jCol, jac, grad, lam=None, obj=None, v=None):
    """The contract in NumPy: (x_bar, g_dot, f_dot), None where not requested."""
    N, n = grad.shape
    m = int(iRow.max()) + 1
    x_bar = g_dot = f_dot = None
    with np.errstate(all="ignore"):
        if lam is not None or obj is not None:
            x_bar = np.multiply(obj[:, None], grad) if obj is not None else np.zeros((N, n))
            if lam is not None:
                for s in range(len(iRow)):
                    x_bar[:, jCol[s]] = np.add(x_bar[:, jCol[s]], np.multiply(jac[:, s], lam[:, iRow[s]]))
        if v is not None:
            g_dot = np.zeros((N, m))
            for s in range(len(iRow)):
                g_dot[:, iRow[s]] = np.add(g_dot[:, iRow[s]], np.multiply(jac[:, s], v[:, jCol[s]]))
            f_dot = np.zeros(N)
            for c in range(n):
                f_dot = np.add(f_dot, np.multiply(grad[:, c], v[:, c]))
    return x_bar, g_dot, f_dot


def replay_torch(iRow, jCol, jac, grad, lam, obj, v):
    """The same contract in torch on the device (the full-size cases), torch.mul and torch.add only."""
    N, n = grad.shape
    m = int(iRow.max()) + 1
    x_bar = torch.mul(obj[:, None], grad)
    g_dot = torch.zeros(N, m, dtype=F64, device=grad.device)
    for s in range(len(iRow)):
        r, c = int(iRow[s]), int(jCol[s])
        x_bar[:, c] = torch.add(x_bar[:, c], torch.mul(jac[:, s], lam[:, r]))
        g_dot[:, r] = torch.add(g_dot[:, r], torch.mul(jac[:, s], v[:, c]))
    f_dot = torch.zeros(N, dtype=F64, device=grad.device)
    for c in range(n):
        f_dot = torch.add(f_dot, torch.mul(grad[:, c], v[:, c]))
    return x_bar, g_dot, f_dot


def replay_eval(prob, x, lam=None, obj=None, v=None, per_instance=None):
    """The materialising caller: cplb_eval_device's J and gradient at x, multiplied on the host."""
    ev = prob.eval(x, g=False, jac=True, cost=False, grad=True, per_instance=per_instance)
    iRow, jCol = prob.GetJacobianStructure()
    np_ = lambda t: None if t is None else t.cpu().numpy()  # noqa: E731
    return replay(iRow, jCol, np_(ev["jac"]), np_(ev["grad"]), np_(lam), np_(obj), np_(v))


def assert_products(got, want, what):
    for key, w in zip(("x_bar", "g_dot", "f_dot"), want):
        if w is None:
            assert key not in got, (what, key)
            continue
        a = got[key].cpu().numpy()
        assert a.shape == w.shape, (what, key, a.shape, w.shape)
        if not same_bits(a, w):
            bad = np.argwhere(~((a == w) | (np.isnan(a) & np.isnan(w))))
            raise AssertionError(f"{what}: {key} differs first at {tuple(bad[0])}: got {a[tuple(bad[0])]!r}, want {w[tuple(bad[0])]!r}")


def _problem(nc, env_name, seed):
    names = ["k%02d" % ((7 * i) % nc) for i in range(nc)]       # vector order != sorted order
    env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[env_name]
    env = env() if env is not None else None
    prob = cpl.BatchedCplProblem(names, 100.0, env)
    configure(prob, env, names, env_name)
    gen = synthetic.superquadric_batch if env_name == "superquadric" else synthetic.ground_batch
    return prob, lambda N: gen(N, nc, seed)


def case_problem(case):
    if case in ("ground32", "noenv32"):
        return _problem(32, {"ground32": "ground", "noenv32": "none"}[case], 51)
    prob, _, gen = make_pair(case)
    return prob, gen


def per_instance_arrays(names, N, rng, device, env_kind):
    nc = len(names)
    arrs = dict(mass=rng.uniform(60.0, 140.0, N), wrench=rng.normal(0.0, 20.0, (N, 6)), mu=rng.uniform(0.3, 0.9, N),
                force_threshold=rng.uniform(0.0, 30.0, (N, nc)), ground_z=rng.uniform(-0.1, 0.2, N), com_ref=rng.normal(0.0, 0.3, (N, 3)),
                com_weight=rng.uniform(0.5, 3.0, N), pos_ref=rng.normal(0.0, 0.3, (N, 3 * nc)), force_ref=rng.normal(0.0, 50.0, (N, 3 * nc)),
                pos_weight=rng.uniform(0.0, 2.0, (N, nc)), force_weight=rng.uniform(0.0, 0.01, (N, nc)))
    assert set(arrs) == {name for name, _, _ in _cabi.INSTANCE_PARAMS}
    if env_kind != _cabi.ENV_GROUND:
        del arrs["ground_z"]
    return arrs, {k: torch.as_tensor(np.ascontiguousarray(a), device=device) for k, a in arrs.items()}


def factors(prob, N, seed, device):
    g = torch.Generator(device="cpu").manual_seed(seed)
    lam = torch.randn(N, prob.m, dtype=F64, generator=g).to(device)
    obj = torch.rand(N, dtype=F64, generator=g).to(device) * 2.0 - 0.5
    v = torch.randn(N, prob.n, dtype=F64, generator=g).to(device)
    return lam, obj, v


CASES = ["ground1", "noenv2", "ground4", "noenv4", "superquadric3", "superquadric4", "superquadric4_fracP_nan", "ground8", "noenv8",
         "superquadric8", "ground32", "noenv32", "superquadric32"]


@pytest.mark.parametrize("per_instance", [False, True], ids=["shared", "per_instance"])
@pytest.mark.parametrize("N", [1, 31, 33, 4096])
@pytest.mark.parametrize("case", CASES)
def test_bit_for_bit_against_the_replay_over_cplb_eval_device(case, N, per_instance, cuda_device):
    """Every environment, 1 to 32 contacts (sorted order != vector order), both parameter sources, partial and several tiles."""
    prob, gen = case_problem(case)
    x = torch.as_tensor(gen(N), device=cuda_device)
    lam, obj, v = factors(prob, N, 7 + N, cuda_device)
    pi = per_instance_arrays(prob.contact_names, N, np.random.default_rng(N), cuda_device, prob._env_kind)[1] if per_instance else None
    got = prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v, per_instance=pi)
    assert_products(got, replay_eval(prob, x, lam, obj, v, pi), f"{case} N={N}")


@pytest.mark.parametrize("case", ["ground1", "noenv2", "ground4", "noenv4", "ground8", "noenv8"])
def test_bit_for_bit_against_the_replay_over_the_oracle(case, cuda_device):
    """Ground and no environment (no pow() upstream): the replay over the C oracle's J and gradient, with shared parameters and
    with every per-instance array (one oracle per instance)."""
    prob, o, gen = make_pair(case)
    N = 48
    xs = gen(N)
    x = torch.as_tensor(xs, device=cuda_device)
    lam, obj, v = factors(prob, N, 3, cuda_device)
    iRow, jCol = o.structure()
    ev = o.eval_batch(xs, want=("jac", "grad"), nthreads=8)
    want = replay(iRow, jCol, ev["jac"], ev["grad"], lam.cpu().numpy(), obj.cpu().numpy(), v.cpu().numpy())
    assert_products(prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v), want, case)

    arrs, pi = per_instance_arrays(prob.contact_names, N, np.random.default_rng(4), cuda_device, prob._env_kind)
    jac, grad = np.empty((N, o.nnz)), np.empty((N, o.n))
    for i in range(N):
        oi = make_pair(case)[1]
        set_oracle_instance(oi, arrs, i)
        e = oi.eval_batch(xs[i:i + 1], want=("jac", "grad"))
        jac[i], grad[i] = e["jac"][0], e["grad"][0]
    want = replay(iRow, jCol, jac, grad, lam.cpu().numpy(), obj.cpu().numpy(), v.cpu().numpy())
    assert_products(prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v, per_instance=pi), want, case + " per-instance")


@pytest.mark.parametrize("case", ["ground4", "noenv4", "superquadric4"])
def test_inf_and_nan_in_the_factors_propagate_like_the_replay(case, cuda_device):
    """Inf and NaN in lambda and v: through Ground's structural zeros 0 * Inf is NaN, exactly as for the materialising caller."""
    prob, gen = case_problem(case)
    N = 64
    x = torch.as_tensor(gen(N), device=cuda_device)
    lam, obj, v = factors(prob, N, 5, cuda_device)
    rows = torch.arange(N, device=cuda_device)
    inf, nan = (torch.full((N,), val, dtype=F64, device=cuda_device) for val in (float("inf"), float("nan")))
    lam[rows, rows % prob.m] = torch.where(rows % 3 == 0, nan, torch.where(rows % 3 == 1, inf, -inf))
    v[rows, (5 * rows) % prob.n] = torch.where(rows % 2 == 0, inf, nan)
    obj[::7] = float("inf")
    got = prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v)
    assert_products(got, replay_eval(prob, x, lam, obj, v), case)
    if case == "ground4":   # an Inf multiplier of an EnvironmentNormal row meets the row's structural zeros at the p columns
        lam2 = torch.zeros(1, prob.m, dtype=F64, device=cuda_device)
        row = prob.GetContactRow(prob.contact_names[0]) + 1
        lam2[0, row] = float("inf")
        xb = prob.JacobianProducts(x[:1].contiguous(), lam=lam2)["x_bar"][0]
        pcol = prob.GetBlockColumn(cpl.BLOCK_POSITION, prob.contact_names[0])
        assert torch.isnan(xb[pcol:pcol + 3]).all()


def test_zero_tangential_force_nan_propagates(cuda_device):
    """F_t = 0 exactly: the FrictionCone Jacobian holds 0/0 = NaN (SURVEY Q3); the products carry it where the replay does."""
    prob = cpl.BatchedCplProblem(["contact1"], 100.0, cpl.Ground())
    x = torch.as_tensor([[0.0, 0.0, 1.0, 0.0, 0.0, 100.0, 0.0, 0.0, 0.0, 0.0, 0.0, 1.0]], dtype=F64, device=cuda_device)
    lam, obj, v = factors(prob, 1, 9, cuda_device)
    got = prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v)
    assert_products(got, replay_eval(prob, x, lam, obj, v), "F_t = 0")
    assert torch.isnan(got["x_bar"]).any() and torch.isnan(got["g_dot"]).any() and not torch.isnan(got["f_dot"]).any()


COMBOS = [("lambda_",), ("obj_factor",), ("lambda_", "obj_factor"), ("v", "g_dot"), ("v", "f_dot"), ("v", "g_dot", "f_dot"),
          ("lambda_", "v", "g_dot"), ("obj_factor", "v", "f_dot"), ("lambda_", "obj_factor", "v", "g_dot", "f_dot")]


@pytest.mark.parametrize("combo", COMBOS, ids=["+".join(c) for c in COMBOS])
def test_each_null_combination_writes_only_its_outputs(combo, cuda_device):
    """Sentinel-filled output buffers with guard bands on both sides: the requested outputs equal the replay with the same NULLs, the
    others and every guard band keep the sentinel."""
    prob, gen = case_problem("ground8")
    N, G = 37, 64
    x = torch.as_tensor(gen(N), device=cuda_device)
    lam, obj, v = factors(prob, N, 11, cuda_device)
    sentinel = -1.2345e300
    size = {"x_bar": N * prob.n, "g_dot": N * prob.m, "f_dot": N}
    bufs = {k: torch.full((L + 2 * G,), sentinel, dtype=F64, device=cuda_device) for k, L in size.items()}
    want_xbar = "lambda_" in combo or "obj_factor" in combo
    args = _cabi.JacobianProductsArgs(N, x.data_ptr(), None, lam.data_ptr() if "lambda_" in combo else None,
                                      obj.data_ptr() if "obj_factor" in combo else None, bufs["x_bar"][G:].data_ptr() if want_xbar else None,
                                      v.data_ptr() if "v" in combo else None, bufs["g_dot"][G:].data_ptr() if "g_dot" in combo else None,
                                      bufs["f_dot"][G:].data_ptr() if "f_dot" in combo else None)
    assert _cabi.load().cplb_jacobian_products_device(prob._h, C.byref(args), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == _cabi.OK
    want = replay_eval(prob, x, lam if "lambda_" in combo else None, obj if "obj_factor" in combo else None, v if "v" in combo else None)
    for key, w in zip(("x_bar", "g_dot", "f_dot"), want):
        b = bufs[key].cpu().numpy()
        requested = want_xbar if key == "x_bar" else key in combo
        assert (b[:G] == sentinel).all() and (b[G + size[key]:] == sentinel).all(), (combo, key, "guard band")
        if requested:
            assert same_bits(b[G:G + size[key]].reshape(w.shape), w), (combo, key)
        else:
            assert (b[G:G + size[key]] == sentinel).all(), (combo, key, "written although not requested")


@pytest.mark.parametrize("nc,env_name,N", [(4, "ground", 1 << 20), (8, "superquadric", 65536)])
def test_full_size_against_the_replay_on_the_device(nc, env_name, N, cuda_device):
    prob, _ = _problem(nc, env_name, 61)
    gen = synthetic.superquadric_batch if env_name == "superquadric" else synthetic.ground_batch
    x = torch.as_tensor(gen(N, nc, 61), device=cuda_device)
    lam, obj, v = factors(prob, N, 13, cuda_device)
    got = prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v)
    ev = prob.eval(x, g=False, jac=True, cost=False, grad=True)
    iRow, jCol = prob.GetJacobianStructure()
    want = replay_torch(iRow, jCol, ev["jac"], ev["grad"], lam, obj, v)
    for key, w in zip(("x_bar", "g_dot", "f_dot"), want):
        a = got[key]
        same = (a.view(torch.int64) == w.view(torch.int64)) | (a.isnan() & w.isnan())
        assert bool(same.all()), (key, int((~same).sum()))


def test_two_streams_run_concurrently(cuda_device):
    """The call enqueues and returns; calls on two streams give the results of two calls in series and count one launch each."""
    prob, gen = case_problem("ground8")
    xa = torch.as_tensor(gen(4096), device=cuda_device)
    xb = torch.as_tensor(synthetic.ground_batch(4096, 8, 99), device=cuda_device)
    fa, fb = factors(prob, 4096, 1, cuda_device), factors(prob, 4096, 2, cuda_device)
    kw = lambda f: dict(lam=f[0], obj_factor=f[1], v=f[2])  # noqa: E731
    serial_a, serial_b = prob.JacobianProducts(xa, **kw(fa)), prob.JacobianProducts(xb, **kw(fb))
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    launches = prob.launch_count()
    with torch.cuda.stream(s1):
        torch.cuda._sleep(200_000_000)
        ra = prob.JacobianProducts(xa, **kw(fa))
        returned_before_done = not s1.query()
    with torch.cuda.stream(s2):
        rb = prob.JacobianProducts(xb, **kw(fb))
    assert returned_before_done
    torch.cuda.synchronize()
    assert prob.launch_count() == launches + 2
    for k in ("x_bar", "g_dot", "f_dot"):
        assert same_bits(ra[k].cpu().numpy(), serial_a[k].cpu().numpy()) and same_bits(rb[k].cpu().numpy(), serial_b[k].cpu().numpy()), k


def test_pybind_and_ctypes_return_the_same_bits(cuda_device):
    # imported as the top-level `pycplb`, the name every pybind test uses, so that the extension is loaded once per session
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
    N = 100
    x = torch.as_tensor(synthetic.ground_batch(N, 4, 3), device=cuda_device)
    lam, obj, v = factors(prob, N, 17, cuda_device)
    want = prob.JacobianProducts(x, lam=lam, obj_factor=obj, v=v)
    out = dict(x_bar=torch.empty(N, pp.n, dtype=F64, device=cuda_device), g_dot=torch.empty(N, pp.m, dtype=F64, device=cuda_device),
               f_dot=torch.empty(N, dtype=F64, device=cuda_device))
    pp.jacobian_products_device(N, x.data_ptr(), lam=lam.data_ptr(), obj_factor=obj.data_ptr(), v=v.data_ptr(),
                                **{k: t.data_ptr() for k, t in out.items()}, stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for k in out:
        assert same_bits(out[k].cpu().numpy(), want[k].cpu().numpy()), k


# ---- autodiff -------------------------------------------------------------------------------------------------------------------

def _smooth_points(prob, N, seed, device):
    """Points away from the friction-cone kink: tangential forces well away from zero, unit-ish normals."""
    rng = np.random.default_rng(seed)
    nc = len(prob.contact_names)
    x = np.empty((N, prob.n))
    x[:, :3] = rng.normal([0.0, 0.0, 1.0], 0.05, (N, 3))
    for k in range(nc):
        b = 3 + 9 * k
        x[:, b:b + 3] = rng.normal([8.0, -5.0, 60.0], 1.0, (N, 3))
        x[:, b + 3:b + 6] = rng.normal([0.3 * (-1) ** k, 0.2, 0.05], 0.05, (N, 3))
        x[:, b + 6:b + 9] = rng.normal([0.1, 0.05, 1.0], 0.02, (N, 3))
    return torch.as_tensor(x, device=device)


@pytest.mark.parametrize("case", ["ground1", "noenv2", "superquadric_2"])
@pytest.mark.parametrize("per_instance", [False, True], ids=["shared", "per_instance"])
def test_gradcheck_reverse_and_forward(case, per_instance, cuda_device):
    if case == "superquadric_2":
        prob, _ = _problem(2, "superquadric", 3)
    else:
        prob, _ = case_problem(case)
    N = 2
    x = _smooth_points(prob, N, 1, cuda_device).requires_grad_(True)
    pi = per_instance_arrays(prob.contact_names, N, np.random.default_rng(8), cuda_device, prob._env_kind)[1] if per_instance else None
    fn = lambda xx: cpl.constraints_and_cost(prob, xx, per_instance=pi)  # noqa: E731
    assert torch.autograd.gradcheck(fn, (x,), eps=1e-6, atol=1e-5, rtol=1e-4)
    assert torch.autograd.gradcheck(fn, (x,), eps=1e-6, atol=1e-5, rtol=1e-4, check_forward_ad=True, check_backward_ad=False,
                                    check_undefined_grad=False)


def test_backward_equals_the_reverse_product(cuda_device):
    prob, gen = case_problem("ground4")
    x = torch.as_tensor(gen(256), device=cuda_device).requires_grad_(True)
    g, cost = cpl.constraints_and_cost(prob, x)
    (g.sum() + cost.sum()).backward()
    N = x.shape[0]
    want = prob.JacobianProducts(x.detach(), lam=torch.ones(N, prob.m, dtype=F64, device=cuda_device),
                                 obj_factor=torch.ones(N, dtype=F64, device=cuda_device))["x_bar"]
    assert torch.equal(x.grad.view(torch.int64), want.view(torch.int64))
    # forward mode through torch.func: one forward product
    v = torch.randn(N, prob.n, dtype=F64, device=cuda_device)
    (g2, c2), (gd, fd) = torch.func.jvp(lambda xx: cpl.constraints_and_cost(prob, xx), (x.detach(),), (v,))
    ref = prob.JacobianProducts(x.detach(), v=v)
    assert torch.equal(gd.view(torch.int64), ref["g_dot"].view(torch.int64)) and torch.equal(fd.view(torch.int64), ref["f_dot"].view(torch.int64))
    assert torch.equal(g2, g.detach()) and torch.equal(c2, cost.detach())


def test_double_backward_raises(cuda_device):
    """A backward pass whose result would itself be differentiated (here through the cotangent w) raises on the second pass."""
    prob, gen = case_problem("ground1")
    x = torch.as_tensor(gen(4), device=cuda_device).requires_grad_(True)
    g, cost = cpl.constraints_and_cost(prob, x)
    w = torch.ones(4, dtype=F64, device=cuda_device, requires_grad=True)
    (gx,) = torch.autograd.grad(cost, x, grad_outputs=w, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        gx.sum().backward()


def test_per_instance_requires_grad_raises(cuda_device):
    prob, gen = case_problem("ground1")
    x = torch.as_tensor(gen(4), device=cuda_device).requires_grad_(True)
    mu = torch.full((4,), 0.5, dtype=F64, device=cuda_device, requires_grad=True)
    with pytest.raises(ValueError, match="requires grad"):
        cpl.constraints_and_cost(prob, x, per_instance={"mu": mu})
