"""Every dispatch target of the component-major launcher against the oracle.

`launch_cm_env` (csrc/cplb_kernels_cm.cuh) picks between two kernels by (contact count, batch size): one thread per
(instance, contact) and -- for shared-parameter 4- and 8-contact batches from a measured crossover on -- one thread per
instance.  Both are product code, so both are forced here (cplb_set_component_major_kernel) on the same inputs, for every
environment kind, both contact counts, every output subset, at the crossover, one below it and well above it, and must

  * agree bit for bit with the instance-major kernel (a third, independent code path) on EVERY instance, and
  * agree with the CPU oracle on a strided sample (bit-exact where no pow() is upstream, <= 1e-12 relative elsewhere).

Reference arithmetic these kernels restate: CentroidalStatics.cpp:44-57 (values), :121-135 (CoM block),
MinimizeCentroidalVariables.cpp:126-147 (cost), :163-191 (gradient)."""
import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi

from helpers import CASES as ALL_CASES
from helpers import assert_parity, make_pair, set_oracle_instance

pytestmark = pytest.mark.gpu

CROSSOVER = {4: 90112, 8: 49152}  # launch_cm_env: whole_from
SUBSETS = [dict(g=True, jac=True), dict(g=True, jac=True, cost=True, grad=True), dict(g=True, jac=False), dict(g=False, jac=True),
           dict(g=False, jac=False, cost=True), dict(g=False, jac=False, grad=True)]
CASES = [("noenv4", 4), ("ground4", 4), ("superquadric4", 4), ("noenv8", 8), ("ground8", 8), ("superquadric8", 8)]


def _sizes(nc):
    return [CROSSOVER[nc] - 1, CROSSOVER[nc], 131072, 1 << 20]


@pytest.mark.parametrize("which", ["crossover-1", "crossover", "131072", "1048576"])
@pytest.mark.parametrize("case,nc", CASES)
def test_both_component_major_kernels_match_oracle_and_instance_major(case, nc, which, cuda_device):
    import torch

    N = dict(zip(["crossover-1", "crossover", "131072", "1048576"], _sizes(nc)))[which]
    prob, o, gen = make_pair(case)  # rich parameters: distinct refs / weights / thresholds per contact
    x = gen(N)
    xd = torch.from_numpy(x).to(cuda_device)
    xt = xd.t().contiguous()
    ref = prob.eval(xd, g=True, jac=True, cost=True, grad=True, layout=cpl.INSTANCE_MAJOR)  # every instance
    torch.cuda.synchronize()
    sub = np.unique(np.concatenate([np.arange(0, N, max(1, N // 1024)), [N - 1, N - 2, N - 33]]))
    want = o.eval_batch(x[sub], nthreads=4)
    subd = torch.from_numpy(sub).to(cuda_device)
    # the instance-major kernel itself against the oracle on the sample (it is the all-instance yardstick below)
    assert_parity({k: ref[k][subd].cpu().numpy() for k in ref}, want, o, f"{case}/N{N}/instance-major", x[sub])

    for kernel in ("split", "whole"):
        prob.SetComponentMajorKernel(kernel)
        for want_flags in SUBSETS:
            launches = prob.launch_count()
            out = prob.eval(xt, layout=cpl.COMPONENT_MAJOR, **want_flags)
            torch.cuda.synchronize()
            assert prob.launch_count() == launches + 1
            tag = f"{case}/N{N}/{kernel}/{'+'.join(k for k in want_flags if want_flags[k])}"
            got = {}
            for k in ("g", "jac", "cost", "grad"):
                if not want_flags.get(k, False):
                    assert out[k] is None, tag
                    continue
                a = out[k] if k == "cost" else out[k].t().contiguous()
                assert torch.equal(a.view(torch.int64), ref[k].view(torch.int64)), f"{tag}: {k} differs from the instance-major kernel"
                got[k] = a[subd].cpu().numpy()
                del a
            assert_parity(got, {k: (want[k] if k in got else None) for k in want}, o, tag, x[sub])
            del out
    prob.SetComponentMajorKernel("auto")


@pytest.mark.parametrize("case", ["ground4", "ground8"])
def test_forced_whole_with_per_instance_parameters_stays_on_the_per_contact_kernel(case, cuda_device):
    """Per-instance parameter arrays exist only in the per-contact kernel; a forced PER_INSTANCE choice must not drop them."""
    import torch

    prob, o, gen = make_pair(case)
    N = 2000
    x = gen(N)
    rng = np.random.default_rng(3)
    wrench = rng.uniform(-50, 50, (N, 6))
    prob.SetComponentMajorKernel("whole")
    out = prob.eval(torch.from_numpy(np.ascontiguousarray(x.T)).to(cuda_device), g=True, jac=False, layout=cpl.COMPONENT_MAJOR,
                    per_instance={"wrench": torch.from_numpy(np.ascontiguousarray(wrench.T)).to(cuda_device)})
    torch.cuda.synchronize()
    g = out["g"].t().cpu().numpy()
    for i in (0, 1, N - 1):
        o.set_wrench(wrench[i])
        assert np.array_equal(g[i], o.eval(x[i], want=("g",))["g"])


def test_two_threads_with_different_output_subsets_share_one_kernel_instantiation(cuda_device):
    """The instance-major launcher raises a kernel's opt-in shared-memory limit per (kernel, device) and never lowers it:
    a thread asking for the Jacobian only (64 KB of tiles per CTA) and a thread asking for the constraint values only
    (27 KB) use the SAME kernel instantiation; a limit lowered by the second would make the first one's next launch fail."""
    import threading

    import torch

    prob, o, gen = make_pair("ground4")
    N = 8192
    x = gen(N)
    xd = torch.from_numpy(x).to(cuda_device)
    ref = prob.eval(xd, g=True, jac=True, layout=cpl.INSTANCE_MAJOR)
    torch.cuda.synchronize()
    errors, results = [], {}

    def work(key):
        try:
            st = torch.cuda.Stream(cuda_device)
            with torch.cuda.stream(st):
                for _ in range(200):
                    out = prob.eval(xd, g=(key == "g"), jac=(key == "jac"), layout=cpl.INSTANCE_MAJOR, stream=st.cuda_stream)
                st.synchronize()
            results[key] = out[key]
        except Exception as e:  # noqa: BLE001
            errors.append((key, e))

    th = [threading.Thread(target=work, args=(k,)) for k in ("jac", "g", "jac", "g")]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    for k in ("g", "jac"):
        assert torch.equal(results[k].view(torch.int64), ref[k].view(torch.int64))


# ---- the two instance-major kernels (cplb_set_instance_major_kernel) -------------------------------------------------------

IM_KERNELS = ["warp", "cta"]


def _eval_im(prob, xd, **want):
    import torch

    out = prob.eval(xd, layout=cpl.INSTANCE_MAJOR, **want)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("kernel", IM_KERNELS)
@pytest.mark.parametrize("case", sorted(ALL_CASES))
def test_instance_major_kernels_every_shape_ragged_sizes_and_subsets(case, kernel, cuda_device):
    """Both instance-major kernels, every problem shape of the suite (1..32 contacts, all environment kinds, permuted names,
    fractional curvatures), ragged batch sizes around the tile sizes, every output subset: against the oracle."""
    import torch

    prob, o, gen = make_pair(case)
    prob.SetInstanceMajorKernel(kernel)
    for N in (1, 3, 4, 5, 15, 16, 17, 31, 32, 33, 63, 65, 129, 1000):
        x = gen(N)
        want = o.eval_batch(x, nthreads=4)
        xd = torch.from_numpy(x).to(cuda_device)
        for flags in SUBSETS:
            if N > 33 and flags is not SUBSETS[1]:
                continue
            out = _eval_im(prob, xd, **flags)
            got = {k: (None if v is None else v.cpu().numpy()) for k, v in out.items()}
            assert_parity(got, {k: (want[k] if flags.get(k, False) else None) for k in want}, o,
                          f"{case}/N{N}/{kernel}/{'+'.join(k for k in flags if flags[k])}", x)


@pytest.mark.parametrize("kernel", IM_KERNELS)
@pytest.mark.parametrize("case,N", [("ground4", 65536), ("superquadric4", 65536), ("noenv4", 65536), ("ground8", 1 << 20), ("noenv8", 200001),
                                    ("superquadric8", 100003), ("ground1", 70001), ("ground12", 30011), ("superquadric32", 5003)])
def test_instance_major_kernels_agree_on_every_instance(case, N, kernel, cuda_device):
    """Full-size batches: the forced kernel against the component-major per-contact kernel on EVERY instance (bit for bit) and
    against the oracle on a strided sample; all four outputs."""
    import torch

    prob, o, gen = make_pair(case)
    x = gen(N)
    xd = torch.from_numpy(x).to(cuda_device)
    prob.SetComponentMajorKernel("split")
    ref = prob.eval(xd.t().contiguous(), g=True, jac=True, cost=True, grad=True, layout=cpl.COMPONENT_MAJOR)
    prob.SetInstanceMajorKernel(kernel)
    out = _eval_im(prob, xd, g=True, jac=True, cost=True, grad=True)
    for key in ("g", "jac", "cost", "grad"):
        a = ref[key] if key == "cost" else ref[key].t().contiguous()
        assert torch.equal(a.view(torch.int64), out[key].view(torch.int64)), f"{case}/{kernel}: {key} differs from the component-major kernel"
    sub = np.unique(np.concatenate([np.arange(0, N, max(1, N // 512)), [N - 1, N - 2]]))
    subd = torch.from_numpy(sub).to(cuda_device)
    assert_parity({key: out[key][subd].cpu().numpy() for key in out}, o.eval_batch(x[sub], nthreads=4), o, f"{case}/N{N}/{kernel}", x[sub])


@pytest.mark.parametrize("kernel", IM_KERNELS)
@pytest.mark.parametrize("case", ["ground4", "noenv8", "superquadric3", "ground12"])
def test_instance_major_kernels_misaligned_buffers_and_guard_bands(case, kernel, cuda_device):
    """8-byte-aligned (not 16) buffers take the plain-copy tile path; sentinel bands around every buffer must survive."""
    import torch

    prob, o, gen = make_pair(case)
    prob.SetInstanceMajorKernel(kernel)
    SENT = -3.5e66
    for N, off in ((37, 1), (37, 0), (1000, 1), (4099, 1)):
        x = gen(N)
        want = o.eval_batch(x, nthreads=4)
        G = 64 + off

        def make(count):
            full = torch.full((count + 2 * G,), SENT, dtype=torch.float64, device=cuda_device)
            return full, full[G:G + count]

        bufs = {key: make(N * L) for key, L in (("g", o.m), ("jac", o.nnz), ("grad", o.n), ("cost", 1))}
        xfull, xin = make(N * o.n)
        xin.copy_(torch.from_numpy(x).reshape(-1))
        out = {key: (v[1].view(N, -1) if key != "cost" else v[1]) for key, v in bufs.items()}
        if off:
            assert xin.data_ptr() % 16 == 8
        prob.eval(xin.view(N, o.n), g=True, jac=True, cost=True, grad=True, layout=cpl.INSTANCE_MAJOR, out=out)
        torch.cuda.synchronize()
        for key, (full, _) in bufs.items():
            assert bool((full[:G] == SENT).all()) and bool((full[-G:] == SENT).all()), f"{case}/{kernel}/{key}: guard band overwritten"
        assert bool((xfull[:G] == SENT).all()) and bool((xfull[-G:] == SENT).all())
        assert_parity({key: out[key].cpu().numpy() for key in out}, want, o, f"guard/{case}/N{N}/{kernel}", x)


@pytest.mark.parametrize("kernel", IM_KERNELS)
@pytest.mark.parametrize("case", ["ground4", "noenv8", "superquadric3"])
def test_instance_major_kernels_per_instance_parameters(case, kernel, cuda_device):
    """cplb_instance_params through both instance-major kernels: N different CplProblems played by the oracle."""
    import torch

    prob, o, gen = make_pair(case)
    prob.SetInstanceMajorKernel(kernel)
    N, nc = 333, o.nc
    x = gen(N)
    rng = np.random.default_rng(7)
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
    pid = {key: torch.from_numpy(np.ascontiguousarray(v)).to(cuda_device) for key, v in pi.items()}
    xd = torch.from_numpy(x).to(cuda_device)
    for flags in (SUBSETS[1], SUBSETS[0], SUBSETS[2]):
        out = prob.eval(xd, layout=cpl.INSTANCE_MAJOR, per_instance=pid, **flags)
        torch.cuda.synchronize()
        got = {key: (None if v is None else v.cpu().numpy()) for key, v in out.items()}
        assert_parity(got, {key: (want[key] if flags.get(key, False) else None) for key in want}, o, f"per-instance/{case}/{kernel}", x)
