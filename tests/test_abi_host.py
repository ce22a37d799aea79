"""CPU tests of the product's host side: the C-ABI library loads and exports every declared
symbol, the layout generator agrees with the oracle's discovered structure, the setters keep the
reference's validation / error behaviour, and evaluation FAILS LOUDLY without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import centroidalplanner_b200 as cpl
from centroidalplanner_b200 import _cabi, synthetic
from oracle import cpl_oracle_py as orc

from helpers import CASES, make_pair

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_symbol_the_header_declares():
    hdr = open(os.path.join(ROOT, "include", "cpl_batched.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(cplb_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 40
    lib = C.CDLL(cpl.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(lib, name), f"libcplb.so does not export {name}"
    assert declared == set(_cabi.PROTOTYPES), declared ^ set(_cabi.PROTOTYPES)
    assert _cabi.load().cplb_abi_version() == 3


def test_instance_params_table_matches_the_header():
    """_cabi.INSTANCE_PARAMS (the ctypes struct and the length checks of the Python API) against cplb_instance_params in
    include/cpl_batched.h: the member names in order, and the per-instance length each member's comment states."""
    hdr = open(os.path.join(ROOT, "include", "cpl_batched.h")).read()
    body = re.search(r"typedef struct cplb_instance_params \{(.*?)\} cplb_instance_params;", hdr, flags=re.S).group(1)
    members = re.findall(r"const double \*(\w+);\s*/\*\s*(\S+)", body)
    assert len(members) == len(re.findall(r";", body))

    def length(text):  # "6" -> (6, 0), "nc" -> (0, 1), "3*nc" -> (0, 3)
        m = re.fullmatch(r"(\d+)|(?:(\d+)\*)?nc", text)
        assert m, text
        return (int(m.group(1)), 0) if m.group(1) else (0, int(m.group(2) or 1))

    assert tuple((name, *length(text)) for name, text in members) == _cabi.INSTANCE_PARAMS
    assert [f[0] for f in _cabi.InstanceParams._fields_] == [name for name, _ in members]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "centroidalplanner_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp", "Makefile")):
                src = open(os.path.join(dirpath, f), errors="replace").read()
                # no import / include / dlopen of anything under oracle/ (prose mentions are fine)
                assert not re.search(r"cpl_oracle|import\s+oracle|from\s+oracle|libcpl_ref|#include\s*[<\"].*oracle", src), \
                    os.path.join(dirpath, f)


@pytest.mark.parametrize("case", sorted(CASES))
def test_layout_matches_oracle_structure(case):
    prob, o, _ = make_pair(case)
    assert (prob.n, prob.m, prob.nnz) == (o.n, o.m, o.nnz)
    r, c = prob.GetJacobianStructure()
    ro, co = o.structure()
    assert np.array_equal(r, ro) and np.array_equal(c, co)  # identical triplet order
    assert np.array_equal(prob.GetSortedOrder(), o.sorted_order())
    lb, ub = prob.GetBoundsOnConstraints()
    lbo, ubo = o.con_bounds()
    assert np.array_equal(lb, lbo) and np.array_equal(ub, ubo)
    lb, ub = prob.GetBoundsOnOptimizationVariables()
    lbo, ubo = o.var_bounds()
    assert np.array_equal(lb, lbo) and np.array_equal(ub, ubo)


def test_layout_of_random_name_sets_matches_oracle_structure():
    """The closed-form layout (csrc/cplb_layout.hpp) against the structure the oracle DISCOVERS by emulating ifopt's assembly,
    for 60 random contact-name sets: 1..32 names with shared prefixes, digits, upper case and underscores (std::map orders
    them bytewise: 'Z' < '_' < 'a', 'c10' < 'c2'), in random vector order, every environment kind."""
    rng = np.random.default_rng(2024)
    alphabet = list("abcXYZ_019")
    for trial in range(60):
        nc = int(rng.integers(1, 33))
        names = set()
        while len(names) < nc:
            names.add("".join(rng.choice(alphabet, size=int(rng.integers(1, 6)))))
        names = list(names)
        rng.shuffle(names)
        kind = ["none", "ground", "superquadric"][trial % 3]
        env = {"none": None, "ground": cpl.Ground, "superquadric": cpl.Superquadric}[kind]
        prob = cpl.BatchedCplProblem(names, 50.0, env() if env else None)
        o = orc.Oracle(names, {"none": orc.ENV_NONE, "ground": orc.ENV_GROUND, "superquadric": orc.ENV_SUPERQUADRIC}[kind], 50.0)
        assert (prob.n, prob.m, prob.nnz) == (o.n, o.m, o.nnz), names
        r, c = prob.GetJacobianStructure()
        ro, co = o.structure()
        assert np.array_equal(r, ro) and np.array_equal(c, co), names
        assert np.array_equal(prob.GetSortedOrder(), o.sorted_order()), names
        assert [names[k] for k in prob.GetSortedOrder()] == sorted(names)            # bytewise, like std::string operator<
        for nm in names:
            j = sorted(names).index(nm)
            assert prob.GetContactRow(nm) == 6 + (6 if kind != "none" else 2) * j


@pytest.mark.parametrize("case", sorted(CASES))
def test_layout_matches_reference_golden_structure(case):
    """(iRow, jCol) and bounds as the reference's own CplProblem + ifopt-style assembly report them
    (tests/golden/ref_vectors.npz, tools/make_golden.py)."""
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_vectors.npz"))
    prob, _, _ = make_pair(case)
    r, c = prob.GetJacobianStructure()
    assert np.array_equal(r, z[f"{case}/iRow"]) and np.array_equal(c, z[f"{case}/jCol"])
    gl, gu = prob.GetBoundsOnConstraints()
    xl, xu = prob.GetBoundsOnOptimizationVariables()
    assert np.array_equal(gl, z[f"{case}/gl"]) and np.array_equal(gu, z[f"{case}/gu"])
    assert np.array_equal(xl, z[f"{case}/xl"]) and np.array_equal(xu, z[f"{case}/xu"])


@pytest.mark.parametrize("case", sorted(CASES))
def test_jacobian_constants_are_constant_in_the_oracle(case):
    """Every slot the product declares constant holds exactly that value for any x in the oracle (and the reference
    golden vectors); FillJacobianConstants writes exactly those slots in either layout."""
    prob, o, gen = make_pair(case)
    mask, val = prob.GetJacobianConstants()
    x = gen(200)
    jac = o.eval_batch(x, want=("jac",))["jac"]
    assert (jac[:, mask] == val[mask]).all()
    varying = (jac != jac[0]).any(axis=0) | np.isnan(jac).any(axis=0)
    assert not (varying & mask).any()
    if case.startswith("ground"):
        assert mask.sum() == 3 * o.nc + 15 * o.nc          # statics identities + Ground's constants
    elif case.startswith("noenv"):
        assert mask.sum() == 3 * o.nc
    else:
        assert mask.sum() == 3 * o.nc + 3 * o.nc           # statics identities + the n-block identity of EnvironmentNormal
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_vectors.npz"))
    assert (z[f"{case}/jac"][:, mask] == val[mask]).all()
    for layout in (cpl.INSTANCE_MAJOR, cpl.COMPONENT_MAJOR):
        buf = np.full((7, prob.nnz) if layout == cpl.INSTANCE_MAJOR else (prob.nnz, 7), -3.0)
        prob.FillJacobianConstants(buf, layout=layout)
        b = buf if layout == cpl.INSTANCE_MAJOR else buf.T
        assert (b[:, mask] == val[mask]).all() and (b[:, ~mask] == -3.0).all()


def test_block_columns_and_contact_rows():
    prob = cpl.BatchedCplProblem(["r_foot", "l_foot", "r_hand", "l_hand"], 100.0, cpl.Ground())
    assert prob.GetBlockColumn(cpl.BLOCK_COM) == 0
    assert prob.GetBlockColumn(cpl.BLOCK_FORCE, "l_foot") == 12
    assert prob.GetBlockColumn(cpl.BLOCK_POSITION, "l_foot") == 15
    assert prob.GetBlockColumn(cpl.BLOCK_NORMAL, "r_foot") == 9
    assert prob.GetContactRow("l_foot") == 6 and prob.GetContactRow("r_hand") == 24
    with pytest.raises(IndexError):
        prob.GetContactRow("nose")


def test_defaults_are_the_references():
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    assert prob.GetMu() == 1.0                                    # Environment.h:46
    assert list(prob.GetCoMRef()) == [0.0, 0.0, 1.0]              # MinimizeCentroidalVariables.cpp:11
    assert prob.GetCoMWeight() == 1.0
    assert list(prob.GetManipulationWrench()) == [0.0] * 6        # CentroidalStatics.cpp:12
    for nm in synthetic.NAMES4:
        assert prob.GetForceThreshold(nm) == 0.0                  # FrictionCone.cpp:14
        assert prob.GetContactPosWeight(nm) == 1.0 and prob.GetContactForceWeight(nm) == 1.0
        assert list(prob.GetPosRef(nm)) == [0, 0, 0] and list(prob.GetForceRef(nm)) == [0, 0, 0]
        lb, ub = prob.GetForceBounds(nm)
        assert list(lb) == [-1000.0] * 3 and list(ub) == [1000.0] * 3  # Variable3D.cpp:12-13
    sq = cpl.Superquadric()
    Cc, R, P = sq.GetParameters()
    assert list(Cc) == [0, 0, 10] and list(R) == [10, 10, 10] and list(P) == [10, 10, 10]  # Superquadric.cpp:7-9


def test_validation_mirrors_the_reference_exceptions():
    with pytest.raises(ValueError, match="Invalid robot mass"):      # CentroidalPlanner.cpp:12-15
        cpl.BatchedCplProblem(synthetic.NAMES4, 0.0, cpl.Ground())
    with pytest.raises(ValueError):
        cpl.BatchedCplProblem(["a", "a"], 1.0, cpl.Ground())
    with pytest.raises(ValueError):
        cpl.BatchedCplProblem([], 1.0, cpl.Ground())
    g = cpl.Ground()
    with pytest.raises(ValueError, match="Invalid friction coefficient"):  # Environment.h:21-22
        g.SetMu(0.0)
    sq = cpl.Superquadric()
    with pytest.raises(ValueError, match="axial radii"):             # Superquadric.cpp:16-19
        sq.SetParameters([0, 0, 1], [0.3, 0.0, 10], [10, 10, 10])
    with pytest.raises(ValueError, match="curvatures"):              # Superquadric.cpp:21-24
        sq.SetParameters([0, 0, 1], [0.3, 0.3, 10], [10, 1.9, 10])
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, g)
    with pytest.raises(IndexError):                                  # std::map::at, CplProblem.cpp:113
        prob.SetForceBounds("nose", [0, 0, 0], [1, 1, 1])
    with pytest.raises(IndexError):                                  # MinimizeCentroidalVariables.cpp:33
        prob.SetPosRef("nose", [0, 0, 0])
    with pytest.raises(ValueError, match="Inconsistent bounds"):     # Variable3D.cpp:35-38
        prob.SetPosBounds("contact1", [0, 0, 1], [1, 1, 0])
    lb, ub = prob.GetPosBounds("contact1")                           # ... stored before the throw (:31-32)
    assert list(lb) == [0, 0, 1] and list(ub) == [1, 1, 0]
    with pytest.raises(ValueError, match="Invalid weight"):          # CentroidalPlanner.cpp:186-189
        prob.SetCoMWeight(-1.0)
    with pytest.raises(ValueError, match="Invalid weight"):
        prob.SetContactForceWeight("contact2", -0.5)
    lib = _cabi.load()                                               # the C level, directly
    assert lib.cplb_set_mu(prob._h, -1.0) == _cabi.INVALID_ARGUMENT
    assert b"friction" in lib.cplb_last_error()
    assert lib.cplb_set_superquadric(prob._h, *(np.ones(3).ctypes.data_as(_cabi.dp),) * 3) == _cabi.RUNTIME_ERROR
    assert lib.cplb_get_dims(None, None, None, None) == _cabi.NULL_POINTER


def test_environment_object_is_shared_like_the_reference():
    """The reference's sets alias one env object (CplProblem.cpp:47-59): a later SetMu is seen."""
    g = cpl.Ground()
    a = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, g)
    b = cpl.BatchedCplProblem(["x", "y"], 50.0, g)
    g.SetMu(0.25)
    g.SetGroundZ(0.4)
    lib = _cabi.load()
    for prob in (a, b):
        mu, z = C.c_double(), C.c_double()
        assert lib.cplb_get_mu(prob._h, C.byref(mu)) == 0 and mu.value == 0.25
        assert lib.cplb_get_ground_z(prob._h, C.byref(z)) == 0 and z.value == 0.4
    c = cpl.BatchedCplProblem(["x", "y"], 50.0, None)   # CoMPlanner variant: _ground_fake holds mu (CplProblem.cpp:282-285)
    c.SetMu(0.3)
    assert c.GetMu() == 0.3 and (c.m, c.nnz) == (10, 60)


def test_get_solution_unpacks_in_sorted_order():
    prob = cpl.BatchedCplProblem(["r_foot", "l_foot"], 100.0, cpl.Ground())
    x = np.arange(21, dtype=np.float64)
    sol = prob.GetSolution(x)
    assert list(sol["com_sol"]) == [0, 1, 2]
    assert list(sol["contact_values_map"]) == ["l_foot", "r_foot"]     # std::map order (CplProblem.cpp:90)
    assert list(sol["contact_values_map"]["l_foot"]["force_value"]) == [12, 13, 14]
    assert list(sol["contact_values_map"]["r_foot"]["normal_value"]) == [9, 10, 11]


def test_evaluation_without_a_gpu_fails_loudly():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is for CPU-only machines")
    prob, _, gen = make_pair("ground4")
    with pytest.raises(RuntimeError, match="no usable CUDA device"):
        prob.eval(gen(8))


def test_pybind11_module_builds_and_keeps_the_exception_mapping():
    """bindings/python/pycplb.cpp (pybind11 over the same C ABI): importable on a CPU box, reference class and method
    names, std::invalid_argument -> ValueError, std::out_of_range -> IndexError, evaluation fails loudly without a GPU."""
    import subprocess
    import sys

    subprocess.check_call(["make", "-C", os.path.join(ROOT, "bindings", "python")], stdout=subprocess.DEVNULL)
    sys.path.insert(0, os.path.join(ROOT, "centroidalplanner_b200"))
    import pycplb

    g = pycplb.Ground()
    g.SetGroundZ(0.1)
    p = pycplb.BatchedProblem(["r_foot", "l_foot"], 100.0, g)
    assert (p.n, p.m, p.nnz) == (21, 18, 90) and list(p.GetSortedOrder()) == [1, 0]
    with pytest.raises(ValueError, match="Invalid friction coefficient"):
        g.SetMu(-1.0)
    with pytest.raises(IndexError):
        p.SetForceThreshold("nose", 1.0)
    with pytest.raises(ValueError, match="Invalid robot mass"):
        pycplb.BatchedProblem(["a"], -1.0, g)
    sq = pycplb.Superquadric()
    with pytest.raises(ValueError, match="curvatures"):
        sq.SetParameters([0, 0, 1], [1, 1, 1], [1.5, 2, 2])
    c = pycplb.BatchedProblem(["a", "b"], 50.0)         # env = nullptr: the CoMPlanner shape
    c.SetMu(0.3)
    assert c.GetMu() == 0.3 and (c.m, c.nnz) == (10, 60)
    import torch

    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no usable CUDA device"):
            p.eval(np.zeros((4, 21)))


def test_eval_argument_checks_happen_before_any_device_work():
    """Bad arguments are INVALID_ARGUMENT / NULL_POINTER on any machine; an empty batch is a no-op that succeeds."""
    import ctypes as C

    lib = _cabi.load()
    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    x = np.zeros((4, prob.n))
    g = np.zeros((4, prob.m))

    def call(fn, **kw):
        a = dict(num_instances=4, layout=cpl.INSTANCE_MAJOR, host_flags=0, ld=0, x=x.ctypes.data, g=g.ctypes.data, jac=None, cost=None,
                 grad=None, per_instance=None)
        a.update(kw)
        args = _cabi.EvalArgs(*[a[k] for k in ("num_instances", "layout", "host_flags", "ld", "x", "g", "jac", "cost", "grad", "per_instance")])
        return fn(prob._h, C.byref(args)) if fn is lib.cplb_eval_host else fn(prob._h, C.byref(args), None)

    for fn in (lib.cplb_eval_host, lib.cplb_eval_device):
        assert call(fn, num_instances=-1) == _cabi.INVALID_ARGUMENT
        assert call(fn, layout=7) == _cabi.INVALID_ARGUMENT
        assert call(fn, x=None) == _cabi.NULL_POINTER
        assert call(fn, layout=cpl.COMPONENT_MAJOR, ld=3) == _cabi.INVALID_ARGUMENT and b"ld" in lib.cplb_last_error()
        assert call(fn, layout=cpl.COMPONENT_MAJOR, ld=1 << 29) == _cabi.INVALID_ARGUMENT and b"2^29" in lib.cplb_last_error()
        assert call(fn, num_instances=0) == _cabi.OK                      # empty batch
        assert call(fn, g=None) == _cabi.OK                               # nothing requested
    assert lib.cplb_eval_host(None, None) == _cabi.NULL_POINTER


def test_queued_host_call_argument_checks():
    """cplb_eval_host_begin / _wait validate before any device work, like cplb_eval_host: NULL ticket pointer, unknown tickets,
    and (without a CUDA device) the same loud failure instead of a CPU evaluation."""
    import torch

    prob = cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
    lib = _cabi.load()
    x = np.zeros((4, prob.n))
    args = _cabi.EvalArgs(4, cpl.INSTANCE_MAJOR, 0, 4, x.ctypes.data, None, None, None, None, None)
    assert lib.cplb_eval_host_begin(prob._h, C.byref(args), None) == _cabi.NULL_POINTER
    with pytest.raises(ValueError, match="unknown ticket"):
        prob.eval_host_wait(3)                     # nothing was ever begun
    prob.eval_host_wait(-1)                        # the ticket of an empty call
    ticket, _ = prob.eval_host_begin(np.zeros((0, prob.n)), {}, g=False, jac=False)   # no instances, no outputs: completes at once
    assert ticket == -1
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no usable CUDA device"):
            prob.eval_host_begin(x, {"g": np.zeros((4, prob.m))}, g=True, jac=False)


def test_kernel_choice_validation():
    """cplb_set_component_major_kernel: unknown choices and the thread-per-instance kernel on a problem it does not exist for
    are refused (CPLB_INVALID_ARGUMENT -> ValueError); host-only, no GPU needed for the check itself."""
    prob, _, _ = make_pair("ground5")
    with pytest.raises(ValueError, match="4 and 8 contacts"):
        prob.SetComponentMajorKernel("whole")
    with pytest.raises(ValueError, match="unknown"):
        prob.SetComponentMajorKernel(7)
    prob.SetComponentMajorKernel(_cabi.KERNEL_PER_CONTACT)
    prob.SetComponentMajorKernel(_cabi.KERNEL_AUTO)


@pytest.mark.parametrize("case", sorted(CASES))
def test_packed_jacobian_map_and_host_unpack(case):
    """cplb_get_packed_jacobian_map lists the x-dependent slots in slot order; cplb_unpack_jacobian (host-only) rebuilds full rows
    from packed slices: checked here on the oracle's values, no GPU involved."""
    prob, o, gen = make_pair(case)
    pmap = prob.GetPackedJacobianMap()
    mask, cval = prob.GetJacobianConstants()
    assert np.array_equal(pmap, np.nonzero(~mask)[0]) and len(pmap) + int(mask.sum()) == prob.nnz
    nc = o.nc
    expect = {orc.ENV_NONE: 6 + 24 * nc, orc.ENV_GROUND: 6 + 24 * nc, orc.ENV_SUPERQUADRIC: 6 + 36 * nc}[o.env_kind]
    assert len(pmap) == expect
    x = gen(50)
    jac = o.eval_batch(x, want=("jac",))["jac"]
    assert same_bits_host(prob.UnpackJacobian(np.ascontiguousarray(jac[:, pmap])), jac)
    with pytest.raises(ValueError):
        prob.UnpackJacobian(jac)            # full rows are not packed slices


@pytest.mark.parametrize("case", sorted(CASES))
def test_jacobian_slot_sources_against_the_oracle(case):
    """cplb_get_jacobian_slot_sources: every slot marked as a copy holds exactly +-x[source] in the reference's values (the p_k
    entries of the moment rows, CentroidalStatics.cpp:108-113; FrictionCone's first row, FrictionCone.cpp:82-84,93-95), the
    constants are the constants, and cplb_expand_jacobian (host-only) rebuilds the oracle's full rows from x and the computed
    slots alone.  No GPU involved."""
    prob, o, gen = make_pair(case)
    kind, src = prob.GetJacobianSlotSources()
    mask, cval = prob.GetJacobianConstants()
    nc = o.nc
    assert np.array_equal(kind == _cabi.SLOT_CONSTANT, mask)
    assert int((kind == _cabi.SLOT_COPY).sum() + (kind == _cabi.SLOT_NEGATED_COPY).sum()) == 12 * nc
    comp = np.nonzero(kind == _cabi.SLOT_COMPUTED)[0]
    expect = {orc.ENV_NONE: 6 + 12 * nc, orc.ENV_GROUND: 6 + 12 * nc, orc.ENV_SUPERQUADRIC: 6 + 24 * nc}[o.env_kind]
    assert len(comp) == expect and np.array_equal(src[comp], np.arange(len(comp)))   # computed slots appear in slot order
    x = gen(64)
    x[0] = 0.0                                                                       # -0.0 and NaN rows of the default start
    jac = o.eval_batch(x, want=("jac",))["jac"]
    for s in np.nonzero(kind == _cabi.SLOT_COPY)[0]:
        assert same_bits_host(jac[:, s], x[:, src[s]]), (case, s)
    for s in np.nonzero(kind == _cabi.SLOT_NEGATED_COPY)[0]:
        assert same_bits_host(jac[:, s], -x[:, src[s]]) and np.array_equal(np.signbit(jac[:, s]), np.signbit(-x[:, src[s]])), (case, s)
    full = prob.ExpandJacobian(x, np.ascontiguousarray(jac[:, comp]))
    assert same_bits_host(full, jac)
    with pytest.raises(ValueError):
        prob.ExpandJacobian(x, jac)
    with pytest.raises(ValueError, match="computed"):
        prob._jac_flag("dense")


def test_slice_helpers_check_their_arguments():
    """cplb_get_jacobian_slot_sources / cplb_expand_jacobian / cplb_unpack_jacobian straight through the C ABI: NULL outputs are a
    size query, NULL inputs and negative counts are errors with a message, zero instances is a no-op."""
    lib = _cabi.load()
    prob, o, gen = make_pair("ground4")
    nv = C.c_int32(-1)
    assert lib.cplb_get_jacobian_slot_sources(prob._h, C.byref(nv), None, None) == _cabi.OK and nv.value == 54
    assert lib.cplb_get_jacobian_slot_sources(None, C.byref(nv), None, None) == _cabi.NULL_POINTER
    x = gen(3)
    comp = np.zeros((3, 54))
    full = np.zeros((3, o.nnz))
    dp = _cabi.dp
    assert lib.cplb_expand_jacobian(prob._h, 0, None, None, None) == _cabi.OK
    assert lib.cplb_expand_jacobian(prob._h, -1, x.ctypes.data_as(dp), comp.ctypes.data_as(dp), full.ctypes.data_as(dp)) == _cabi.INVALID_ARGUMENT
    assert b"negative" in lib.cplb_last_error()
    assert lib.cplb_expand_jacobian(prob._h, 3, None, comp.ctypes.data_as(dp), full.ctypes.data_as(dp)) == _cabi.NULL_POINTER
    assert lib.cplb_expand_jacobian(prob._h, 3, x.ctypes.data_as(dp), comp.ctypes.data_as(dp), None) == _cabi.NULL_POINTER
    assert lib.cplb_unpack_jacobian(prob._h, 3, None, full.ctypes.data_as(dp)) == _cabi.NULL_POINTER
    # solver options: defaults as documented in the header
    opt = _cabi.SolverOptions()
    lib.cplb_solver_default_options(C.byref(opt))
    assert (opt.tol, opt.max_iter, opt.max_backtracks, opt.tail_instances) == (1e-3, 500, 30, -1)


def same_bits_host(a, b):
    na, nb = np.isnan(a), np.isnan(b)
    return bool((na == nb).all() and (a[~na] == b[~nb]).all())


def test_header_is_valid_c99_and_usable_from_plain_c(tmp_path):
    """include/cpl_batched.h compiled by gcc as strict C99 and driven from a C program (no C++, no Python, no GPU)."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc") or "gcc"
    exe = str(tmp_path / "abi_c_check")
    pkg = os.path.join(ROOT, "centroidalplanner_b200")
    subprocess.check_call([gcc, "-std=c99", "-pedantic", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "native", "abi_c_check.c"), "-o", exe, "-L", pkg, "-lcplb", f"-Wl,-rpath,{pkg}"])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0 and "C ABI ok" in r.stdout, (r.returncode, r.stdout, r.stderr)


def test_solution_extraction_and_printing_cpp_vs_python(tmp_path):
    """CplProblem::GetSolution + operator<<(Solution) (src/CplProblem.cpp:85-106, 319-346): the C++ facade and the Python
    mirror unpack x by the same column map into sorted-name order and print the same text."""
    import shutil
    import subprocess

    gxx = shutil.which("g++") or "g++"
    exe = str(tmp_path / "solution_check")
    pkg = os.path.join(ROOT, "centroidalplanner_b200")
    subprocess.check_call([gxx, "-std=c++14", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", os.path.join(pkg, "cpp", "include"), os.path.join(ROOT, "tests", "native", "solution_check.cpp"),
                           "-o", exe, "-L", pkg, "-lcplb", f"-Wl,-rpath,{pkg}"])
    names = ["r_foot", "l_foot", "r_hand"]
    prob = cpl.BatchedCplProblem(names, 100.0, cpl.Ground())
    x = np.array([0.0401, 0.01695, 0.99591] + [34.78973, -69.5, 156.02521, 0.09298, -0.03415, 0.1, 0.0, 0.0, 1.0]
                 + [-106.8, 1e-7, 345.35119, -0.23352, 0.20405, 0.1, -0.0, 0.0, 1.0] + [1234567.0, 2.5, 1.0 / 3.0, 0.14, -0.06, 0.1, 0.6, 0.0, 0.8])
    r = subprocess.run([exe] + [repr(float(v)) for v in x], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, (r.returncode, r.stderr)
    sol = prob.GetSolution(x)
    assert list(sol["contact_values_map"]) == ["l_foot", "r_foot", "r_hand"]
    assert r.stdout == prob.FormatSolution(sol)
    assert r.stdout.splitlines()[0] == "CoM:  0.0401 0.01695 0.99591"
    assert r.stdout.splitlines()[1] == "F_l_foot:  -106.8   1e-07 345.351"          # l_foot is the SECOND name of the caller's vector
    assert r.stdout.splitlines()[3] == "F_r_hand: 1.23457e+06         2.5    0.333333"


def test_missing_extension_fails_loudly(monkeypatch, tmp_path):
    """No silent fallback: without libcplb.so the package cannot create a problem at all."""
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "libcplb.so"))
    with pytest.raises(ImportError, match="no CPU fallback"):
        cpl.BatchedCplProblem(synthetic.NAMES4, 100.0, cpl.Ground())
