"""Host-side mirror of the reference's problem interface over the C ABI.

`BatchedCplProblem` plays the role of `cpl::solver::CplProblem` (include/CentroidalPlanner/Ifopt/
CplProblem.h:19-115, src/CplProblem.cpp) for N instances at once: same constructor arguments,
same setter/getter names, same error behaviour (std::invalid_argument -> ValueError,
std::out_of_range -> IndexError, std::runtime_error -> RuntimeError, i.e. pybind11's mapping),
and the four `ifopt::Problem` evaluation entry points IPOPT drives, batched.  `Ground` and
`Superquadric` mirror cpl::env (Environment.h:13-48, Ground.h, Superquadric.h).

Everything numeric happens in libcplb.so on the GPU; torch is used only to own device memory and
streams.  NumPy / CPU-tensor inputs go through `cplb_eval_host` (host buffers, copies inside).
"""
from __future__ import annotations

import ctypes as C
import weakref
from dataclasses import dataclass

import numpy as np

from . import _cabi

_EXC = {
    _cabi.INVALID_ARGUMENT: ValueError,
    _cabi.OUT_OF_RANGE: IndexError,
    _cabi.RUNTIME_ERROR: RuntimeError,
    _cabi.CUDA_ERROR: RuntimeError,
    _cabi.NULL_POINTER: ValueError,
}


def _check(status):
    if status != _cabi.OK:
        msg = _cabi.load().cplb_last_error().decode(errors="replace")
        raise _EXC.get(status, RuntimeError)(msg)


def _v3(v, n=3):
    a = np.ascontiguousarray(np.asarray(v, dtype=np.float64).reshape(n))
    return a, a.ctypes.data_as(_cabi.dp)


class EnvironmentClass:
    """cpl::env::EnvironmentClass (Environment.h:13-48): friction coefficient, default 1.0."""

    _kind = _cabi.ENV_NONE

    def __init__(self):
        self._mu = 1.0
        self._problems = weakref.WeakSet()

    def SetMu(self, mu):
        if mu <= 0.0:
            raise ValueError("Invalid friction coefficient")
        self._mu = float(mu)
        self._push()

    def GetMu(self):
        return self._mu

    def _attach(self, problem):
        self._problems.add(problem)
        self._push_to(problem)

    def _push(self):
        for p in list(self._problems):
            self._push_to(p)

    def _push_to(self, problem):
        _check(problem._lib.cplb_set_mu(problem._h, self._mu))


class Ground(EnvironmentClass):
    """cpl::env::Ground (Ground.h:13-40, src/Ground.cpp): the plane z = ground_z."""

    _kind = _cabi.ENV_GROUND

    def __init__(self):
        super().__init__()
        self._ground_z = 0.0

    def SetGroundZ(self, ground_z):
        self._ground_z = float(ground_z)
        self._push()

    def GetGroundZ(self):
        return self._ground_z

    def _push_to(self, problem):
        super()._push_to(problem)
        if problem._env_kind == _cabi.ENV_GROUND:
            _check(problem._lib.cplb_set_ground_z(problem._h, self._ground_z))


class Superquadric(EnvironmentClass):
    """cpl::env::Superquadric (Superquadric.h:13-49, src/Superquadric.cpp:5-37)."""

    _kind = _cabi.ENV_SUPERQUADRIC

    def __init__(self):
        super().__init__()
        self._C = np.array([0.0, 0.0, 10.0])
        self._R = np.array([10.0, 10.0, 10.0])
        self._P = np.array([10.0, 10.0, 10.0])

    def SetParameters(self, Cc, R, P):
        Cc, R, P = (np.asarray(v, dtype=np.float64).reshape(3) for v in (Cc, R, P))
        if (R <= 0.0).any():
            raise ValueError("Invalid superquadric axial radii")
        if (P < 2.0).any():
            raise ValueError("Invalid superquadric axial curvatures: must be >= 2")
        self._C, self._R, self._P = Cc.copy(), R.copy(), P.copy()
        self._push()

    def GetParameters(self):
        return self._C.copy(), self._R.copy(), self._P.copy()

    def _push_to(self, problem):
        super()._push_to(problem)
        _, c = _v3(self._C)
        _, r = _v3(self._R)
        _, p = _v3(self._P)
        _check(problem._lib.cplb_set_superquadric(problem._h, c, r, p))


@dataclass
class DerivativeTestReport:
    """BatchedCplProblem.DerivativeTest: per instance (CUDA tensors, instance-major), see cplb_derivative_test_device."""
    num_wrong: object          # (N,) int32  wrong entries: gradient + every (row, col) of the dense Jacobian
    num_wrong_outside: object  # (N,) int32  of those, Jacobian entries outside the declared structure
    max_rel_error: object      # (N,) float64  rel of the worst entry (NaN stays NaN)
    worst_row: object          # (N,) int32  -1 = cost gradient
    worst_col: object          # (N,) int32
    jac_fd: object             # (N, nnz) float64  forward differences at the structural slots
    grad_fd: object            # (N, n) float64


def _is_torch(t):
    return type(t).__module__.startswith("torch")


class BatchedCplProblem:
    """N instances of one CplProblem shape, evaluated on one B200.

    contact_names / robot_mass / env as in CplProblem::CplProblem (src/CplProblem.cpp:6-11);
    env=None selects the CoMPlanner variant (FrictionCone only, src/CplProblem.cpp:63-71).
    """

    def __init__(self, contact_names, robot_mass, env=None, device=None, devices=None):
        """device: CUDA ordinal (None: the current device at the first evaluation).  devices: a list of ordinals makes this a
        SHARDED problem (cplb_create_sharded): host-buffer evaluations then cut the batch into one contiguous range per device
        and drive all of them from this process; device tensors go through eval_shard()."""
        self._lib = _cabi.load()
        self._names = [str(s) for s in contact_names]
        self._env = env
        self._env_kind = _cabi.ENV_NONE if env is None else env._kind
        self._ground_fake = Ground() if env is None else None  # CplProblem.cpp:14
        arr = (C.c_char_p * len(self._names))(*[s.encode() for s in self._names])
        h = C.c_void_p()
        if devices is not None:
            if device is not None:
                raise ValueError("give either device or devices")
            devs = np.ascontiguousarray(np.asarray(list(devices), dtype=np.int32))
            _check(self._lib.cplb_create_sharded(len(self._names), arr, self._env_kind, float(robot_mass), len(devs),
                                                 devs.ctypes.data_as(_cabi.ip), C.byref(h)))
        else:
            dev = -1 if device is None else int(device)
            _check(self._lib.cplb_create(len(self._names), arr, self._env_kind, float(robot_mass), dev, C.byref(h)))
        self._h = h
        n, m, nnz = C.c_int32(), C.c_int32(), C.c_int32()
        _check(self._lib.cplb_get_dims(self._h, C.byref(n), C.byref(m), C.byref(nnz)))
        self.n, self.m, self.nnz = n.value, m.value, nnz.value
        (env if env is not None else self._ground_fake)._attach(self)

    def __del__(self):
        h = getattr(self, "_h", None)
        if h:
            self._lib.cplb_destroy(h)
            self._h = None

    # ---- layout ------------------------------------------------------------------------------
    @property
    def contact_names(self):
        return list(self._names)

    def GetNumberOfOptimizationVariables(self):
        return self.n

    def GetNumberOfConstraints(self):
        return self.m

    def GetJacobianStructure(self):
        """(iRow, jCol) exactly as IpoptAdapter::eval_jac_g(values=NULL) would fill them."""
        r = np.zeros(self.nnz, dtype=np.int32)
        c = np.zeros(self.nnz, dtype=np.int32)
        _check(self._lib.cplb_get_jacobian_structure(self._h, r.ctypes.data_as(_cabi.ip), c.ctypes.data_as(_cabi.ip)))
        return r, c

    def GetSortedOrder(self):
        p = np.zeros(len(self._names), dtype=np.int32)
        _check(self._lib.cplb_get_sorted_order(self._h, p.ctypes.data_as(_cabi.ip)))
        return p

    def GetBlockColumn(self, block, contact_name=None):
        col = C.c_int32()
        name = None if contact_name is None else str(contact_name).encode()
        _check(self._lib.cplb_get_block_column(self._h, int(block), name, C.byref(col)))
        return col.value

    def GetContactRow(self, contact_name):
        row = C.c_int32()
        _check(self._lib.cplb_get_contact_row(self._h, str(contact_name).encode(), C.byref(row)))
        return row.value

    def GetBoundsOnOptimizationVariables(self):
        lb, ub = np.zeros(self.n), np.zeros(self.n)
        _check(self._lib.cplb_get_variable_bounds(self._h, lb.ctypes.data_as(_cabi.dp), ub.ctypes.data_as(_cabi.dp)))
        return lb, ub

    def GetBoundsOnConstraints(self):
        lb, ub = np.zeros(self.m), np.zeros(self.m)
        _check(self._lib.cplb_get_constraint_bounds(self._h, lb.ctypes.data_as(_cabi.dp), ub.ctypes.data_as(_cabi.dp)))
        return lb, ub

    # ---- CplProblem forwarders (src/CplProblem.cpp:109-316) ----------------------------------
    def _set_bounds(self, block, name, lb, ub):
        _, l = _v3(lb)
        _, u = _v3(ub)
        _check(self._lib.cplb_set_bounds(self._h, block, None if name is None else str(name).encode(), l, u))

    def _get_bounds(self, block, name):
        lb, ub = np.zeros(3), np.zeros(3)
        _check(self._lib.cplb_get_bounds(self._h, block, None if name is None else str(name).encode(),
                                         lb.ctypes.data_as(_cabi.dp), ub.ctypes.data_as(_cabi.dp)))
        return lb, ub

    def SetForceBounds(self, contact_name, force_lb, force_ub):
        self._set_bounds(_cabi.BLOCK_FORCE, contact_name, force_lb, force_ub)

    def GetForceBounds(self, contact_name):
        return self._get_bounds(_cabi.BLOCK_FORCE, contact_name)

    def SetPosBounds(self, contact_name, pos_lb, pos_ub):
        self._set_bounds(_cabi.BLOCK_POSITION, contact_name, pos_lb, pos_ub)

    def GetPosBounds(self, contact_name):
        return self._get_bounds(_cabi.BLOCK_POSITION, contact_name)

    def SetNormalBounds(self, contact_name, normal_lb, normal_ub):
        self._set_bounds(_cabi.BLOCK_NORMAL, contact_name, normal_lb, normal_ub)

    def GetNormalBounds(self, contact_name):
        return self._get_bounds(_cabi.BLOCK_NORMAL, contact_name)

    def _set3(self, fn, name, v):
        _, p = _v3(v)
        _check(fn(self._h, str(name).encode(), p))

    def _get3(self, fn, name):
        out = np.zeros(3)
        _check(fn(self._h, str(name).encode(), out.ctypes.data_as(_cabi.dp)))
        return out

    def _get1(self, fn, *args):
        out = C.c_double()
        _check(fn(self._h, *args, C.byref(out)))
        return out.value

    def SetPosRef(self, contact_name, pos_ref):
        self._set3(self._lib.cplb_set_pos_ref, contact_name, pos_ref)

    def GetPosRef(self, contact_name):
        return self._get3(self._lib.cplb_get_pos_ref, contact_name)

    def SetForceRef(self, contact_name, force_ref):
        self._set3(self._lib.cplb_set_force_ref, contact_name, force_ref)

    def GetForceRef(self, contact_name):
        return self._get3(self._lib.cplb_get_force_ref, contact_name)

    def SetCoMRef(self, com_ref):
        _, p = _v3(com_ref)
        _check(self._lib.cplb_set_com_ref(self._h, p))

    def GetCoMRef(self):
        out = np.zeros(3)
        _check(self._lib.cplb_get_com_ref(self._h, out.ctypes.data_as(_cabi.dp)))
        return out

    def SetCoMWeight(self, W_CoM):
        _check(self._lib.cplb_set_com_weight(self._h, float(W_CoM)))

    def GetCoMWeight(self):
        return self._get1(self._lib.cplb_get_com_weight)

    def SetPosWeight(self, W_p):
        _check(self._lib.cplb_set_pos_weight(self._h, float(W_p)))

    def SetContactPosWeight(self, contact_name, W_p):
        _check(self._lib.cplb_set_contact_pos_weight(self._h, str(contact_name).encode(), float(W_p)))

    def GetContactPosWeight(self, contact_name):
        return self._get1(self._lib.cplb_get_contact_pos_weight, str(contact_name).encode())

    def SetForceWeight(self, W_F):
        _check(self._lib.cplb_set_force_weight(self._h, float(W_F)))

    def SetContactForceWeight(self, contact_name, W_F):
        _check(self._lib.cplb_set_contact_force_weight(self._h, str(contact_name).encode(), float(W_F)))

    def GetContactForceWeight(self, contact_name):
        return self._get1(self._lib.cplb_get_contact_force_weight, str(contact_name).encode())

    def SetManipulationWrench(self, wrench_manip):
        _, p = _v3(wrench_manip, 6)
        _check(self._lib.cplb_set_manipulation_wrench(self._h, p))

    def GetManipulationWrench(self):
        out = np.zeros(6)
        _check(self._lib.cplb_get_manipulation_wrench(self._h, out.ctypes.data_as(_cabi.dp)))
        return out

    def SetMu(self, mu):
        # CplProblem::SetMu (src/CplProblem.cpp:275-287): forwards to the env, or to _ground_fake
        (self._env if self._env is not None else self._ground_fake).SetMu(mu)

    def GetMu(self):
        return (self._env if self._env is not None else self._ground_fake).GetMu()

    def SetForceThreshold(self, contact_name, F_thr):
        _check(self._lib.cplb_set_force_threshold(self._h, str(contact_name).encode(), float(F_thr)))

    def GetForceThreshold(self, contact_name):
        return self._get1(self._lib.cplb_get_force_threshold, str(contact_name).encode())

    def SetReductionOrder(self, order):
        """0: (v0+v1)+v2 (default, Eigen >= 3.3); 1: v0+(v1+v2).  See cplb_set_reduction_order."""
        _check(self._lib.cplb_set_reduction_order(self._h, int(order)))

    def SetMass(self, mass):
        _check(self._lib.cplb_set_mass(self._h, float(mass)))

    def SetComponentMajorKernel(self, kernel):
        """cplb_set_component_major_kernel: KERNEL_AUTO / KERNEL_PER_CONTACT / KERNEL_PER_INSTANCE (or 'auto', 'split', 'whole')."""
        kernel = {"auto": _cabi.KERNEL_AUTO, "split": _cabi.KERNEL_PER_CONTACT, "whole": _cabi.KERNEL_PER_INSTANCE}.get(kernel, kernel)
        _check(self._lib.cplb_set_component_major_kernel(self._h, int(kernel)))

    def SetInstanceMajorKernel(self, kernel):
        """cplb_set_instance_major_kernel: KERNEL_AUTO / KERNEL_WARP_TILE / KERNEL_CTA_TILE (or 'auto', 'warp', 'cta')."""
        kernel = {"auto": _cabi.KERNEL_AUTO, "warp": _cabi.KERNEL_WARP_TILE, "cta": _cabi.KERNEL_CTA_TILE}.get(kernel, kernel)
        _check(self._lib.cplb_set_instance_major_kernel(self._h, int(kernel)))

    def GetNumShards(self):
        v = C.c_int32()
        _check(self._lib.cplb_get_num_shards(self._h, C.byref(v)))
        return v.value

    def GetShard(self, shard, num_instances):
        """(device ordinal, begin, end): the contiguous instance range of a batch of num_instances that shard evaluates."""
        d, b, e = C.c_int32(), C.c_int64(), C.c_int64()
        _check(self._lib.cplb_get_shard(self._h, int(shard), int(num_instances), C.byref(d), C.byref(b), C.byref(e)))
        return d.value, b.value, e.value

    def GetDevice(self):
        d = C.c_int32()
        _check(self._lib.cplb_get_device(self._h, C.byref(d)))
        return d.value

    # ---- evaluation --------------------------------------------------------------------------
    def _shape(self, length, N, layout):
        return (N, length) if layout == _cabi.INSTANCE_MAJOR else (length, N)

    def GetJacobianConstants(self):
        """(is_constant[nnz] bool, value[nnz]): structural slots whose value does not depend on x."""
        mask = np.zeros(self.nnz, dtype=np.uint8)
        val = np.zeros(self.nnz)
        _check(self._lib.cplb_get_jacobian_constants(self._h, mask.ctypes.data_as(C.POINTER(C.c_uint8)), val.ctypes.data_as(_cabi.dp)))
        return mask.astype(bool), val

    def GetPackedJacobianMap(self):
        """packed_to_slot[nv]: element q of a packed Jacobian slice (jac_packed=True) is structural slot packed_to_slot[q]."""
        nv = C.c_int32()
        _check(self._lib.cplb_get_packed_jacobian_map(self._h, C.byref(nv), None))
        m = np.zeros(nv.value, dtype=np.int32)
        _check(self._lib.cplb_get_packed_jacobian_map(self._h, C.byref(nv), m.ctypes.data_as(_cabi.ip)))
        return m

    def UnpackJacobian(self, packed):
        """cplb_unpack_jacobian: (N, nv) packed host slices -> (N, nnz) full rows, constants included."""
        a = np.ascontiguousarray(packed.numpy() if _is_torch(packed) else packed, dtype=np.float64)
        nv = len(self.GetPackedJacobianMap())
        if a.ndim != 2 or a.shape[1] != nv:
            raise ValueError(f"packed has shape {a.shape}, expected (N, {nv})")
        full = np.empty((a.shape[0], self.nnz))
        _check(self._lib.cplb_unpack_jacobian(self._h, a.shape[0], a.ctypes.data_as(_cabi.dp), full.ctypes.data_as(_cabi.dp)))
        return full

    def GetJacobianSlotSources(self):
        """(kind[nnz], source[nnz]) of cplb_get_jacobian_slot_sources: where each structural slot's value comes from
        (_cabi.SLOT_CONSTANT / SLOT_COPY x[source] / SLOT_NEGATED_COPY -x[source] / SLOT_COMPUTED element `source` of a
        jac_packed='computed' slice)."""
        kind = np.zeros(self.nnz, dtype=np.int32)
        src = np.zeros(self.nnz, dtype=np.int32)
        nv = C.c_int32()
        _check(self._lib.cplb_get_jacobian_slot_sources(self._h, C.byref(nv), kind.ctypes.data_as(_cabi.ip), src.ctypes.data_as(_cabi.ip)))
        return kind, src

    def ExpandJacobian(self, x, computed):
        """cplb_expand_jacobian: (N, n) x and (N, nv) computed host slices -> (N, nnz) full rows, constants and copies included."""
        xa = np.ascontiguousarray(x.numpy() if _is_torch(x) else x, dtype=np.float64)
        a = np.ascontiguousarray(computed.numpy() if _is_torch(computed) else computed, dtype=np.float64)
        nv = self._jac_len("computed")
        if a.ndim != 2 or a.shape[1] != nv or xa.shape != (a.shape[0], self.n):
            raise ValueError(f"x has shape {xa.shape}, computed {a.shape}; expected (N, {self.n}) and (N, {nv})")
        full = np.empty((a.shape[0], self.nnz))
        _check(self._lib.cplb_expand_jacobian(self._h, a.shape[0], xa.ctypes.data_as(_cabi.dp), a.ctypes.data_as(_cabi.dp), full.ctypes.data_as(_cabi.dp)))
        return full

    def FillJacobianConstants(self, jac_host, layout=_cabi.INSTANCE_MAJOR):
        """Write the constant slots of a host jac buffer once; later host evaluations into the same buffer may then
        pass jac_constants_present=True and skip transferring them."""
        a = jac_host.numpy() if _is_torch(jac_host) else jac_host
        if a.dtype != np.float64 or not a.flags.c_contiguous or a.ndim != 2:
            raise ValueError("jac_host must be a C-contiguous 2-D float64 array")
        N = a.shape[0] if layout == _cabi.INSTANCE_MAJOR else a.shape[1]
        if tuple(a.shape) != self._shape(self.nnz, N, layout):
            raise ValueError(f"jac_host has shape {tuple(a.shape)}, expected {self._shape(self.nnz, N, layout)}")
        _check(self._lib.cplb_fill_jacobian_constants(self._h, N, layout, N, a.ctypes.data_as(_cabi.dp)))

    def _instance_params(self, per_instance, N, layout, on_device):
        """dict name -> array (cplb_instance_params fields) -> (ctypes struct, keep-alive list); shapes follow x's
        layout: (N,) / (N, len) instance-major, (len, N) component-major.  on_device: x's torch device, or None (host)."""
        if not per_instance:
            return None, []
        lens = {"mass": 1, "wrench": 6, "mu": 1, "force_threshold": len(self._names), "ground_z": 1, "com_ref": 3, "com_weight": 1,
                "pos_ref": 3 * len(self._names), "force_ref": 3 * len(self._names), "pos_weight": len(self._names),
                "force_weight": len(self._names)}
        st, keep = _cabi.InstanceParams(), []
        for name, arr in per_instance.items():
            if name not in lens:
                raise ValueError(f"unknown per-instance parameter '{name}'")
            L = lens[name]
            if on_device is not None:
                import torch

                if not (_is_torch(arr) and arr.is_cuda and arr.dtype == torch.float64 and arr.is_contiguous()):
                    raise ValueError(f"per-instance array '{name}' must be a contiguous float64 CUDA tensor")
                if arr.device != on_device:
                    raise ValueError(f"per-instance array '{name}' lives on {arr.device}, x on {on_device}")
                if arr.numel() != N * L:
                    raise ValueError(f"per-instance array '{name}' has {arr.numel()} elements, expected {N} x {L}")
                setattr(st, name, arr.data_ptr())
            else:
                arr = np.ascontiguousarray(arr.numpy() if _is_torch(arr) else np.asarray(arr, dtype=np.float64), dtype=np.float64)
                if arr.size != N * L:
                    raise ValueError(f"per-instance array '{name}' has {arr.size} elements, expected {N} x {L}")
                setattr(st, name, arr.ctypes.data)
            keep.append(arr)
        return st, keep

    def eval(self, x, g=True, jac=True, cost=False, grad=False, layout=_cabi.INSTANCE_MAJOR, out=None, stream=None,
             jac_constants_present=False, per_instance=None, inputs_ready=False, jac_packed=False):
        """One batched evaluation.  x: (N, n) [instance-major] or (n, N) [component-major], fp64,
        a torch CUDA tensor (device path, asynchronous on the current stream) or a NumPy array /
        CPU tensor (host path through cplb_eval_host).  Returns a dict of outputs of the same kind."""
        out = dict(out or {})
        if _is_torch(x) and x.is_cuda:
            return self._eval_device(x, g, jac, cost, grad, layout, out, stream, per_instance, inputs_ready, jac_packed=jac_packed)
        return self._eval_host(x, g, jac, cost, grad, layout, out, jac_constants_present, per_instance, jac_packed=jac_packed)

    @staticmethod
    def _is_computed(jac_packed):
        """jac_packed: False (full rows), True (x-dependent slots), 'computed' (only the slots that take arithmetic)."""
        if isinstance(jac_packed, str):
            if jac_packed != "computed":
                raise ValueError(f"jac_packed={jac_packed!r}: expected False, True or 'computed'")
            return True
        return False

    def _jac_flag(self, jac_packed):
        if self._is_computed(jac_packed):
            return _cabi.JAC_COMPUTED
        return _cabi.JAC_PACKED if jac_packed else 0

    def _jac_len(self, jac_packed):
        if self._is_computed(jac_packed):
            if getattr(self, "_nv2", None) is None:
                nv = C.c_int32()
                _check(self._lib.cplb_get_jacobian_slot_sources(self._h, C.byref(nv), None, None))
                self._nv2 = nv.value
            return self._nv2
        if not jac_packed:
            return self.nnz
        if getattr(self, "_nv", None) is None:
            self._nv = len(self.GetPackedJacobianMap())
        return self._nv

    def _eval_device(self, x, g, jac, cost, grad, layout, out, stream, per_instance=None, inputs_ready=False, shard=None, jac_packed=False):
        import torch

        if x.dtype != torch.float64 or not x.is_contiguous() or x.dim() != 2:
            raise ValueError("x must be a contiguous 2-D float64 tensor")
        N = x.shape[0] if layout == _cabi.INSTANCE_MAJOR else x.shape[1]
        if tuple(x.shape) != self._shape(self.n, N, layout):
            raise ValueError(f"x has shape {tuple(x.shape)}, expected {self._shape(self.n, N, layout)} for this layout")
        bound = self.GetDevice() if shard is None else self.GetShard(shard, 0)[0]
        if bound >= 0 and bound != x.device.index:
            raise ValueError(f"this problem evaluates on cuda:{bound}; x lives on {x.device}")

        def buf(key, want, length):
            if not want:
                return None
            shape = (N,) if length is None else self._shape(length, N, layout)
            t = out.get(key)
            if t is None:
                return torch.empty(shape, dtype=torch.float64, device=x.device)
            if not (_is_torch(t) and t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
                raise ValueError(f"out['{key}'] must be a contiguous float64 CUDA tensor")
            if t.device != x.device:
                raise ValueError(f"out['{key}'] lives on {t.device}, x on {x.device}")
            if tuple(t.shape) != shape:
                raise ValueError(f"out['{key}'] has shape {tuple(t.shape)}, expected {shape}")
            return t

        res = {"g": buf("g", g, self.m), "jac": buf("jac", jac, self._jac_len(jac_packed)), "cost": buf("cost", cost, None),
               "grad": buf("grad", grad, self.n)}
        pi, keep = self._instance_params(per_instance, N, layout, x.device)
        args = _cabi.EvalArgs(N, layout, (_cabi.DEVICE_INPUTS_READY if inputs_ready else 0) | self._jac_flag(jac_packed), N, x.data_ptr(), *[None if res[k] is None else res[k].data_ptr()
                                                              for k in ("g", "jac", "cost", "grad")],
                              C.pointer(pi) if pi is not None else None)
        s = torch.cuda.current_stream(x.device).cuda_stream if stream is None else stream
        # a problem created without a device binds to the calling thread's CURRENT device at its first evaluation: make that x's
        with torch.cuda.device(x.device):
            if shard is None:
                _check(self._lib.cplb_eval_device(self._h, C.byref(args), C.c_void_p(s)))
            else:
                _check(self._lib.cplb_eval_device_shard(self._h, shard, C.byref(args), C.c_void_p(s)))
        return res

    def eval_shard(self, shard, x, g=True, jac=True, cost=False, grad=False, layout=_cabi.INSTANCE_MAJOR, out=None, stream=None,
                   per_instance=None, inputs_ready=False, jac_packed=False):
        """cplb_eval_device_shard: x (and the outputs) are CUDA tensors on the shard's device holding that shard's instances."""
        return self._eval_device(x, g, jac, cost, grad, layout, dict(out or {}), stream, per_instance, inputs_ready, shard=int(shard),
                                 jac_packed=jac_packed)

    def eval_host_begin(self, x, out, g=True, jac=True, cost=False, grad=False, layout=_cabi.INSTANCE_MAJOR,
                        jac_constants_present=False, per_instance=None, jac_packed=False):
        """cplb_eval_host_begin: enqueue one host-buffer evaluation and return (ticket, outputs) without waiting.  `x` and
        every array in `out` must be PINNED NumPy arrays (cplb_host_alloc) that stay alive and untouched until
        `eval_host_wait(ticket)`; with two buffer sets (begin k+1, wait k) consecutive batches keep the PCIe link busy."""
        return self._eval_host(x, g, jac, cost, grad, layout, dict(out), jac_constants_present, per_instance, begin=True, jac_packed=jac_packed)

    def eval_host_wait(self, ticket):
        _check(self._lib.cplb_eval_host_wait(self._h, int(ticket)))

    def _eval_host(self, x, g, jac, cost, grad, layout, out, jac_constants_present=False, per_instance=None, begin=False, jac_packed=False):
        is_t = _is_torch(x)
        xa = x.numpy() if is_t else np.asarray(x, dtype=np.float64)
        xa = np.ascontiguousarray(xa)
        if xa.ndim != 2:
            raise ValueError("x must be 2-D")
        N = xa.shape[0] if layout == _cabi.INSTANCE_MAJOR else xa.shape[1]
        if xa.shape != self._shape(self.n, N, layout):
            raise ValueError(f"x has shape {xa.shape}, expected {self._shape(self.n, N, layout)} for this layout")

        def buf(key, want, length):
            if not want:
                return None
            shape = (N,) if length is None else self._shape(length, N, layout)
            t = out.get(key)
            if t is None:
                return np.empty(shape)
            t = t.numpy() if _is_torch(t) else t
            if not isinstance(t, np.ndarray) or t.dtype != np.float64 or not t.flags.c_contiguous:
                raise ValueError(f"out['{key}'] must be a C-contiguous float64 array")
            if tuple(t.shape) != shape:
                raise ValueError(f"out['{key}'] has shape {tuple(t.shape)}, expected {shape}")
            return t

        res = {"g": buf("g", g, self.m), "jac": buf("jac", jac, self._jac_len(jac_packed)), "cost": buf("cost", cost, None),
               "grad": buf("grad", grad, self.n)}
        hflags = (_cabi.HOST_JAC_CONSTANTS_PRESENT if jac_constants_present else 0) | self._jac_flag(jac_packed)
        pi, keep = self._instance_params(per_instance, N, layout, None)
        args = _cabi.EvalArgs(N, layout, hflags, N, xa.ctypes.data, *[None if res[k] is None else res[k].ctypes.data
                                                                     for k in ("g", "jac", "cost", "grad")],
                              C.pointer(pi) if pi is not None else None)
        if begin:
            ticket = C.c_int32(-1)
            _check(self._lib.cplb_eval_host_begin(self._h, C.byref(args), C.byref(ticket)))
            return ticket.value, res
        _check(self._lib.cplb_eval_host(self._h, C.byref(args)))
        return res

    def DerivativeTest(self, x, per_instance=None, perturbation=1e-8, tol=1e-4, stream=None):
        """IPOPT's first-order derivative test (the reference turns it on before every solve, src/CentroidalPlanner.cpp:26) for N
        instances at once: the Jacobian and the cost gradient at x (N, n) -- a contiguous float64 CUDA tensor -- against forward
        differences of g and f, every entry of the dense Jacobian included.  Asynchronous on the current stream (or `stream`);
        per_instance: dict of per-instance parameter arrays as for eval().  Returns a DerivativeTestReport."""
        import torch

        if not (_is_torch(x) and x.is_cuda):
            raise ValueError("DerivativeTest needs x as a CUDA tensor (there is no CPU evaluation path)")
        if x.dtype != torch.float64 or not x.is_contiguous() or x.dim() != 2 or x.shape[1] != self.n:
            raise ValueError(f"x must be a contiguous (N, {self.n}) float64 tensor, got {tuple(x.shape)} {x.dtype}")
        bound = self.GetDevice()
        if bound >= 0 and bound != x.device.index:
            raise ValueError(f"this problem evaluates on cuda:{bound}; x lives on {x.device}")
        N, dev = x.shape[0], x.device
        i32, f64 = torch.int32, torch.float64
        rep = DerivativeTestReport(num_wrong=torch.empty(N, dtype=i32, device=dev), num_wrong_outside=torch.empty(N, dtype=i32, device=dev),
                                   max_rel_error=torch.empty(N, dtype=f64, device=dev), worst_row=torch.empty(N, dtype=i32, device=dev),
                                   worst_col=torch.empty(N, dtype=i32, device=dev), jac_fd=torch.empty(N, self.nnz, dtype=f64, device=dev),
                                   grad_fd=torch.empty(N, self.n, dtype=f64, device=dev))
        out = _cabi.DerivativeTestOutputs(*[getattr(rep, k).data_ptr() for k in ("num_wrong", "num_wrong_outside", "max_rel_error", "worst_row",
                                                                                 "worst_col", "jac_fd", "grad_fd")])
        opt = _cabi.DerivativeTestOptions(float(perturbation), float(tol))
        pi, keep = self._instance_params(per_instance, N, _cabi.INSTANCE_MAJOR, dev)
        s = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
        with torch.cuda.device(dev):
            _check(self._lib.cplb_derivative_test_device(self._h, N, x.data_ptr(), None if pi is None else C.byref(pi), C.byref(opt),
                                                         C.byref(out), C.c_void_p(s)))
        del keep
        return rep

    # the four ifopt::Problem entry points IpoptAdapter calls, batched
    def EvaluateConstraints(self, x, **kw):
        return self.eval(x, g=True, jac=False, **kw)["g"]

    def EvalNonzerosOfJacobian(self, x, **kw):
        return self.eval(x, g=False, jac=True, **kw)["jac"]

    def EvaluateCostFunction(self, x, **kw):
        return self.eval(x, g=False, jac=False, cost=True, **kw)["cost"]

    def EvaluateCostFunctionGradient(self, x, **kw):
        return self.eval(x, g=False, jac=False, grad=True, **kw)["grad"]

    def GetSolution(self, x_i):
        """CplProblem::GetSolution (src/CplProblem.cpp:85-106) for one instance's x[n]:
        {'com_sol': (3,), 'contact_values_map': {name: {'force_value','position_value','normal_value'}}}
        with the map in sorted-name order like std::map."""
        x_i = np.asarray(x_i, dtype=np.float64).reshape(self.n)
        cv = {}
        for k in self.GetSortedOrder():
            b = 3 + 9 * int(k)
            cv[self._names[k]] = {"force_value": x_i[b:b + 3].copy(), "position_value": x_i[b + 3:b + 6].copy(),
                                  "normal_value": x_i[b + 6:b + 9].copy()}
        return {"com_sol": x_i[0:3].copy(), "contact_values_map": cv}

    @staticmethod
    def FormatSolution(sol):
        """`std::cout << sol` (operator<< of src/CplProblem.cpp:319-346): CoM, then every F_, p_, n_ line in map order.
        Vectors print like an Eigen row with the default IOFormat [M]: '%g' coefficients right-aligned to the widest."""
        def row(v):
            txt = ["%g" % float(c) for c in v]
            w = max(len(t) for t in txt)
            return " ".join(t.rjust(w) for t in txt)

        lines = ["CoM: " + row(sol["com_sol"])]
        for tag, key in (("F_", "force_value"), ("p_", "position_value"), ("n_", "normal_value")):
            lines += [tag + name + ": " + row(v[key]) for name, v in sol["contact_values_map"].items()]
        return "\n".join(lines) + "\n"

    # ---- measurement helpers -----------------------------------------------------------------
    def launch_count(self):
        v = C.c_int64()
        _check(self._lib.cplb_get_launch_count(self._h, C.byref(v)))
        return v.value

    def timing_begin(self):
        _check(self._lib.cplb_timing_begin(self._h))

    def timing_end(self):
        ms, k = C.c_double(), C.c_int64()
        _check(self._lib.cplb_timing_end(self._h, C.byref(ms), C.byref(k)))
        return ms.value, k.value
