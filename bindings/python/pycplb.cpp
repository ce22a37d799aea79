// bindings/python/pycplb.cpp -- pybind11 module over the SAME C ABI (include/cpl_batched.h), through the C++ facade
// (cplb/batched_problem.hpp).  Successor of the reference's bindings/python/pyCpl.cpp:12-71, which binds only the
// planner facade: this one binds the environments with the reference's class/method names and the array-level
// batched evaluation.  Exceptions map like pybind11 maps the reference's: std::invalid_argument -> ValueError,
// std::out_of_range -> IndexError, std::runtime_error -> RuntimeError.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cplb/batched_problem.hpp>

namespace py = pybind11;
using cplb::Vec3;
using cplb::Vec6;
using darray = py::array_t<double, py::array::c_style | py::array::forcecast>;

static Vec3 v3(const std::vector<double>& v)
{
    if (v.size() != 3) throw std::invalid_argument("expected 3 values");
    return Vec3{{v[0], v[1], v[2]}};
}

PYBIND11_MODULE(pycplb, m)
{
    m.doc() = "B200 batched evaluator for CentroidalPlanner's IFOPT problem (pybind11 over the cplb C ABI)";

    py::class_<cplb::env::EnvironmentClass, cplb::env::EnvironmentClass::Ptr>(m, "EnvironmentClass")
        .def("SetMu", &cplb::env::EnvironmentClass::SetMu)
        .def("GetMu", &cplb::env::EnvironmentClass::GetMu);
    py::class_<cplb::env::Ground, cplb::env::EnvironmentClass, cplb::env::Ground::Ptr>(m, "Ground")  // pyCpl.cpp:21-24
        .def(py::init<>())
        .def("SetGroundZ", &cplb::env::Ground::SetGroundZ)
        .def("GetGroundZ", &cplb::env::Ground::GetGroundZ);
    py::class_<cplb::env::Superquadric, cplb::env::EnvironmentClass, cplb::env::Superquadric::Ptr>(m, "Superquadric")  // pyCpl.cpp:26-29
        .def(py::init<>())
        .def("SetParameters", [](cplb::env::Superquadric& s, std::vector<double> C, std::vector<double> R, std::vector<double> P) {
            s.SetParameters(v3(C), v3(R), v3(P));
        })
        .def("GetParameters", [](const cplb::env::Superquadric& s) {
            Vec3 C, R, P;
            s.GetParameters(C, R, P);
            return py::make_tuple(C, R, P);
        });

    py::class_<cplb::BatchedProblem, cplb::BatchedProblem::Ptr>(m, "BatchedProblem")
        .def(py::init<std::vector<std::string>, double, cplb::env::EnvironmentClass::Ptr, int>(), py::arg("contact_names"),
             py::arg("robot_mass"), py::arg("env") = cplb::env::EnvironmentClass::Ptr(), py::arg("device") = -1)
        // the same problem sharded over several GPUs of the box (cplb_create_sharded)
        .def(py::init([](std::vector<std::string> names, double mass, cplb::env::EnvironmentClass::Ptr env, std::vector<int> devices) {
                 return std::make_shared<cplb::BatchedProblem>(std::move(names), mass, std::move(env), devices);
             }),
             py::arg("contact_names"), py::arg("robot_mass"), py::arg("env"), py::arg("devices"))
        .def("GetNumberOfShards", &cplb::BatchedProblem::GetNumberOfShards)
        .def("GetShard", [](const cplb::BatchedProblem& p, int shard, int64_t N) {
            int device = -1;
            int64_t b = 0, e = 0;
            p.GetShard(shard, N, device, b, e);
            return py::make_tuple(device, b, e);
        })
        .def("GetPackedJacobianMap", [](const cplb::BatchedProblem& p) {
            const std::vector<int32_t> m = p.GetPackedJacobianMap();
            return py::array_t<int32_t>(m.size(), m.data());
        })
        .def("GetJacobianSlotSources", [](const cplb::BatchedProblem& p) {
            std::vector<int32_t> kind, source;
            p.GetJacobianSlotSources(kind, source);
            return py::make_tuple(py::array_t<int32_t>(kind.size(), kind.data()), py::array_t<int32_t>(source.size(), source.data()));
        })
        .def_property_readonly("n", &cplb::BatchedProblem::GetNumberOfOptimizationVariables)
        .def_property_readonly("m", &cplb::BatchedProblem::GetNumberOfConstraints)
        .def_property_readonly("nnz", &cplb::BatchedProblem::GetNumberOfJacobianNonzeros)
        .def("GetJacobianStructure", [](const cplb::BatchedProblem& p) {
            std::vector<int32_t> r, c;
            p.GetJacobianStructure(r, c);
            return py::make_tuple(py::array_t<int32_t>(r.size(), r.data()), py::array_t<int32_t>(c.size(), c.data()));
        })
        .def("GetSortedOrder", &cplb::BatchedProblem::GetSortedOrder)
        .def("GetBoundsOnConstraints", [](const cplb::BatchedProblem& p) {
            std::vector<double> l, u;
            p.GetBoundsOnConstraints(l, u);
            return py::make_tuple(l, u);
        })
        .def("GetBoundsOnOptimizationVariables", [](const cplb::BatchedProblem& p) {
            std::vector<double> l, u;
            p.GetBoundsOnOptimizationVariables(l, u);
            return py::make_tuple(l, u);
        })
        .def("SetForceBounds", [](cplb::BatchedProblem& p, const std::string& n, std::vector<double> l, std::vector<double> u) { p.SetForceBounds(n, v3(l), v3(u)); })
        .def("SetPosBounds", [](cplb::BatchedProblem& p, const std::string& n, std::vector<double> l, std::vector<double> u) { p.SetPosBounds(n, v3(l), v3(u)); })
        .def("SetNormalBounds", [](cplb::BatchedProblem& p, const std::string& n, std::vector<double> l, std::vector<double> u) { p.SetNormalBounds(n, v3(l), v3(u)); })
        .def("SetPosRef", [](cplb::BatchedProblem& p, const std::string& n, std::vector<double> r) { p.SetPosRef(n, v3(r)); })
        .def("GetPosRef", &cplb::BatchedProblem::GetPosRef)
        .def("SetForceRef", [](cplb::BatchedProblem& p, const std::string& n, std::vector<double> r) { p.SetForceRef(n, v3(r)); })
        .def("GetForceRef", &cplb::BatchedProblem::GetForceRef)
        .def("SetCoMRef", [](cplb::BatchedProblem& p, std::vector<double> r) { p.SetCoMRef(v3(r)); })
        .def("GetCoMRef", &cplb::BatchedProblem::GetCoMRef)
        .def("SetCoMWeight", &cplb::BatchedProblem::SetCoMWeight)
        .def("GetCoMWeight", &cplb::BatchedProblem::GetCoMWeight)
        .def("SetPosWeight", &cplb::BatchedProblem::SetPosWeight)
        .def("SetContactPosWeight", &cplb::BatchedProblem::SetContactPosWeight)
        .def("GetContactPosWeight", &cplb::BatchedProblem::GetContactPosWeight)
        .def("SetForceWeight", &cplb::BatchedProblem::SetForceWeight)
        .def("SetContactForceWeight", &cplb::BatchedProblem::SetContactForceWeight)
        .def("GetContactForceWeight", &cplb::BatchedProblem::GetContactForceWeight)
        .def("SetManipulationWrench", [](cplb::BatchedProblem& p, std::vector<double> w) {
            if (w.size() != 6) throw std::invalid_argument("expected 6 values");
            p.SetManipulationWrench(Vec6{{w[0], w[1], w[2], w[3], w[4], w[5]}});
        })
        .def("GetManipulationWrench", &cplb::BatchedProblem::GetManipulationWrench)
        .def("SetReductionOrder", &cplb::BatchedProblem::SetReductionOrder)
        .def("SetMu", &cplb::BatchedProblem::SetMu)
        .def("GetMu", &cplb::BatchedProblem::GetMu)
        .def("SetForceThreshold", &cplb::BatchedProblem::SetForceThreshold)
        .def("GetForceThreshold", &cplb::BatchedProblem::GetForceThreshold)
        // host arrays, instance-major: x (N, n) -> dict of (N, m), (N, nnz), (N,), (N, n)
        .def("eval", [](cplb::BatchedProblem& p, darray x, bool g, bool jac, bool cost, bool grad, int jac_packed) {
            // jac_packed: 0 full rows, 1 (True) CPLB_JAC_PACKED slices, 2 CPLB_JAC_COMPUTED slices
            if (jac_packed < 0 || jac_packed > 2) throw std::invalid_argument("jac_packed must be 0, 1 or 2");
            if (x.ndim() != 2 || x.shape(1) != p.GetNumberOfOptimizationVariables()) throw std::invalid_argument("x must be (N, n)");
            const py::ssize_t N = x.shape(0);
            py::dict out;
            darray ag, aj, ac, agr;
            if (g) ag = darray({N, (py::ssize_t)p.GetNumberOfConstraints()});
            if (jac) {
                py::ssize_t len = (py::ssize_t)p.GetNumberOfJacobianNonzeros();
                if (jac_packed == 1) len = (py::ssize_t)p.GetPackedJacobianMap().size();
                if (jac_packed == 2) {
                    std::vector<int32_t> kind, source;
                    len = (py::ssize_t)p.GetJacobianSlotSources(kind, source);
                }
                aj = darray({N, len});
            }
            if (cost) ac = darray({N});
            if (grad) agr = darray({N, (py::ssize_t)p.GetNumberOfOptimizationVariables()});
            {
                py::gil_scoped_release nogil;
                p.EvaluateHost(N, x.data(), g ? ag.mutable_data() : nullptr, jac ? aj.mutable_data() : nullptr,
                               cost ? ac.mutable_data() : nullptr, grad ? agr.mutable_data() : nullptr, nullptr,
                               jac_packed == 2 ? CPLB_JAC_COMPUTED : (jac_packed == 1 ? CPLB_JAC_PACKED : 0));
            }
            out["g"] = g ? py::object(ag) : py::none();
            out["jac"] = jac ? py::object(aj) : py::none();
            out["cost"] = cost ? py::object(ac) : py::none();
            out["grad"] = grad ? py::object(agr) : py::none();
            return out;
        }, py::arg("x"), py::arg("g") = true, py::arg("jac") = true, py::arg("cost") = false, py::arg("grad") = false, py::arg("jac_packed") = 0)
        // raw device pointers of ONE shard of a sharded problem, on that shard's device and stream
        .def("eval_device_shard", [](cplb::BatchedProblem& p, int shard, int64_t N, int layout, int64_t ld, uintptr_t x, uintptr_t g,
                                     uintptr_t jac, uintptr_t cost, uintptr_t grad, uintptr_t stream) {
            p.EvaluateDeviceShard(shard, N, (cplb_layout)layout, ld, reinterpret_cast<const double*>(x), reinterpret_cast<double*>(g),
                                  reinterpret_cast<double*>(jac), reinterpret_cast<double*>(cost), reinterpret_cast<double*>(grad),
                                  reinterpret_cast<void*>(stream));
        }, py::arg("shard"), py::arg("num_instances"), py::arg("layout"), py::arg("ld"), py::arg("x"), py::arg("g") = 0, py::arg("jac") = 0,
             py::arg("cost") = 0, py::arg("grad") = 0, py::arg("stream") = 0)
        // N lock-step solves on the GPU (cplb_solve_device); every array argument is a raw device pointer
        .def("solve_device", [](cplb::BatchedProblem& p, int64_t N, uintptr_t x0, uintptr_t x, uintptr_t status, uintptr_t iterations,
                                uintptr_t cost, uintptr_t constr_viol, uintptr_t dual_inf, uintptr_t lam, uintptr_t stream, double tol, int max_iter) {
            cplb_solver_options o;
            cplb_solver_default_options(&o);
            o.tol = tol;
            o.max_iter = max_iter;
            cplb::BatchedProblem::SolveCounters c;
            {
                py::gil_scoped_release nogil;
                c = p.SolveDevice(N, reinterpret_cast<const double*>(x0), reinterpret_cast<double*>(x), reinterpret_cast<int32_t*>(status),
                                  reinterpret_cast<int32_t*>(iterations), reinterpret_cast<double*>(cost), reinterpret_cast<double*>(constr_viol),
                                  reinterpret_cast<double*>(dual_inf), reinterpret_cast<double*>(lam), reinterpret_cast<void*>(stream), &o);
            }
            return py::make_tuple(c.rounds, c.evaluations, c.instance_evaluations);
        }, py::arg("num_instances"), py::arg("x0"), py::arg("x"), py::arg("status"), py::arg("iterations"), py::arg("cost"),
             py::arg("constr_viol"), py::arg("dual_inf"), py::arg("lam") = 0, py::arg("stream") = 0, py::arg("tol") = 1e-3, py::arg("max_iter") = 500)
        // first-order derivative test at x (cplb_derivative_test_device); every array argument is a raw device pointer (0 = not wanted)
        .def("derivative_test_device", [](cplb::BatchedProblem& p, int64_t N, uintptr_t x, uintptr_t num_wrong, uintptr_t num_wrong_outside,
                                          uintptr_t max_rel_error, uintptr_t worst_row, uintptr_t worst_col, uintptr_t jac_fd, uintptr_t grad_fd,
                                          uintptr_t stream, double perturbation, double tol) {
            cplb_derivative_test_options o{perturbation, tol};
            cplb_derivative_test_outputs out{reinterpret_cast<int32_t*>(num_wrong), reinterpret_cast<int32_t*>(num_wrong_outside),
                                             reinterpret_cast<double*>(max_rel_error), reinterpret_cast<int32_t*>(worst_row),
                                             reinterpret_cast<int32_t*>(worst_col), reinterpret_cast<double*>(jac_fd), reinterpret_cast<double*>(grad_fd)};
            py::gil_scoped_release nogil;
            p.DerivativeTestDevice(N, reinterpret_cast<const double*>(x), out, reinterpret_cast<void*>(stream), &o);
        }, py::arg("num_instances"), py::arg("x"), py::arg("num_wrong") = 0, py::arg("num_wrong_outside") = 0, py::arg("max_rel_error") = 0,
             py::arg("worst_row") = 0, py::arg("worst_col") = 0, py::arg("jac_fd") = 0, py::arg("grad_fd") = 0, py::arg("stream") = 0,
             py::arg("perturbation") = 1e-8, py::arg("tol") = 1e-4)
        // Jacobian products at x (cplb_jacobian_products_device); raw device pointers, instance-major (0 = NULL)
        .def("jacobian_products_device", [](cplb::BatchedProblem& p, int64_t N, uintptr_t x, uintptr_t lam, uintptr_t obj_factor, uintptr_t x_bar,
                                            uintptr_t v, uintptr_t g_dot, uintptr_t f_dot, uintptr_t stream) {
            const cplb_jacobian_products_args a{N, reinterpret_cast<const double*>(x), nullptr, reinterpret_cast<const double*>(lam),
                                                reinterpret_cast<const double*>(obj_factor), reinterpret_cast<double*>(x_bar),
                                                reinterpret_cast<const double*>(v), reinterpret_cast<double*>(g_dot), reinterpret_cast<double*>(f_dot)};
            py::gil_scoped_release nogil;
            p.JacobianProductsDevice(a, reinterpret_cast<void*>(stream));
        }, py::arg("num_instances"), py::arg("x"), py::arg("lam") = 0, py::arg("obj_factor") = 0, py::arg("x_bar") = 0, py::arg("v") = 0,
             py::arg("g_dot") = 0, py::arg("f_dot") = 0, py::arg("stream") = 0)
        // raw device pointers (e.g. torch.Tensor.data_ptr()), either layout, asynchronous on `stream`
        .def("eval_device", [](cplb::BatchedProblem& p, int64_t N, int layout, int64_t ld, uintptr_t x, uintptr_t g, uintptr_t jac,
                               uintptr_t cost, uintptr_t grad, uintptr_t stream) {
            p.EvaluateDevice(N, (cplb_layout)layout, ld, reinterpret_cast<const double*>(x), reinterpret_cast<double*>(g),
                             reinterpret_cast<double*>(jac), reinterpret_cast<double*>(cost), reinterpret_cast<double*>(grad),
                             reinterpret_cast<void*>(stream));
        }, py::arg("num_instances"), py::arg("layout"), py::arg("ld"), py::arg("x"), py::arg("g") = 0, py::arg("jac") = 0,
             py::arg("cost") = 0, py::arg("grad") = 0, py::arg("stream") = 0);

    m.attr("INSTANCE_MAJOR") = (int)CPLB_INSTANCE_MAJOR;
    m.attr("COMPONENT_MAJOR") = (int)CPLB_COMPONENT_MAJOR;
    py::register_exception<cplb::CudaError>(m, "CudaError", PyExc_RuntimeError);
}
