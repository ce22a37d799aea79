// cplb/batched_problem.hpp -- C++ host facade over the C ABI (include/cpl_batched.h).
//
// Mirrors the reference's C++ interface for the path so that host code written against
// cpl::solver::CplProblem / cpl::env::{Ground,Superquadric} ports by renaming the namespace:
// same constructor arguments, same setter/getter names, same exception types
// (std::invalid_argument / std::out_of_range / std::runtime_error, see the status mapping below).
// Header-only; links against libcplb.so only.  No Eigen / ifopt needed here (plain arrays);
// the IFOPT component views live in cplb/ifopt_views.hpp.
#ifndef CPLB_BATCHED_PROBLEM_HPP
#define CPLB_BATCHED_PROBLEM_HPP

#include <array>
#include <cstdint>
#include <map>
#include <memory>
#include <ostream>
#include <sstream>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "cpl_batched.h"

namespace cplb {

using Vec3 = std::array<double, 3>;
using Vec6 = std::array<double, 6>;

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// cplb_status -> the exception the reference throws at the same place
inline void check(cplb_status st)
{
    if (st == CPLB_OK) return;
    const std::string msg = cplb_last_error();
    switch (st) {
    case CPLB_INVALID_ARGUMENT: throw std::invalid_argument(msg);
    case CPLB_OUT_OF_RANGE: throw std::out_of_range(msg);
    case CPLB_NULL_POINTER: throw std::invalid_argument(msg);
    case CPLB_CUDA_ERROR: throw CudaError(msg);
    default: throw std::runtime_error(msg);
    }
}

namespace solver {

// cpl::solver::ContactValues / Solution (include/CentroidalPlanner/Ifopt/Types.h:8-21): what CplProblem::GetSolution
// hands back for one instance -- the only "wire format" the reference defines.
struct ContactValues {
    Vec3 force_value;
    Vec3 position_value;
    Vec3 normal_value;
};

struct Solution {
    std::map<std::string, ContactValues> contact_values_map;  // std::map: sorted-name order, like the reference's
    Vec3 com_sol;
};

namespace detail {
// One 3-vector the way `os << v.transpose()` prints an Eigen::Vector3d with the default Eigen::IOFormat [M: Eigen's
// print_matrix -- every coefficient formatted with the stream's own precision/flags, right-aligned to the widest one,
// coefficients separated by one blank]
inline void print_row(std::ostream& os, const Vec3& v)
{
    std::string txt[3];
    size_t width = 0;
    for (int i = 0; i < 3; i++) {
        std::ostringstream one;
        one.copyfmt(os);
        one.width(0);
        one << v[i];
        txt[i] = one.str();
        if (txt[i].size() > width) width = txt[i].size();
    }
    for (int i = 0; i < 3; i++) {
        if (i) os << " ";
        os << std::string(width - txt[i].size(), ' ') << txt[i];
    }
}
}  // namespace detail

// operator<<(std::ostream&, const Solution&) of src/CplProblem.cpp:319-346: CoM, then all forces, all positions, all
// normals, each group in map (sorted-name) order
inline std::ostream& operator<<(std::ostream& os, const Solution& sol)
{
    os << "CoM: ";
    detail::print_row(os, sol.com_sol);
    os << "\n";
    const char* tag[3] = {"F_", "p_", "n_"};
    for (int what = 0; what < 3; what++)
        for (auto& elem : sol.contact_values_map) {
            os << tag[what] + elem.first + ": ";
            detail::print_row(os, what == 0 ? elem.second.force_value : what == 1 ? elem.second.position_value : elem.second.normal_value);
            os << "\n";
        }
    return os;
}

}  // namespace solver

namespace env {

class BatchedProblemAccess;

// cpl::env::EnvironmentClass (include/CentroidalPlanner/Environment/Environment.h:13-48)
class EnvironmentClass {
public:
    typedef std::shared_ptr<EnvironmentClass> Ptr;
    virtual ~EnvironmentClass() = default;
    void SetMu(const double& mu)
    {
        if (mu <= 0.0) throw std::invalid_argument("Invalid friction coefficient");
        _mu = mu;
        Push();
    }
    double GetMu() const { return _mu; }
    virtual cplb_env_kind Kind() const = 0;

    // problems built on this environment see later parameter changes, like the reference's shared_ptr aliasing
    void Attach(cplb_problem* p)
    {
        _attached.push_back(p);
        PushTo(p);
    }
    void Detach(cplb_problem* p)
    {
        for (auto it = _attached.begin(); it != _attached.end(); ++it)
            if (*it == p) {
                _attached.erase(it);
                break;
            }
    }

protected:
    void Push()
    {
        for (auto* p : _attached) PushTo(p);
    }
    virtual void PushTo(cplb_problem* p) { check(cplb_set_mu(p, _mu)); }
    double _mu = 1.0;
    std::vector<cplb_problem*> _attached;
};

// cpl::env::Ground (Ground.h:13-40, src/Ground.cpp)
class Ground : public EnvironmentClass {
public:
    typedef std::shared_ptr<Ground> Ptr;
    void SetGroundZ(const double& ground_z)
    {
        _ground_z = ground_z;
        Push();
    }
    double GetGroundZ() const { return _ground_z; }
    cplb_env_kind Kind() const override { return CPLB_ENV_GROUND; }

protected:
    void PushTo(cplb_problem* p) override
    {
        EnvironmentClass::PushTo(p);
        double z;
        if (cplb_get_ground_z(p, &z) == CPLB_OK) check(cplb_set_ground_z(p, _ground_z));  // not for the _ground_fake of env == nullptr
    }
    double _ground_z = 0.0;
};

// cpl::env::Superquadric (Superquadric.h:13-49, src/Superquadric.cpp:5-37)
class Superquadric : public EnvironmentClass {
public:
    typedef std::shared_ptr<Superquadric> Ptr;
    void SetParameters(const Vec3& C, const Vec3& R, const Vec3& P)
    {
        if ((R[0] <= 0.0) || (R[1] <= 0.0) || (R[2] <= 0.0)) throw std::invalid_argument("Invalid superquadric axial radii");
        if ((P[0] < 2.0) || (P[1] < 2.0) || (P[2] < 2.0))
            throw std::invalid_argument("Invalid superquadric axial curvatures: must be >= 2");
        _C = C;
        _R = R;
        _P = P;
        Push();
    }
    void GetParameters(Vec3& C, Vec3& R, Vec3& P) const
    {
        C = _C;
        R = _R;
        P = _P;
    }
    cplb_env_kind Kind() const override { return CPLB_ENV_SUPERQUADRIC; }

protected:
    void PushTo(cplb_problem* p) override
    {
        EnvironmentClass::PushTo(p);
        check(cplb_set_superquadric(p, _C.data(), _R.data(), _P.data()));
    }
    Vec3 _C{{0.0, 0.0, 10.0}}, _R{{10.0, 10.0, 10.0}}, _P{{10.0, 10.0, 10.0}};
};

}  // namespace env

// One problem shape evaluated for N instances: the batched counterpart of cpl::solver::CplProblem
// (include/CentroidalPlanner/Ifopt/CplProblem.h:19-115).
class BatchedProblem {
public:
    typedef std::shared_ptr<BatchedProblem> Ptr;

    BatchedProblem(std::vector<std::string> contact_names, double robot_mass, env::EnvironmentClass::Ptr env, int device = -1)
        : _contact_names(std::move(contact_names)), _env(std::move(env))
    {
        std::vector<const char*> names;
        for (auto& s : _contact_names) names.push_back(s.c_str());
        check(cplb_create((int32_t)names.size(), names.data(), _env ? _env->Kind() : CPLB_ENV_NONE, robot_mass, device, &_p));
        check(cplb_get_dims(_p, &_n, &_m, &_nnz));
        if (!_env) _ground_fake = std::make_shared<env::Ground>();  // CplProblem.cpp:14
        (_env ? _env : env::EnvironmentClass::Ptr(_ground_fake))->Attach(_p);
    }
    // The same problem sharded over several GPUs of this box (cplb_create_sharded): EvaluateHost / EvaluateHostBegin then cut the
    // batch into one contiguous range per device and drive all of them from the calling thread; device-resident buffers go through
    // EvaluateDeviceShard.
    BatchedProblem(std::vector<std::string> contact_names, double robot_mass, env::EnvironmentClass::Ptr env, const std::vector<int>& devices)
        : _contact_names(std::move(contact_names)), _env(std::move(env))
    {
        std::vector<const char*> names;
        for (auto& s : _contact_names) names.push_back(s.c_str());
        std::vector<int32_t> devs(devices.begin(), devices.end());
        check(cplb_create_sharded((int32_t)names.size(), names.data(), _env ? _env->Kind() : CPLB_ENV_NONE, robot_mass, (int32_t)devs.size(),
                                  devs.data(), &_p));
        check(cplb_get_dims(_p, &_n, &_m, &_nnz));
        if (!_env) _ground_fake = std::make_shared<env::Ground>();  // CplProblem.cpp:14
        (_env ? _env : env::EnvironmentClass::Ptr(_ground_fake))->Attach(_p);
    }
    ~BatchedProblem()
    {
        (_env ? _env : env::EnvironmentClass::Ptr(_ground_fake))->Detach(_p);
        cplb_destroy(_p);
    }
    BatchedProblem(const BatchedProblem&) = delete;
    BatchedProblem& operator=(const BatchedProblem&) = delete;

    cplb_problem* handle() const { return _p; }
    const std::vector<std::string>& contact_names() const { return _contact_names; }
    int GetNumberOfOptimizationVariables() const { return _n; }
    int GetNumberOfConstraints() const { return _m; }
    int GetNumberOfJacobianNonzeros() const { return _nnz; }
    int GetNumberOfShards() const
    {
        int32_t v = 1;
        check(cplb_get_num_shards(_p, &v));
        return v;
    }
    // device ordinal and instance range [begin, end) of one shard for a batch of N instances
    void GetShard(int shard, int64_t N, int& device, int64_t& begin, int64_t& end) const
    {
        int32_t d = -1;
        check(cplb_get_shard(_p, shard, N, &d, &begin, &end));
        device = d;
    }
    bool has_environment() const { return (bool)_env; }

    void GetJacobianStructure(std::vector<int32_t>& iRow, std::vector<int32_t>& jCol) const
    {
        iRow.resize(_nnz);
        jCol.resize(_nnz);
        check(cplb_get_jacobian_structure(_p, iRow.data(), jCol.data()));
    }
    // the x-dependent Jacobian slots in slot order (element q of a CPLB_JAC_PACKED slice is slot map[q]) and the values of the others
    std::vector<int32_t> GetPackedJacobianMap() const
    {
        int32_t nv = 0;
        check(cplb_get_packed_jacobian_map(_p, &nv, nullptr));
        std::vector<int32_t> map((size_t)nv);
        check(cplb_get_packed_jacobian_map(_p, &nv, map.data()));
        return map;
    }
    // where each structural slot's value comes from (cplb_get_jacobian_slot_sources: CPLB_SLOT_* kinds); returns the number of
    // doubles per instance of a CPLB_JAC_COMPUTED slice
    int32_t GetJacobianSlotSources(std::vector<int32_t>& kind, std::vector<int32_t>& source) const
    {
        int32_t nv = 0;
        kind.resize(_nnz);
        source.resize(_nnz);
        check(cplb_get_jacobian_slot_sources(_p, &nv, kind.data(), source.data()));
        return nv;
    }
    void GetJacobianConstants(std::vector<uint8_t>& is_constant, std::vector<double>& value) const
    {
        is_constant.resize(_nnz);
        value.resize(_nnz);
        check(cplb_get_jacobian_constants(_p, is_constant.data(), value.data()));
    }
    std::vector<int32_t> GetSortedOrder() const
    {
        std::vector<int32_t> v(_contact_names.size());
        check(cplb_get_sorted_order(_p, v.data()));
        return v;
    }
    int GetContactRow(const std::string& name) const
    {
        int32_t r;
        check(cplb_get_contact_row(_p, name.c_str(), &r));
        return r;
    }
    int GetBlockColumn(cplb_block block, const std::string& name) const
    {
        int32_t c;
        check(cplb_get_block_column(_p, block, name.c_str(), &c));
        return c;
    }
    void GetBoundsOnOptimizationVariables(std::vector<double>& lb, std::vector<double>& ub) const
    {
        lb.resize(_n);
        ub.resize(_n);
        check(cplb_get_variable_bounds(_p, lb.data(), ub.data()));
    }
    void GetBoundsOnConstraints(std::vector<double>& lb, std::vector<double>& ub) const
    {
        lb.resize(_m);
        ub.resize(_m);
        check(cplb_get_constraint_bounds(_p, lb.data(), ub.data()));
    }

    // ---- the CplProblem forwarders (src/CplProblem.cpp:109-316) ----
    void SetForceBounds(const std::string& n, const Vec3& lb, const Vec3& ub) { check(cplb_set_bounds(_p, CPLB_BLOCK_FORCE, n.c_str(), lb.data(), ub.data())); }
    void GetForceBounds(const std::string& n, Vec3& lb, Vec3& ub) const { check(cplb_get_bounds(_p, CPLB_BLOCK_FORCE, n.c_str(), lb.data(), ub.data())); }
    void SetPosBounds(const std::string& n, const Vec3& lb, const Vec3& ub) { check(cplb_set_bounds(_p, CPLB_BLOCK_POSITION, n.c_str(), lb.data(), ub.data())); }
    void GetPosBounds(const std::string& n, Vec3& lb, Vec3& ub) const { check(cplb_get_bounds(_p, CPLB_BLOCK_POSITION, n.c_str(), lb.data(), ub.data())); }
    void SetNormalBounds(const std::string& n, const Vec3& lb, const Vec3& ub) { check(cplb_set_bounds(_p, CPLB_BLOCK_NORMAL, n.c_str(), lb.data(), ub.data())); }
    void GetNormalBounds(const std::string& n, Vec3& lb, Vec3& ub) const { check(cplb_get_bounds(_p, CPLB_BLOCK_NORMAL, n.c_str(), lb.data(), ub.data())); }
    void SetPosRef(const std::string& n, const Vec3& r) { check(cplb_set_pos_ref(_p, n.c_str(), r.data())); }
    Vec3 GetPosRef(const std::string& n) const { Vec3 r; check(cplb_get_pos_ref(_p, n.c_str(), r.data())); return r; }
    void SetForceRef(const std::string& n, const Vec3& r) { check(cplb_set_force_ref(_p, n.c_str(), r.data())); }
    Vec3 GetForceRef(const std::string& n) const { Vec3 r; check(cplb_get_force_ref(_p, n.c_str(), r.data())); return r; }
    void SetCoMRef(const Vec3& r) { check(cplb_set_com_ref(_p, r.data())); }
    Vec3 GetCoMRef() const { Vec3 r; check(cplb_get_com_ref(_p, r.data())); return r; }
    void SetCoMWeight(double w) { check(cplb_set_com_weight(_p, w)); }
    double GetCoMWeight() const { double w; check(cplb_get_com_weight(_p, &w)); return w; }
    void SetPosWeight(double w) { check(cplb_set_pos_weight(_p, w)); }
    void SetContactPosWeight(const std::string& n, double w) { check(cplb_set_contact_pos_weight(_p, n.c_str(), w)); }
    double GetContactPosWeight(const std::string& n) const { double w; check(cplb_get_contact_pos_weight(_p, n.c_str(), &w)); return w; }
    void SetForceWeight(double w) { check(cplb_set_force_weight(_p, w)); }
    void SetContactForceWeight(const std::string& n, double w) { check(cplb_set_contact_force_weight(_p, n.c_str(), w)); }
    double GetContactForceWeight(const std::string& n) const { double w; check(cplb_get_contact_force_weight(_p, n.c_str(), &w)); return w; }
    void SetManipulationWrench(const Vec6& w) { check(cplb_set_manipulation_wrench(_p, w.data())); }
    Vec6 GetManipulationWrench() const { Vec6 w; check(cplb_get_manipulation_wrench(_p, w.data())); return w; }
    void SetReductionOrder(int order) { check(cplb_set_reduction_order(_p, order)); }  // Eigen 3-term reductions: 0 (default) or 1
    void SetMu(double mu) { (_env ? _env : env::EnvironmentClass::Ptr(_ground_fake))->SetMu(mu); }  // CplProblem.cpp:275-287
    double GetMu() const { return (_env ? _env : env::EnvironmentClass::Ptr(_ground_fake))->GetMu(); }
    void SetForceThreshold(const std::string& n, double t) { check(cplb_set_force_threshold(_p, n.c_str(), t)); }
    double GetForceThreshold(const std::string& n) const { double t; check(cplb_get_force_threshold(_p, n.c_str(), &t)); return t; }

    // CplProblem::GetSolution (src/CplProblem.cpp:85-106) for one instance's x[n]: unpack by the column map
    // (CoM 0..2; contact k of the caller's vector: F 3+9k, p +3, n +6) into the name-keyed map
    void GetSolution(const double* x_i, solver::Solution& sol) const
    {
        for (int c = 0; c < 3; c++) sol.com_sol[c] = x_i[c];
        for (size_t k = 0; k < _contact_names.size(); k++) {
            const double* b = x_i + 3 + 9 * k;
            solver::ContactValues v;
            for (int c = 0; c < 3; c++) {
                v.force_value[c] = b[c];
                v.position_value[c] = b[3 + c];
                v.normal_value[c] = b[6 + c];
            }
            sol.contact_values_map[_contact_names[k]] = v;
        }
    }

    // ---- evaluation (host buffers, instance-major: instance i owns x[i*n..], g[i*m..], jac[i*nnz..]) ----
    // per_instance: optional per-instance parameter arrays (host pointers, instance-major), nullptr = shared parameters
    // host_flags: 0, CPLB_JAC_PACKED (jac then holds GetPackedJacobianMap().size() doubles per instance: the x-dependent slots only)
    // or CPLB_JAC_COMPUTED (GetJacobianSlotSources(): only the slots that take arithmetic)
    void EvaluateHost(int64_t N, const double* x, double* g, double* jac, double* cost, double* grad,
                      const cplb_instance_params* per_instance = nullptr, int32_t host_flags = 0)
    {
        cplb_eval_args a{};
        a.num_instances = N;
        a.host_flags = host_flags;
        a.layout = CPLB_INSTANCE_MAJOR;
        a.x = x;
        a.g = g;
        a.jac = jac;
        a.cost = cost;
        a.grad = grad;
        a.per_instance = per_instance;
        check(cplb_eval_host(_p, &a));
    }
    // the same for a queue of batches: Begin enqueues and returns a ticket, Wait returns when that batch's outputs have landed
    // (pinned host buffers, untouched in between; cplb_eval_host_begin / cplb_eval_host_wait)
    int32_t EvaluateHostBegin(int64_t N, const double* x, double* g, double* jac, double* cost, double* grad,
                              const cplb_instance_params* per_instance = nullptr, int32_t host_flags = 0)
    {
        cplb_eval_args a{};
        a.num_instances = N;
        a.host_flags = host_flags;
        a.layout = CPLB_INSTANCE_MAJOR;
        a.x = x;
        a.g = g;
        a.jac = jac;
        a.cost = cost;
        a.grad = grad;
        a.per_instance = per_instance;
        int32_t ticket = -1;
        check(cplb_eval_host_begin(_p, &a, &ticket));
        return ticket;
    }
    void EvaluateHostWait(int32_t ticket) { check(cplb_eval_host_wait(_p, ticket)); }
    // device buffers, either layout, asynchronous on `stream`
    void EvaluateDevice(int64_t N, cplb_layout layout, int64_t ld, const double* x, double* g, double* jac, double* cost,
                        double* grad, void* stream, const cplb_instance_params* per_instance = nullptr)
    {
        cplb_eval_args a{};
        a.num_instances = N;
        a.layout = layout;
        a.ld = ld;
        a.x = x;
        a.g = g;
        a.jac = jac;
        a.cost = cost;
        a.grad = grad;
        a.per_instance = per_instance;
        check(cplb_eval_device(_p, &a, stream));
    }

    // one shard's device-resident buffers (its instances only) on that shard's device and stream
    void EvaluateDeviceShard(int shard, int64_t N, cplb_layout layout, int64_t ld, const double* x, double* g, double* jac, double* cost,
                             double* grad, void* stream, const cplb_instance_params* per_instance = nullptr)
    {
        cplb_eval_args a{};
        a.num_instances = N;
        a.layout = layout;
        a.ld = ld;
        a.x = x;
        a.g = g;
        a.jac = jac;
        a.cost = cost;
        a.grad = grad;
        a.per_instance = per_instance;
        check(cplb_eval_device_shard(_p, shard, &a, stream));
    }

    // N lock-step solves on the GPU (cplb_solve_device): the batched counterpart of cpl::CentroidalPlanner::Solve
    // (src/CentroidalPlanner.cpp:22-34); all pointers are device pointers, lam may be nullptr.  NOT IPOPT (see the C header).
    struct SolveCounters {
        int32_t rounds = 0;
        int64_t evaluations = 0, instance_evaluations = 0, tail_instances = 0;
    };
    SolveCounters SolveDevice(int64_t N, const double* x0, double* x, int32_t* status, int32_t* iterations, double* cost, double* constr_viol,
                              double* dual_inf, double* lam, void* stream, const cplb_solver_options* options = nullptr,
                              const cplb_instance_params* per_instance = nullptr)
    {
        SolveCounters c;
        cplb_solve_outputs out{};
        out.x = x;
        out.status = status;
        out.iterations = iterations;
        out.cost = cost;
        out.constr_viol = constr_viol;
        out.dual_inf = dual_inf;
        out.lam = lam;
        out.rounds = &c.rounds;
        out.evaluations = &c.evaluations;
        out.instance_evaluations = &c.instance_evaluations;
        out.tail_instances = &c.tail_instances;
        check(cplb_solve_device(_p, N, x0, per_instance, options, &out, stream));
        return c;
    }

    // IPOPT's first-order derivative test for N instances at x (cplb_derivative_test_device): what `derivative_test first-order`
    // checks before every solve of the reference (src/CentroidalPlanner.cpp:26).  Device pointers; any output may be nullptr;
    // asynchronous on `stream`.
    void DerivativeTestDevice(int64_t N, const double* x, const cplb_derivative_test_outputs& out, void* stream,
                              const cplb_derivative_test_options* options = nullptr, const cplb_instance_params* per_instance = nullptr)
    {
        check(cplb_derivative_test_device(_p, N, x, per_instance, options, &out, stream));
    }

    // Products with the Jacobian at x without materialising it (cplb_jacobian_products_device): x_bar = obj_factor * grad f +
    // J^T lambda and/or g_dot = J v, f_dot = grad f . v.  Device pointers in `args`; asynchronous on `stream`.
    void JacobianProductsDevice(const cplb_jacobian_products_args& args, void* stream) { check(cplb_jacobian_products_device(_p, &args, stream)); }

private:
    std::vector<std::string> _contact_names;
    env::EnvironmentClass::Ptr _env;
    std::shared_ptr<env::Ground> _ground_fake;
    cplb_problem* _p = nullptr;
    int32_t _n = 0, _m = 0, _nnz = 0;
};

}  // namespace cplb
#endif
