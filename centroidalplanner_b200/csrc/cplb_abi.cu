// cplb_abi.cu -- implementation of the C ABI declared in include/cpl_batched.h.
// Host-only code (parameter bookkeeping with the reference's validation predicates, layout, the
// host<->device pipeline); the arithmetic lives in cplb_kernels.cu.  There is NO CPU evaluation
// path in this library: without a CUDA device every evaluation fails with CPLB_CUDA_ERROR.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "cpl_batched.h"
#include "cplb_derivtest.h"
#include "cplb_kernels.h"
#include "cplb_layout.hpp"
#include "cplb_params.h"
#include "cplb_products.h"
#include "cplb_solver.h"

namespace {

thread_local char g_last_error[512] = "";

cplb_status fail(cplb_status st, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof g_last_error, fmt, ap);
    va_end(ap);
    return st;
}

cplb_status cuda_fail(cudaError_t e, const char* what)
{
    return fail(CPLB_CUDA_ERROR, "%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
}

#define CPLB_CUDA(call)                                      \
    do {                                                     \
        cudaError_t e__ = (call);                            \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

#define CPLB_REQUIRE(ptr)                                                          \
    do {                                                                           \
        if ((ptr) == nullptr) return fail(CPLB_NULL_POINTER, "%s is NULL", #ptr); \
    } while (0)

constexpr int kHostStreams = 3;
constexpr int kHostTickets = 4;  // asynchronous host calls that may be outstanding at once

struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

}  // namespace

struct cplb_problem {
    std::vector<std::string> names;
    cplb_env_kind env = CPLB_ENV_NONE;
    int device = 0;
    double mass = 100.0;
    double sqC[3] = {0.0, 0.0, 10.0}, sqR[3] = {10.0, 10.0, 10.0}, sqP[3] = {10.0, 10.0, 10.0};
    cplb::Layout layout;
    CplbParams P{};
    std::vector<double> x_lb, x_ub;
    std::atomic<long long> launches{0};
    int cm_kernel = CPLB_CM_AUTO;  // cplb_set_component_major_kernel
    int im_kernel = CPLB_IM_AUTO;  // cplb_set_instance_major_kernel

    // kernel timing (cplb_timing_begin/end)
    std::mutex timing_mu;
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> events;

    // cplb_eval_host pipeline, one per device of the problem (cplb_create: one; cplb_create_sharded: one per shard)
    struct HostPipe {
        int device = -1;
        cudaStream_t streams[kHostStreams] = {};
        double* stage[kHostStreams] = {};
        double* bounce[kHostStreams] = {};  // pinned mirrors of stage[], used when the caller's buffers are pageable
        size_t bounce_bytes = 0;
        size_t stage_bytes = 0;
        bool streams_ready = false;
        // cplb_eval_host_begin / _wait: completion events of the outstanding asynchronous calls (ring of tickets)
        cudaEvent_t host_done[kHostTickets][kHostStreams] = {};
        bool host_done_ready = false;
        int next_stream = 0;
    };
    std::mutex host_mu;
    std::vector<HostPipe> pipes;  // pipes[0].device mirrors `device` for a single-device problem
    bool sharded = false;
    int next_ticket = 0;

    // cplb_solve_device: device slabs of the native solve round (grown on demand, freed with the problem)
    std::mutex solver_mu;
    cplb::solver::Workspace* solver_ws = nullptr;

    // cplb_derivative_test_device: structural slot of every dense Jacobian entry (row-major m x n, -1 outside the structure),
    // uploaded at the first call (the structure never changes after creation)
    std::mutex derivtest_mu;
    int32_t* slot_of = nullptr;

    int find(const char* name) const
    {
        if (!name) return -1;
        for (size_t k = 0; k < names.size(); k++)
            if (names[k] == name) return (int)k;
        return -1;
    }

    void refresh_derived()
    {
        // _m * _g with _g = (0, 0, -9.81) (CentroidalStatics.cpp:15,57): one multiply per component
        const double g[3] = {0.0, 0.0, -9.81};
        for (int i = 0; i < 3; i++) P.mg[i] = mass * g[i];
        P.mass = mass;
        for (int q = 0; q < 3; q++) {
            P.sqC[q] = sqC[q];
            P.sqR[q] = sqR[q];
            P.sqP[q] = sqP[q];
            const double twoP = sqP[q] * 2.0;
            P.sqPoverRP[q] = sqP[q] / std::pow(sqR[q], sqP[q]);
            P.sqRmP[q] = std::pow(sqR[q], -sqP[q]);
            P.sqRm2P[q] = std::pow(sqR[q], -twoP);
            P.sqR2P[q] = std::pow(sqR[q], twoP);
        }
        // integer-curvature fast path of the kernels (cplb_device.cuh, superquadric())
        bool ints = true;
        double pmax = 0.0;
        for (int q = 0; q < 3; q++) {
            ints = ints && sqP[q] >= 2.0 && sqP[q] <= 63.0 && sqP[q] == std::floor(sqP[q]);
            pmax = sqP[q] > pmax ? sqP[q] : pmax;
        }
        for (int q = 0; q < 3; q++) P.sqIntP[q] = ints ? (int)sqP[q] : 0;
        int bits = 0;
        for (int e = ints ? (int)pmax - 2 : 0; e > 0; e >>= 1) bits++;  // largest chain exponent is P - 2
        P.sqBits = bits;
        P.sqWindow = ints ? (int)(900.0 / (2.0 * pmax)) : 0;
    }
};

extern "C" {

const char* cplb_last_error(void) { return g_last_error; }
int32_t cplb_abi_version(void) { return CPLB_ABI_VERSION; }

static cplb_status create_impl(int32_t num_contacts, const char* const* contact_names, cplb_env_kind env, double robot_mass,
                               int32_t num_devices, const int32_t* devices, bool sharded, cplb_problem** out)
{
    CPLB_REQUIRE(out);
    *out = nullptr;
    CPLB_REQUIRE(contact_names);
    if (num_contacts < 1) return fail(CPLB_INVALID_ARGUMENT, "at least one contact is required");
    if (num_contacts > CPLB_MAX_CONTACTS)
        return fail(CPLB_INVALID_ARGUMENT, "at most %d contacts are supported (got %d)", CPLB_MAX_CONTACTS, num_contacts);
    if (env != CPLB_ENV_NONE && env != CPLB_ENV_GROUND && env != CPLB_ENV_SUPERQUADRIC)
        return fail(CPLB_INVALID_ARGUMENT, "unknown environment kind %d", (int)env);
    if (!(robot_mass > 0.0)) return fail(CPLB_INVALID_ARGUMENT, "Invalid robot mass");  // CentroidalPlanner.cpp:12-15

    bool any_explicit = false;
    for (int d = 0; d < num_devices; d++) any_explicit = any_explicit || devices[d] >= 0;
    if (any_explicit) {  // explicit ordinals are validated now; -1 binds to the caller's current device at first evaluation
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            return fail(CPLB_CUDA_ERROR, "no usable CUDA device (%s); this library has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        for (int d = 0; d < num_devices; d++) {
            if (devices[d] >= ndev) return fail(CPLB_INVALID_ARGUMENT, "device %d out of range (%d devices)", devices[d], ndev);
            if (sharded && devices[d] < 0) return fail(CPLB_INVALID_ARGUMENT, "a sharded problem needs explicit device ordinals (devices[%d] = %d)", d, devices[d]);
        }
    } else if (sharded) {
        return fail(CPLB_INVALID_ARGUMENT, "a sharded problem needs explicit device ordinals");
    }

    cplb_problem* p = new (std::nothrow) cplb_problem();
    if (!p) return fail(CPLB_RUNTIME_ERROR, "out of host memory");
    for (int k = 0; k < num_contacts; k++) {
        if (!contact_names[k]) {
            delete p;
            return fail(CPLB_NULL_POINTER, "contact_names[%d] is NULL", k);
        }
        if (p->find(contact_names[k]) >= 0) {
            delete p;
            return fail(CPLB_INVALID_ARGUMENT, "duplicate contact name '%s'", contact_names[k]);
        }
        p->names.emplace_back(contact_names[k]);
    }
    p->env = env;
    p->device = devices[0];
    p->sharded = sharded;
    p->pipes.resize((size_t)num_devices);
    for (int d = 0; d < num_devices; d++) p->pipes[(size_t)d].device = devices[d];
    p->mass = robot_mass;
    p->layout.build(p->names, env != CPLB_ENV_NONE, env == CPLB_ENV_GROUND);

    CplbParams& P = p->P;
    std::memset(&P, 0, sizeof P);
    P.nc = num_contacts;
    P.env = (int)env;
    P.n = p->layout.n;
    P.m = p->layout.m;
    P.nnz = p->layout.nnz;
    for (int j = 0; j < num_contacts; j++) P.perm[j] = p->layout.perm[j];
    P.mu = 1.0;          // Environment.h:46
    P.ground_z = 0.0;    // Ground.cpp:7
    P.com_ref[2] = 1.0;  // MinimizeCentroidalVariables.cpp:11
    P.W_com = 1.0;       // :13
    for (int k = 0; k < num_contacts; k++) {
        P.W_p[k] = 1.0;  // :24-25
        P.W_F[k] = 1.0;
    }
    p->refresh_derived();
    p->x_lb.assign(P.n, -1000.0);  // Variable3D.cpp:12-13
    p->x_ub.assign(P.n, 1000.0);
    *out = p;
    return CPLB_OK;
}

cplb_status cplb_create(int32_t num_contacts, const char* const* contact_names, cplb_env_kind env, double robot_mass,
                        int32_t device, cplb_problem** out)
{
    return create_impl(num_contacts, contact_names, env, robot_mass, 1, &device, false, out);
}

cplb_status cplb_create_sharded(int32_t num_contacts, const char* const* contact_names, cplb_env_kind env, double robot_mass,
                                int32_t num_devices, const int32_t* devices, cplb_problem** out)
{
    CPLB_REQUIRE(out);
    *out = nullptr;
    CPLB_REQUIRE(devices);
    if (num_devices < 1 || num_devices > CPLB_MAX_SHARDS)
        return fail(CPLB_INVALID_ARGUMENT, "num_devices must be in 1..%d (got %d)", CPLB_MAX_SHARDS, (int)num_devices);
    return create_impl(num_contacts, contact_names, env, robot_mass, num_devices, devices, true, out);
}

void cplb_destroy(cplb_problem* p)
{
    if (!p) return;
    if (p->device >= 0) {
        DeviceGuard dg(p->device);
        for (auto& ev : p->events) {
            cudaEventDestroy(ev.first);
            cudaEventDestroy(ev.second);
        }
    }
    if (p->solver_ws) {
        DeviceGuard dg(p->device >= 0 ? p->device : 0);
        cplb::solver::workspace_free(p->solver_ws);
    }
    if (p->slot_of) {
        DeviceGuard dg(p->device);
        cudaFree(p->slot_of);
    }
    for (auto& pipe : p->pipes) {
        if (pipe.device < 0 || !pipe.streams_ready) continue;
        DeviceGuard dg(pipe.device);
        if (pipe.host_done_ready)
            for (int t = 0; t < kHostTickets; t++)
                for (int s = 0; s < kHostStreams; s++) cudaEventDestroy(pipe.host_done[t][s]);
        for (int s = 0; s < kHostStreams; s++) {
            cudaStreamSynchronize(pipe.streams[s]);
            cudaStreamDestroy(pipe.streams[s]);
            if (pipe.stage[s]) cudaFree(pipe.stage[s]);
            if (pipe.bounce[s]) cudaFreeHost(pipe.bounce[s]);
        }
    }
    delete p;
}

// ---- layout ---------------------------------------------------------------------------------

cplb_status cplb_get_dims(const cplb_problem* p, int32_t* n, int32_t* m, int32_t* nnz)
{
    CPLB_REQUIRE(p);
    if (n) *n = p->layout.n;
    if (m) *m = p->layout.m;
    if (nnz) *nnz = p->layout.nnz;
    return CPLB_OK;
}

cplb_status cplb_get_jacobian_structure(const cplb_problem* p, int32_t* iRow, int32_t* jCol)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(iRow);
    CPLB_REQUIRE(jCol);
    std::memcpy(iRow, p->layout.iRow.data(), sizeof(int32_t) * p->layout.nnz);
    std::memcpy(jCol, p->layout.jCol.data(), sizeof(int32_t) * p->layout.nnz);
    return CPLB_OK;
}

cplb_status cplb_get_sorted_order(const cplb_problem* p, int32_t* sorted_to_vector)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(sorted_to_vector);
    for (int j = 0; j < p->layout.nc; j++) sorted_to_vector[j] = p->layout.perm[j];
    return CPLB_OK;
}

static cplb_status block_column(const cplb_problem* p, cplb_block block, const char* name, int* col)
{
    if (block == CPLB_BLOCK_COM) {
        *col = 0;
        return CPLB_OK;
    }
    if (block != CPLB_BLOCK_FORCE && block != CPLB_BLOCK_POSITION && block != CPLB_BLOCK_NORMAL)
        return fail(CPLB_INVALID_ARGUMENT, "unknown variable block %d", (int)block);
    const int k = p->find(name);
    if (k < 0) return fail(CPLB_OUT_OF_RANGE, "map::at: unknown contact '%s'", name ? name : "(null)");
    *col = 3 + 9 * k + 3 * ((int)block - 1);
    return CPLB_OK;
}

cplb_status cplb_get_block_column(const cplb_problem* p, cplb_block block, const char* contact_name, int32_t* col)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(col);
    int c = 0;
    cplb_status st = block_column(p, block, contact_name, &c);
    if (st == CPLB_OK) *col = c;
    return st;
}

cplb_status cplb_get_contact_row(const cplb_problem* p, const char* contact_name, int32_t* row)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(row);
    const int k = p->find(contact_name);
    if (k < 0) return fail(CPLB_OUT_OF_RANGE, "map::at: unknown contact '%s'", contact_name ? contact_name : "(null)");
    *row = p->layout.contact_row(p->layout.rank[k]);
    return CPLB_OK;
}

cplb_status cplb_get_jacobian_constants(const cplb_problem* p, uint8_t* is_constant, double* value)
{
    CPLB_REQUIRE(p);
    for (int s = 0; s < p->layout.nnz; s++) {
        if (is_constant) is_constant[s] = p->layout.is_const[s];
        if (value) value[s] = p->layout.const_value[s];
    }
    return CPLB_OK;
}

cplb_status cplb_fill_jacobian_constants(const cplb_problem* p, int64_t num_instances, int32_t layout, int64_t ld, double* jac_host)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(jac_host);
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (layout != CPLB_INSTANCE_MAJOR && layout != CPLB_COMPONENT_MAJOR) return fail(CPLB_INVALID_ARGUMENT, "unknown layout %d", layout);
    const cplb::Layout& L = p->layout;
    const long long pitch = ld == 0 ? num_instances : ld;
    if (layout == CPLB_COMPONENT_MAJOR && pitch < num_instances) return fail(CPLB_INVALID_ARGUMENT, "ld is smaller than num_instances");
    for (int s = 0; s < L.nnz; s++) {
        if (!L.is_const[s]) continue;
        const double v = L.const_value[s];
        if (layout == CPLB_INSTANCE_MAJOR)
            for (long long i = 0; i < num_instances; i++) jac_host[i * L.nnz + s] = v;
        else
            for (long long i = 0; i < num_instances; i++) jac_host[(long long)s * pitch + i] = v;
    }
    return CPLB_OK;
}

cplb_status cplb_get_packed_jacobian_map(const cplb_problem* p, int32_t* num_packed, int32_t* packed_to_slot)
{
    CPLB_REQUIRE(p);
    const auto& map = p->layout.packed_to_slot;
    if (num_packed) *num_packed = (int32_t)map.size();
    if (packed_to_slot) std::memcpy(packed_to_slot, map.data(), sizeof(int32_t) * map.size());
    return CPLB_OK;
}

cplb_status cplb_unpack_jacobian(const cplb_problem* p, int64_t num_instances, const double* packed, double* full)
{
    CPLB_REQUIRE(p);
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (num_instances == 0) return CPLB_OK;
    CPLB_REQUIRE(packed);
    CPLB_REQUIRE(full);
    const cplb::Layout& L = p->layout;
    const int nv = (int)L.packed_to_slot.size();
    for (long long i = 0; i < num_instances; i++) {
        double* row = full + i * L.nnz;
        const double* src = packed + i * nv;
        for (int s = 0; s < L.nnz; s++)
            if (L.is_const[s]) row[s] = L.const_value[s];
        for (int q = 0; q < nv; q++) row[L.packed_to_slot[q]] = src[q];
    }
    return CPLB_OK;
}

cplb_status cplb_get_jacobian_slot_sources(const cplb_problem* p, int32_t* num_computed, int32_t* kind, int32_t* source)
{
    CPLB_REQUIRE(p);
    const cplb::Layout& L = p->layout;
    if (num_computed) *num_computed = (int32_t)L.computed_to_slot.size();
    if (kind) std::memcpy(kind, L.slot_kind.data(), sizeof(int32_t) * L.slot_kind.size());
    if (source) std::memcpy(source, L.slot_source.data(), sizeof(int32_t) * L.slot_source.size());
    return CPLB_OK;
}

cplb_status cplb_expand_jacobian(const cplb_problem* p, int64_t num_instances, const double* x, const double* computed, double* full)
{
    CPLB_REQUIRE(p);
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (num_instances == 0) return CPLB_OK;
    CPLB_REQUIRE(x);
    CPLB_REQUIRE(computed);
    CPLB_REQUIRE(full);
    const cplb::Layout& L = p->layout;
    const int nv = (int)L.computed_to_slot.size();
    for (long long i = 0; i < num_instances; i++) {
        double* row = full + i * L.nnz;
        const double* src = computed + i * nv;
        const double* xi = x + i * L.n;
        for (int s = 0; s < L.nnz; s++) {
            switch (L.slot_kind[s]) {
            case cplb::Layout::kConstant: row[s] = L.const_value[s]; break;
            case cplb::Layout::kCopy: row[s] = xi[L.slot_source[s]]; break;
            case cplb::Layout::kNegatedCopy: row[s] = -xi[L.slot_source[s]]; break;
            default: row[s] = src[L.slot_source[s]]; break;
            }
        }
    }
    return CPLB_OK;
}

cplb_status cplb_get_variable_bounds(const cplb_problem* p, double* lower, double* upper)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(lower);
    CPLB_REQUIRE(upper);
    std::memcpy(lower, p->x_lb.data(), sizeof(double) * p->layout.n);
    std::memcpy(upper, p->x_ub.data(), sizeof(double) * p->layout.n);
    return CPLB_OK;
}

cplb_status cplb_get_constraint_bounds(const cplb_problem* p, double* lower, double* upper)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(lower);
    CPLB_REQUIRE(upper);
    const cplb::Layout& L = p->layout;
    for (int r = 0; r < L.m; r++) {  // ifopt::Bounds(0,0) everywhere ...
        lower[r] = 0.0;
        upper[r] = 0.0;
    }
    for (int j = 0; j < L.nc; j++) {  // ... except the FrictionCone rows: ifopt::BoundSmallerZero = (-1e20, 0)
        const int row = L.contact_row(j) + (L.has_env ? 4 : 0);
        lower[row] = lower[row + 1] = -1.0e20;
    }
    return CPLB_OK;
}

// ---- parameters ---------------------------------------------------------------------------

cplb_status cplb_set_mass(cplb_problem* p, double mass)
{
    CPLB_REQUIRE(p);
    if (!(mass > 0.0)) return fail(CPLB_INVALID_ARGUMENT, "Invalid robot mass");
    p->mass = mass;
    p->refresh_derived();
    return CPLB_OK;
}
cplb_status cplb_get_mass(const cplb_problem* p, double* mass)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(mass);
    *mass = p->mass;
    return CPLB_OK;
}

cplb_status cplb_set_reduction_order(cplb_problem* p, int32_t order)
{
    CPLB_REQUIRE(p);
    if (order != 0 && order != 1) return fail(CPLB_INVALID_ARGUMENT, "reduction order must be 0 ((v0+v1)+v2) or 1 (v0+(v1+v2))");
    p->P.reduction_order = order;
    return CPLB_OK;
}

cplb_status cplb_set_component_major_kernel(cplb_problem* p, int32_t kernel)
{
    CPLB_REQUIRE(p);
    if (kernel != CPLB_KERNEL_AUTO && kernel != CPLB_KERNEL_PER_CONTACT && kernel != CPLB_KERNEL_PER_INSTANCE)
        return fail(CPLB_INVALID_ARGUMENT, "unknown component-major kernel choice %d", (int)kernel);
    if (kernel == CPLB_KERNEL_PER_INSTANCE && p->layout.nc != 4 && p->layout.nc != 8)
        return fail(CPLB_INVALID_ARGUMENT, "the thread-per-instance kernel exists for 4 and 8 contacts only (this problem has %d)", p->layout.nc);
    p->cm_kernel = kernel == CPLB_KERNEL_AUTO ? CPLB_CM_AUTO : (kernel == CPLB_KERNEL_PER_CONTACT ? CPLB_CM_SPLIT : CPLB_CM_WHOLE);
    return CPLB_OK;
}

cplb_status cplb_set_instance_major_kernel(cplb_problem* p, int32_t kernel)
{
    CPLB_REQUIRE(p);
    if (kernel != CPLB_KERNEL_AUTO && kernel != CPLB_KERNEL_WARP_TILE && kernel != CPLB_KERNEL_CTA_TILE)
        return fail(CPLB_INVALID_ARGUMENT, "unknown instance-major kernel choice %d", (int)kernel);
    p->im_kernel = kernel == CPLB_KERNEL_AUTO ? CPLB_IM_AUTO : (kernel == CPLB_KERNEL_WARP_TILE ? CPLB_IM_WARP_TILE : CPLB_IM_CTA_TILE);
    return CPLB_OK;
}

cplb_status cplb_get_device(const cplb_problem* p, int32_t* device)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(device);
    *device = p->device;
    return CPLB_OK;
}

cplb_status cplb_set_manipulation_wrench(cplb_problem* p, const double wrench[6])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(wrench);
    for (int i = 0; i < 6; i++) p->P.wrench[i] = wrench[i];
    return CPLB_OK;
}
cplb_status cplb_get_manipulation_wrench(const cplb_problem* p, double wrench[6])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(wrench);
    for (int i = 0; i < 6; i++) wrench[i] = p->P.wrench[i];
    return CPLB_OK;
}

cplb_status cplb_set_mu(cplb_problem* p, double mu)
{
    CPLB_REQUIRE(p);
    if (mu <= 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid friction coefficient");  // Environment.h:21-22
    p->P.mu = mu;
    return CPLB_OK;
}
cplb_status cplb_get_mu(const cplb_problem* p, double* mu)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(mu);
    *mu = p->P.mu;
    return CPLB_OK;
}

cplb_status cplb_set_ground_z(cplb_problem* p, double ground_z)
{
    CPLB_REQUIRE(p);
    if (p->env != CPLB_ENV_GROUND) return fail(CPLB_RUNTIME_ERROR, "the problem's environment is not a Ground");
    p->P.ground_z = ground_z;
    return CPLB_OK;
}
cplb_status cplb_get_ground_z(const cplb_problem* p, double* ground_z)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ground_z);
    if (p->env != CPLB_ENV_GROUND) return fail(CPLB_RUNTIME_ERROR, "the problem's environment is not a Ground");
    *ground_z = p->P.ground_z;
    return CPLB_OK;
}

cplb_status cplb_set_superquadric(cplb_problem* p, const double C[3], const double R[3], const double Pw[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(C);
    CPLB_REQUIRE(R);
    CPLB_REQUIRE(Pw);
    if (p->env != CPLB_ENV_SUPERQUADRIC) return fail(CPLB_RUNTIME_ERROR, "the problem's environment is not a Superquadric");
    if (R[0] <= 0.0 || R[1] <= 0.0 || R[2] <= 0.0)  // Superquadric.cpp:16-19
        return fail(CPLB_INVALID_ARGUMENT, "Invalid superquadric axial radii");
    if (Pw[0] < 2.0 || Pw[1] < 2.0 || Pw[2] < 2.0)  // :21-24
        return fail(CPLB_INVALID_ARGUMENT, "Invalid superquadric axial curvatures: must be >= 2");
    for (int q = 0; q < 3; q++) {
        p->sqC[q] = C[q];
        p->sqR[q] = R[q];
        p->sqP[q] = Pw[q];
    }
    p->refresh_derived();
    return CPLB_OK;
}
cplb_status cplb_get_superquadric(const cplb_problem* p, double C[3], double R[3], double Pw[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(C);
    CPLB_REQUIRE(R);
    CPLB_REQUIRE(Pw);
    if (p->env != CPLB_ENV_SUPERQUADRIC) return fail(CPLB_RUNTIME_ERROR, "the problem's environment is not a Superquadric");
    for (int q = 0; q < 3; q++) {
        C[q] = p->sqC[q];
        R[q] = p->sqR[q];
        Pw[q] = p->sqP[q];
    }
    return CPLB_OK;
}

#define CPLB_CONTACT(k, p, name)                                                                        \
    const int k = (p)->find(name);                                                                      \
    if (k < 0) return fail(CPLB_OUT_OF_RANGE, "map::at: unknown contact '%s'", (name) ? (name) : "(null)")

cplb_status cplb_set_force_threshold(cplb_problem* p, const char* contact_name, double F_thr)
{
    CPLB_REQUIRE(p);
    CPLB_CONTACT(k, p, contact_name);
    p->P.F_thr[k] = F_thr;
    return CPLB_OK;
}
cplb_status cplb_get_force_threshold(const cplb_problem* p, const char* contact_name, double* F_thr)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(F_thr);
    CPLB_CONTACT(k, p, contact_name);
    *F_thr = p->P.F_thr[k];
    return CPLB_OK;
}

cplb_status cplb_set_bounds(cplb_problem* p, cplb_block block, const char* contact_name, const double lower[3],
                            const double upper[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(lower);
    CPLB_REQUIRE(upper);
    int col = 0;
    cplb_status st = block_column(p, block, contact_name, &col);
    if (st != CPLB_OK) return st;
    bool bad = false;
    for (int i = 0; i < 3; i++) {  // Variable3D::SetBounds stores first, then checks (Variable3D.cpp:31-38)
        p->x_lb[col + i] = lower[i];
        p->x_ub[col + i] = upper[i];
        if (upper[i] - lower[i] < 0) bad = true;
    }
    if (bad) return fail(CPLB_INVALID_ARGUMENT, "Inconsistent bounds");
    return CPLB_OK;
}
cplb_status cplb_get_bounds(const cplb_problem* p, cplb_block block, const char* contact_name, double lower[3], double upper[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(lower);
    CPLB_REQUIRE(upper);
    int col = 0;
    cplb_status st = block_column(p, block, contact_name, &col);
    if (st != CPLB_OK) return st;
    for (int i = 0; i < 3; i++) {
        lower[i] = p->x_lb[col + i];
        upper[i] = p->x_ub[col + i];
    }
    return CPLB_OK;
}

cplb_status cplb_set_pos_ref(cplb_problem* p, const char* contact_name, const double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    CPLB_CONTACT(k, p, contact_name);
    for (int i = 0; i < 3; i++) p->P.p_ref[k][i] = ref[i];
    return CPLB_OK;
}
cplb_status cplb_get_pos_ref(const cplb_problem* p, const char* contact_name, double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    CPLB_CONTACT(k, p, contact_name);
    for (int i = 0; i < 3; i++) ref[i] = p->P.p_ref[k][i];
    return CPLB_OK;
}
cplb_status cplb_set_force_ref(cplb_problem* p, const char* contact_name, const double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    CPLB_CONTACT(k, p, contact_name);
    for (int i = 0; i < 3; i++) p->P.F_ref[k][i] = ref[i];
    return CPLB_OK;
}
cplb_status cplb_get_force_ref(const cplb_problem* p, const char* contact_name, double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    CPLB_CONTACT(k, p, contact_name);
    for (int i = 0; i < 3; i++) ref[i] = p->P.F_ref[k][i];
    return CPLB_OK;
}
cplb_status cplb_set_com_ref(cplb_problem* p, const double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    for (int i = 0; i < 3; i++) p->P.com_ref[i] = ref[i];
    return CPLB_OK;
}
cplb_status cplb_get_com_ref(const cplb_problem* p, double ref[3])
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(ref);
    for (int i = 0; i < 3; i++) ref[i] = p->P.com_ref[i];
    return CPLB_OK;
}
// Weight checks (< 0 -> std::invalid_argument "Invalid weight") are the planner facade's
// (CentroidalPlanner.cpp:186-189, 203-206, 233-236, 256-259, 286-289); kept here so every binding gets them.
cplb_status cplb_set_com_weight(cplb_problem* p, double W)
{
    CPLB_REQUIRE(p);
    if (W < 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid weight");
    p->P.W_com = W;
    return CPLB_OK;
}
cplb_status cplb_get_com_weight(const cplb_problem* p, double* W)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(W);
    *W = p->P.W_com;
    return CPLB_OK;
}
cplb_status cplb_set_pos_weight(cplb_problem* p, double W)
{
    CPLB_REQUIRE(p);
    if (W < 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid weight");
    for (int k = 0; k < p->layout.nc; k++) p->P.W_p[k] = W;
    return CPLB_OK;
}
cplb_status cplb_set_force_weight(cplb_problem* p, double W)
{
    CPLB_REQUIRE(p);
    if (W < 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid weight");
    for (int k = 0; k < p->layout.nc; k++) p->P.W_F[k] = W;
    return CPLB_OK;
}
cplb_status cplb_set_contact_pos_weight(cplb_problem* p, const char* contact_name, double W)
{
    CPLB_REQUIRE(p);
    CPLB_CONTACT(k, p, contact_name);
    if (W < 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid weight");
    p->P.W_p[k] = W;
    return CPLB_OK;
}
cplb_status cplb_get_contact_pos_weight(const cplb_problem* p, const char* contact_name, double* W)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(W);
    CPLB_CONTACT(k, p, contact_name);
    *W = p->P.W_p[k];
    return CPLB_OK;
}
cplb_status cplb_set_contact_force_weight(cplb_problem* p, const char* contact_name, double W)
{
    CPLB_REQUIRE(p);
    CPLB_CONTACT(k, p, contact_name);
    if (W < 0.0) return fail(CPLB_INVALID_ARGUMENT, "Invalid weight");
    p->P.W_F[k] = W;
    return CPLB_OK;
}
cplb_status cplb_get_contact_force_weight(const cplb_problem* p, const char* contact_name, double* W)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(W);
    CPLB_CONTACT(k, p, contact_name);
    *W = p->P.W_F[k];
    return CPLB_OK;
}

// ---- evaluation -----------------------------------------------------------------------------

// Binds a problem created with device = -1 to the calling thread's current device.  This is where a
// machine without a GPU fails: loudly, with CPLB_CUDA_ERROR -- there is no CPU evaluation path.
static cplb_status bind_device(cplb_problem* p)
{
    if (p->device >= 0) return CPLB_OK;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(CPLB_CUDA_ERROR, "no usable CUDA device (%s); this library has no CPU fallback",
                    e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    int dev = 0;
    CPLB_CUDA(cudaGetDevice(&dev));
    p->device = dev;
    p->pipes[0].device = dev;
    return CPLB_OK;
}

static cplb_status check_args(const cplb_problem* p, const cplb_eval_args* a, unsigned* flags, long long* ld)
{
    if (a->num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (a->layout != CPLB_INSTANCE_MAJOR && a->layout != CPLB_COMPONENT_MAJOR)
        return fail(CPLB_INVALID_ARGUMENT, "unknown layout %d", a->layout);
    if (a->num_instances > 0 && a->x == nullptr) return fail(CPLB_NULL_POINTER, "x is NULL");
    unsigned f = 0;
    if (a->g) f |= CPLB_WANT_G;
    if (a->jac) f |= CPLB_WANT_J;
    if (a->cost) f |= CPLB_WANT_COST;
    if (a->grad) f |= CPLB_WANT_GRAD;
    *flags = f;
    long long pitch = a->ld == 0 ? a->num_instances : a->ld;
    if (a->layout == CPLB_COMPONENT_MAJOR && pitch < a->num_instances)
        return fail(CPLB_INVALID_ARGUMENT, "ld (%lld) is smaller than num_instances (%lld)", pitch, (long long)a->num_instances);
    if (a->layout == CPLB_COMPONENT_MAJOR && pitch >= (1LL << 29))
        return fail(CPLB_INVALID_ARGUMENT, "ld (%lld) must be below 2^29: the kernels hold the row pitch in bytes in 32 bits", pitch);
    *ld = pitch;
    if (a->host_flags & CPLB_JAC_PACKED) {
        if (a->layout != CPLB_INSTANCE_MAJOR) return fail(CPLB_INVALID_ARGUMENT, "CPLB_JAC_PACKED needs INSTANCE_MAJOR buffers (COMPONENT_MAJOR host calls skip whole rows with CPLB_HOST_JAC_CONSTANTS_PRESENT instead)");
        *flags |= CPLB_JAC_PACKED_K;
    }
    if (a->host_flags & CPLB_JAC_COMPUTED) {
        if (a->layout != CPLB_INSTANCE_MAJOR) return fail(CPLB_INVALID_ARGUMENT, "CPLB_JAC_COMPUTED needs INSTANCE_MAJOR buffers");
        if (a->host_flags & CPLB_JAC_PACKED) return fail(CPLB_INVALID_ARGUMENT, "CPLB_JAC_PACKED and CPLB_JAC_COMPUTED name two different slice formats: pass one of them");
        *flags |= CPLB_JAC_COMPUTED_K;
    }
    (void)p;
    return CPLB_OK;
}

// cplb_instance_params holds the same pointers as CplbInstParams::arr, member i being array i of CplbInstArray
constexpr size_t inst_array_offset(int a) { return offsetof(CplbInstParams, arr) + a * sizeof(const double*); }
static_assert(sizeof(cplb_instance_params) == sizeof(CplbInstParams), "cplb_instance_params and CplbInstParams differ in size");
static_assert(offsetof(cplb_instance_params, mass) == inst_array_offset(CPLB_IA_MASS), "mass");
static_assert(offsetof(cplb_instance_params, wrench) == inst_array_offset(CPLB_IA_WRENCH), "wrench");
static_assert(offsetof(cplb_instance_params, mu) == inst_array_offset(CPLB_IA_MU), "mu");
static_assert(offsetof(cplb_instance_params, force_threshold) == inst_array_offset(CPLB_IA_F_THR), "force_threshold");
static_assert(offsetof(cplb_instance_params, ground_z) == inst_array_offset(CPLB_IA_GROUND_Z), "ground_z");
static_assert(offsetof(cplb_instance_params, com_ref) == inst_array_offset(CPLB_IA_COM_REF), "com_ref");
static_assert(offsetof(cplb_instance_params, com_weight) == inst_array_offset(CPLB_IA_W_COM), "com_weight");
static_assert(offsetof(cplb_instance_params, pos_ref) == inst_array_offset(CPLB_IA_P_REF), "pos_ref");
static_assert(offsetof(cplb_instance_params, force_ref) == inst_array_offset(CPLB_IA_F_REF), "force_ref");
static_assert(offsetof(cplb_instance_params, pos_weight) == inst_array_offset(CPLB_IA_W_P), "pos_weight");
static_assert(offsetof(cplb_instance_params, force_weight) == inst_array_offset(CPLB_IA_W_F), "force_weight");

// The caller's per-instance arrays (abi may be NULL) as CplbInstParams; false when none is set.
static bool instance_arrays(const cplb_instance_params* abi, CplbInstParams* q)
{
    *q = CplbInstParams{};
    if (abi) std::memcpy(q, abi, sizeof *q);
    for (const double* a : q->arr)
        if (a) return true;
    return false;
}

static cplb_status launch(cplb_problem* p, const CplbIo& io, int layout, unsigned flags, cudaStream_t st,
                          const CplbInstParams* q = nullptr)
{
    cudaError_t e = layout == CPLB_COMPONENT_MAJOR ? cplb::launch_component_major(p->P, io, flags, q, p->cm_kernel, st)
                                                   : cplb::launch_instance_major(p->P, io, flags, q, p->im_kernel, st);
    if (e != cudaSuccess) return cuda_fail(e, "kernel launch");
    p->launches.fetch_add(1, std::memory_order_relaxed);
    return CPLB_OK;
}

static cplb_status eval_device_on(cplb_problem* p, int device, const cplb_eval_args* args, unsigned flags, long long ld, void* cuda_stream)
{
    DeviceGuard dg(device);
    if (!dg.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", device);
    cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
    CplbIo io{args->x, args->g, args->jac, args->cost, args->grad, ld, args->num_instances};

    bool timed = false;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    {
        std::lock_guard<std::mutex> lk(p->timing_mu);
        timed = p->timing;
    }
    if (timed) {
        CPLB_CUDA(cudaEventCreate(&e0));
        CPLB_CUDA(cudaEventCreate(&e1));
        CPLB_CUDA(cudaEventRecord(e0, stream));
    }
    CplbInstParams q;
    const bool per_inst = instance_arrays(args->per_instance, &q);
    if (args->host_flags & CPLB_DEVICE_INPUTS_READY) flags |= CPLB_INPUTS_READY;
    cplb_status st = launch(p, io, args->layout, flags, stream, per_inst ? &q : nullptr);
    if (timed) {
        cudaEventRecord(e1, stream);
        std::lock_guard<std::mutex> lk(p->timing_mu);
        p->events.emplace_back(e0, e1);
    }
    return st;
}

cplb_status cplb_eval_device(cplb_problem* p, const cplb_eval_args* args, void* cuda_stream)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(args);
    unsigned flags = 0;
    long long ld = 0;
    cplb_status st = check_args(p, args, &flags, &ld);
    if (st != CPLB_OK) return st;
    if (p->pipes.size() > 1)
        return fail(CPLB_INVALID_ARGUMENT, "this problem is sharded over %d devices: device buffers belong to one of them, use cplb_eval_device_shard",
                    (int)p->pipes.size());
    if (args->num_instances == 0 || (flags & 15u) == 0) return CPLB_OK;
    st = bind_device(p);
    if (st != CPLB_OK) return st;
    return eval_device_on(p, p->device, args, flags, ld, cuda_stream);
}

cplb_status cplb_eval_device_shard(cplb_problem* p, int32_t shard, const cplb_eval_args* args, void* cuda_stream)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(args);
    if (shard < 0 || shard >= (int32_t)p->pipes.size()) return fail(CPLB_INVALID_ARGUMENT, "shard %d out of range (%d shards)", (int)shard, (int)p->pipes.size());
    unsigned flags = 0;
    long long ld = 0;
    cplb_status st = check_args(p, args, &flags, &ld);
    if (st != CPLB_OK) return st;
    if (args->num_instances == 0 || (flags & 15u) == 0) return CPLB_OK;
    st = bind_device(p);
    if (st != CPLB_OK) return st;
    return eval_device_on(p, p->pipes[(size_t)shard].device, args, flags, ld, cuda_stream);
}

// Contiguous index ranges of a batch of N instances over the problem's devices (SURVEY 8(e): GPU r of G evaluates
// [r*N/G, (r+1)*N/G)); boundaries are rounded to multiples of 32 instances so that every shard's slices keep the 16-byte
// alignment and tile alignment of the whole buffer.
static void shard_range(long long N, int shard, int shards, long long* begin, long long* end)
{
    long long per = (N + shards - 1) / shards;
    per = (per + 31) & ~31LL;
    long long b = per * shard, e = b + per;
    if (b > N) b = N;
    if (e > N) e = N;
    *begin = b;
    *end = e;
}

cplb_status cplb_get_num_shards(const cplb_problem* p, int32_t* num_shards)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(num_shards);
    *num_shards = (int32_t)p->pipes.size();
    return CPLB_OK;
}

cplb_status cplb_get_shard(const cplb_problem* p, int32_t shard, int64_t num_instances, int32_t* device, int64_t* begin, int64_t* end)
{
    CPLB_REQUIRE(p);
    if (shard < 0 || shard >= (int32_t)p->pipes.size()) return fail(CPLB_INVALID_ARGUMENT, "shard %d out of range (%d shards)", (int)shard, (int)p->pipes.size());
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    long long b = 0, e = 0;
    shard_range(num_instances, shard, (int)p->pipes.size(), &b, &e);
    if (device) *device = p->pipes[(size_t)shard].device;
    if (begin) *begin = b;
    if (end) *end = e;
    return CPLB_OK;
}

using HostPipe = cplb_problem::HostPipe;

// doubles per instance of the Jacobian slice of this evaluation: every structural slot, or only the x-dependent ones
static int jac_len(const cplb_problem* p, unsigned flags)
{
    if (flags & CPLB_JAC_COMPUTED_K) return (int)p->layout.computed_to_slot.size();
    return (flags & CPLB_JAC_PACKED_K) ? (int)p->layout.packed_to_slot.size() : p->layout.nnz;
}

static cplb_status ensure_host_pipeline(HostPipe& pipe, size_t bytes_per_stream)
{
    if (!pipe.streams_ready) {
        for (int s = 0; s < kHostStreams; s++) CPLB_CUDA(cudaStreamCreateWithFlags(&pipe.streams[s], cudaStreamNonBlocking));
        pipe.streams_ready = true;
    }
    if (bytes_per_stream > pipe.stage_bytes) {
        for (int s = 0; s < kHostStreams; s++) {
            if (pipe.stage[s]) {
                CPLB_CUDA(cudaStreamSynchronize(pipe.streams[s]));
                CPLB_CUDA(cudaFree(pipe.stage[s]));
                pipe.stage[s] = nullptr;
            }
        }
        pipe.stage_bytes = 0;
        for (int s = 0; s < kHostStreams; s++) CPLB_CUDA(cudaMalloc(&pipe.stage[s], bytes_per_stream));
        pipe.stage_bytes = bytes_per_stream;
    }
    return CPLB_OK;
}

static bool is_pinned(const void* ptr)
{
    if (!ptr) return true;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost || attr.type == cudaMemoryTypeManaged;
}

// Pageable caller buffers: cudaMemcpyAsync on them is synchronous and, measured, several times slower than a host
// memcpy through a pinned buffer.  Each stream gets a pinned mirror of its device staging buffer; a chunk is packed
// into it, travels H2D / kernel / D2H asynchronously, and is unpacked when the stream's turn comes round again.
struct HostInput {  // one host input array (x or a per-instance parameter array): len elements per instance
    const double* user;
    int len;
    size_t off;  // offset (doubles) inside a staging buffer
    int arr;     // CplbInstArray; -1 for x
};

// x and every per-instance array that is present, laid out after the output sections of a staging buffer
static std::vector<HostInput> host_inputs(const cplb_problem* p, const cplb_eval_args* args, long long chunk, size_t first_free, size_t* end)
{
    std::vector<HostInput> in;
    in.push_back(HostInput{args->x, p->layout.n, 0, -1});
    size_t off = first_free;
    CplbInstParams user;
    instance_arrays(args->per_instance, &user);
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
        if (user.arr[a]) {
            const int len = cplb_inst_len(a, p->layout.nc);
            in.push_back(HostInput{user.arr[a], len, off, a});
            off += (size_t)len * chunk;
        }
    *end = off;
    return in;
}

// instances [begin, end) of the caller's buffers through one device's pipeline; the calling thread's current device is pipe.device
static cplb_status eval_host_bounced(cplb_problem* p, HostPipe& pipe, const cplb_eval_args* args, unsigned flags, long long ld, long long chunk,
                                     size_t stage_bytes, long long begin, long long end)
{
    const int n = p->layout.n, m = p->layout.m, nnz = jac_len(p, flags);
    const bool cm = args->layout == CPLB_COMPONENT_MAJOR;
    const bool skip_const = (args->host_flags & CPLB_HOST_JAC_CONSTANTS_PRESENT) != 0;
    if (stage_bytes > pipe.bounce_bytes) {
        for (int s = 0; s < kHostStreams; s++) {
            if (pipe.bounce[s]) {
                CPLB_CUDA(cudaStreamSynchronize(pipe.streams[s]));
                CPLB_CUDA(cudaFreeHost(pipe.bounce[s]));
                pipe.bounce[s] = nullptr;
            }
        }
        pipe.bounce_bytes = 0;
        for (int s = 0; s < kHostStreams; s++) CPLB_CUDA(cudaHostAlloc((void**)&pipe.bounce[s], stage_bytes, cudaHostAllocDefault));
        pipe.bounce_bytes = stage_bytes;
    }
    struct Pending { long long i0 = 0, cnt = 0; };
    Pending pend[kHostStreams];
    // sections of a staging buffer, in doubles: x | g | jac | grad | cost  (rows of `chunk` for component-major)
    const size_t ox = 0, og = ox + (size_t)n * chunk, oj = og + ((flags & CPLB_WANT_G) ? (size_t)m * chunk : 0),
                 ogr = oj + ((flags & CPLB_WANT_J) ? (size_t)nnz * chunk : 0), oc = ogr + ((flags & CPLB_WANT_GRAD) ? (size_t)n * chunk : 0);
    size_t in_end = 0;
    const std::vector<HostInput> inputs = host_inputs(p, args, chunk, oc + ((flags & CPLB_WANT_COST) ? (size_t)chunk : 0), &in_end);
    auto unpack_one = [&](double* user, const double* h, int len, long long i0, long long cnt) {
        if (!user) return;
        if (cm) for (int e = 0; e < len; e++) std::memcpy(user + (long long)e * ld + i0, h + (size_t)e * chunk, (size_t)cnt * sizeof(double));
        else std::memcpy(user + i0 * len, h, (size_t)cnt * len * sizeof(double));
    };
    auto drain = [&](int s) -> cplb_status {
        if (pend[s].cnt == 0) return CPLB_OK;
        CPLB_CUDA(cudaStreamSynchronize(pipe.streams[s]));
        const double* h = pipe.bounce[s];
        unpack_one(args->g, h + og, m, pend[s].i0, pend[s].cnt);
        if (cm && skip_const && args->jac) {  // rows of x-independent slots stay as the caller pre-filled them
            for (const auto& r : p->layout.var_runs)
                for (int e = r.begin; e < r.end; e++)
                    std::memcpy(args->jac + (long long)e * ld + pend[s].i0, h + oj + (size_t)e * chunk, (size_t)pend[s].cnt * sizeof(double));
        } else {
            unpack_one(args->jac, h + oj, nnz, pend[s].i0, pend[s].cnt);
        }
        unpack_one(args->grad, h + ogr, n, pend[s].i0, pend[s].cnt);
        if (args->cost) std::memcpy(args->cost + pend[s].i0, h + oc, (size_t)pend[s].cnt * sizeof(double));
        pend[s].cnt = 0;
        return CPLB_OK;
    };
    // a failure leaves nothing in flight: the caller may free or reuse its buffers as soon as the call has returned
    auto bail = [&](cplb_status st) {
        for (int t = 0; t < kHostStreams; t++) cudaStreamSynchronize(pipe.streams[t]);
        return st;
    };
    int s = 0;
    for (long long i0 = begin; i0 < end; i0 += chunk, s = (s + 1) % kHostStreams) {
        const long long cnt = (end - i0) < chunk ? (end - i0) : chunk;
        cplb_status st = drain(s);
        if (st != CPLB_OK) return bail(st);
        cudaStream_t stream = pipe.streams[s];
        double* h = pipe.bounce[s];
        double* d = pipe.stage[s];
        CplbInstParams q{};
        for (const auto& in : inputs) {
            double* hb = h + in.off;
            if (cm) for (int e = 0; e < in.len; e++) std::memcpy(hb + (size_t)e * chunk, in.user + (long long)e * ld + i0, (size_t)cnt * sizeof(double));
            else std::memcpy(hb, in.user + i0 * in.len, (size_t)cnt * in.len * sizeof(double));
            cudaError_t e = cudaMemcpyAsync(d + in.off, hb, (size_t)in.len * chunk * sizeof(double), cudaMemcpyHostToDevice, stream);
            if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMemcpyAsync (host to device)"));
            if (in.arr >= 0) q.arr[in.arr] = d + in.off;
        }
        CplbIo io{d + ox, (flags & CPLB_WANT_G) ? d + og : nullptr, (flags & CPLB_WANT_J) ? d + oj : nullptr,
                  (flags & CPLB_WANT_COST) ? d + oc : nullptr, (flags & CPLB_WANT_GRAD) ? d + ogr : nullptr, chunk, cnt};
        st = launch(p, io, args->layout, flags, stream, inputs.size() > 1 ? &q : nullptr);
        if (st != CPLB_OK) return bail(st);
        const size_t out_doubles = (oc - og) + ((flags & CPLB_WANT_COST) ? (size_t)chunk : 0);
        if (out_doubles) {
            cudaError_t e = cudaMemcpyAsync(h + og, d + og, out_doubles * sizeof(double), cudaMemcpyDeviceToHost, stream);
            if (e != cudaSuccess) return bail(cuda_fail(e, "cudaMemcpyAsync (device to host)"));
        }
        pend[s].i0 = i0;
        pend[s].cnt = cnt;
    }
    for (int t = 0; t < kHostStreams; t++) {
        cplb_status st = drain(t);
        if (st != CPLB_OK) return bail(st);
    }
    return CPLB_OK;
}

// One chunk [i0, i0 + cnt) of a pinned-buffer call on stream s of one device's pipeline: H2D, kernel, D2H, all asynchronous.
static cplb_status enqueue_chunk(cplb_problem* p, HostPipe& pipe, int s, const cplb_eval_args* args, unsigned flags, long long ld, long long chunk,
                                 long long i0, long long cnt)
{
    const int n = p->layout.n, m = p->layout.m, nnz = jac_len(p, flags);
    const bool cm = args->layout == CPLB_COMPONENT_MAJOR;
    const bool skip_const = (args->host_flags & CPLB_HOST_JAC_CONSTANTS_PRESENT) != 0;
    cudaStream_t stream = pipe.streams[s];
    double* d = pipe.stage[s];
    double* dx = d;
    d += (size_t)n * chunk;
    double *dg_ = nullptr, *dj = nullptr, *dc = nullptr, *dgr = nullptr;
    if (flags & CPLB_WANT_G) { dg_ = d; d += (size_t)m * chunk; }
    if (flags & CPLB_WANT_J) { dj = d; d += (size_t)nnz * chunk; }
    if (flags & CPLB_WANT_GRAD) { dgr = d; d += (size_t)n * chunk; }
    if (flags & CPLB_WANT_COST) { dc = d; d += (size_t)chunk; }
    // device-side chunk buffers use pitch `chunk` (component-major) or are dense (instance-major)
    CplbInstParams user, q{};
    const bool per_inst = instance_arrays(args->per_instance, &user);
    auto h2d = [&](double* dst, const double* src, int len) -> cplb_status {
        if (cm) CPLB_CUDA(cudaMemcpy2DAsync(dst, chunk * sizeof(double), src + i0, ld * sizeof(double), cnt * sizeof(double), len, cudaMemcpyHostToDevice, stream));
        else CPLB_CUDA(cudaMemcpyAsync(dst, src + i0 * len, (size_t)cnt * len * sizeof(double), cudaMemcpyHostToDevice, stream));
        return CPLB_OK;
    };
    cplb_status st = h2d(dx, args->x, n);
    if (st != CPLB_OK) return st;
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
        if (user.arr[a]) {
            const int len = cplb_inst_len(a, p->layout.nc);
            st = h2d(d, user.arr[a], len);
            if (st != CPLB_OK) return st;
            q.arr[a] = d;
            d += (size_t)len * chunk;
        }
    CplbIo io{dx, dg_, dj, dc, dgr, chunk, cnt};
    st = launch(p, io, args->layout, flags, stream, per_inst ? &q : nullptr);
    if (st != CPLB_OK) return st;
    if (cm) {
        if (dg_) CPLB_CUDA(cudaMemcpy2DAsync(args->g + i0, ld * sizeof(double), dg_, chunk * sizeof(double), cnt * sizeof(double), m, cudaMemcpyDeviceToHost, stream));
        if (dj && skip_const) {  // only the rows of x-dependent slots
            for (const auto& r : p->layout.var_runs)
                CPLB_CUDA(cudaMemcpy2DAsync(args->jac + (long long)r.begin * ld + i0, ld * sizeof(double), dj + (size_t)r.begin * chunk,
                                            chunk * sizeof(double), cnt * sizeof(double), r.end - r.begin, cudaMemcpyDeviceToHost, stream));
        } else if (dj) {
            CPLB_CUDA(cudaMemcpy2DAsync(args->jac + i0, ld * sizeof(double), dj, chunk * sizeof(double), cnt * sizeof(double), nnz, cudaMemcpyDeviceToHost, stream));
        }
        if (dgr) CPLB_CUDA(cudaMemcpy2DAsync(args->grad + i0, ld * sizeof(double), dgr, chunk * sizeof(double), cnt * sizeof(double), n, cudaMemcpyDeviceToHost, stream));
    } else {
        if (dg_) CPLB_CUDA(cudaMemcpyAsync(args->g + i0 * m, dg_, (size_t)cnt * m * sizeof(double), cudaMemcpyDeviceToHost, stream));
        // instance-major: the x-dependent slots are 96..432-byte runs inside each 1.4 KB row; strided 2-D DMA copies
        // of such runs, and a scatter kernel writing them straight into the mapped host buffer, both measured no
        // faster than one contiguous copy of whole rows (2.16 / 2.17 vs 2.15 ms for 65,536 instances), so the rows
        // travel whole -- the constant slots are simply rewritten with the same values
        if (dj) CPLB_CUDA(cudaMemcpyAsync(args->jac + i0 * nnz, dj, (size_t)cnt * nnz * sizeof(double), cudaMemcpyDeviceToHost, stream));
        if (dgr) CPLB_CUDA(cudaMemcpyAsync(args->grad + i0 * n, dgr, (size_t)cnt * n * sizeof(double), cudaMemcpyDeviceToHost, stream));
    }
    if (dc) CPLB_CUDA(cudaMemcpyAsync(args->cost + i0, dc, (size_t)cnt * sizeof(double), cudaMemcpyDeviceToHost, stream));
    return CPLB_OK;
}

// ticket == nullptr: synchronous (returns when the outputs have landed).  Otherwise the work is only enqueued, a completion
// event per stream is recorded into the next ticket slot and its index returned; pinned buffers are required then.
// A sharded problem cuts [0, N) into one contiguous range per device and drives every device's pipeline from this call:
// with pinned buffers everything is asynchronous, so the chunks of all devices are enqueued round robin by the calling thread;
// pageable buffers are packed / unpacked by one worker thread per device.
static cplb_status eval_host_impl(cplb_problem* p, const cplb_eval_args* args, int32_t* ticket)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(args);
    if (ticket) *ticket = -1;
    unsigned flags = 0;
    long long ld = 0;
    cplb_status st = check_args(p, args, &flags, &ld);
    if (st != CPLB_OK) return st;
    const long long N = args->num_instances;
    if (N == 0 || (flags & 15u) == 0) return CPLB_OK;
    st = bind_device(p);
    if (st != CPLB_OK) return st;
    std::lock_guard<std::mutex> lk(p->host_mu);
    const int shards = (int)p->pipes.size();
    DeviceGuard restore(p->pipes[0].device);  // every cudaSetDevice below is undone when the call returns
    if (!restore.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", p->pipes[0].device);

    const int n = p->layout.n, m = p->layout.m, nnz = jac_len(p, flags);
    // 32,768-instance chunks (few, long copies: the download engine is the bound), big enough for efficient PCIe bursts, small
    // enough that three chunks in flight overlap H2D, kernel and D2H.  A synchronous call starts with one short chunk so that
    // its first download begins early; a queued call is preceded by the previous call's downloads anyway.
    long long longest = 0;
    for (int sh = 0; sh < shards; sh++) {
        long long b, e;
        shard_range(N, sh, shards, &b, &e);
        if (e - b > longest) longest = e - b;
    }
    long long chunk = 32768;
    if (chunk > longest) chunk = longest;
    chunk = (chunk + 31) & ~31LL;  // keeps every chunk's slices 16-byte aligned and tile-aligned
    size_t per_inst = (size_t)n;
    if (flags & CPLB_WANT_G) per_inst += m;
    if (flags & CPLB_WANT_J) per_inst += nnz;
    if (flags & CPLB_WANT_COST) per_inst += 1;
    if (flags & CPLB_WANT_GRAD) per_inst += n;
    CplbInstParams user;
    instance_arrays(args->per_instance, &user);
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
        if (user.arr[a]) per_inst += cplb_inst_len(a, p->layout.nc);
    const size_t stage_bytes = per_inst * (size_t)chunk * sizeof(double);
    auto set_device = [&](int sh) -> cplb_status {
        if (shards > 1) CPLB_CUDA(cudaSetDevice(p->pipes[(size_t)sh].device));
        return CPLB_OK;
    };
    for (int sh = 0; sh < shards; sh++) {
        long long b, e;
        shard_range(N, sh, shards, &b, &e);
        if (b == e) continue;
        st = set_device(sh);
        if (st == CPLB_OK) st = ensure_host_pipeline(p->pipes[(size_t)sh], stage_bytes);
        if (st != CPLB_OK) return st;
    }

    bool all_pinned = is_pinned(args->x) && is_pinned(args->g) && is_pinned(args->jac) && is_pinned(args->cost) && is_pinned(args->grad);
    for (const double* a : user.arr) all_pinned = all_pinned && is_pinned(a);
    if (!all_pinned) {
        if (ticket) return fail(CPLB_INVALID_ARGUMENT, "cplb_eval_host_begin needs pinned host buffers (cplb_host_alloc)");
        if (shards == 1) return eval_host_bounced(p, p->pipes[0], args, flags, ld, chunk, stage_bytes, 0, N);
        std::vector<std::thread> workers;
        std::vector<cplb_status> status((size_t)shards, CPLB_OK);
        std::vector<std::string> message((size_t)shards);
        for (int sh = 0; sh < shards; sh++) {
            long long b, e;
            shard_range(N, sh, shards, &b, &e);
            if (b == e) continue;
            workers.emplace_back([&, sh, b, e] {
                HostPipe& pipe = p->pipes[(size_t)sh];
                if (cudaSetDevice(pipe.device) != cudaSuccess) {
                    status[(size_t)sh] = CPLB_CUDA_ERROR;
                    message[(size_t)sh] = "cudaSetDevice failed in a shard worker";
                    return;
                }
                status[(size_t)sh] = eval_host_bounced(p, pipe, args, flags, ld, chunk, stage_bytes, b, e);
                if (status[(size_t)sh] != CPLB_OK) message[(size_t)sh] = g_last_error;  // the worker's thread-local message
            });
        }
        for (auto& w : workers) w.join();
        for (int sh = 0; sh < shards; sh++)
            if (status[(size_t)sh] != CPLB_OK) return fail(status[(size_t)sh], "shard %d (device %d): %s", sh, p->pipes[(size_t)sh].device, message[(size_t)sh].c_str());
        return CPLB_OK;
    }
    if (ticket) {
        for (int sh = 0; sh < shards; sh++) {
            HostPipe& pipe = p->pipes[(size_t)sh];
            if (pipe.host_done_ready || !pipe.streams_ready) continue;
            st = set_device(sh);
            if (st != CPLB_OK) return st;
            for (int t = 0; t < kHostTickets; t++)
                for (int q = 0; q < kHostStreams; q++) CPLB_CUDA(cudaEventCreateWithFlags(&pipe.host_done[t][q], cudaEventDisableTiming));
            pipe.host_done_ready = true;
        }
    }

    // On any failure after the first enqueue nothing may stay in flight: the caller gets an error and no ticket, so it has
    // nothing to wait on before it frees or reuses its buffers.
    auto bail = [&](cplb_status err) {
        char keep[sizeof g_last_error];
        std::memcpy(keep, g_last_error, sizeof keep);
        for (int sh = 0; sh < shards; sh++) {
            HostPipe& pipe = p->pipes[(size_t)sh];
            if (!pipe.streams_ready) continue;
            if (shards > 1) cudaSetDevice(pipe.device);
            for (int t = 0; t < kHostStreams; t++) cudaStreamSynchronize(pipe.streams[t]);
        }
        std::memcpy(g_last_error, keep, sizeof keep);
        return err;
    };
    // The round robin over a pipeline's streams continues across calls: the first chunk of a queued call then lands on the
    // stream whose previous work finished longest ago instead of behind the previous call's last download.  Chunks of the
    // devices are enqueued interleaved (chunk 0 of every shard, then chunk 1, ...) so that every device starts at once.
    struct Cursor { long long next, end; bool first; };
    std::vector<Cursor> cur((size_t)shards);
    for (int sh = 0; sh < shards; sh++) {
        long long b, e;
        shard_range(N, sh, shards, &b, &e);
        cur[(size_t)sh] = Cursor{b, e, true};
    }
    for (bool any = true; any;) {
        any = false;
        for (int sh = 0; sh < shards; sh++) {
            Cursor& c = cur[(size_t)sh];
            if (c.next >= c.end) continue;
            any = true;
            HostPipe& pipe = p->pipes[(size_t)sh];
            const long long len = c.end - c.next;
            long long want = chunk;
            if (c.first && !ticket && len > chunk) want = chunk / 4;
            const long long cnt = len < want ? len : want;
            st = set_device(sh);
            if (st == CPLB_OK) st = enqueue_chunk(p, pipe, pipe.next_stream, args, flags, ld, chunk, c.next, cnt);
            pipe.next_stream = (pipe.next_stream + 1) % kHostStreams;
            if (st != CPLB_OK) return bail(st);
            c.next += cnt;
            c.first = false;
        }
    }
    if (!ticket) {
        for (int sh = 0; sh < shards; sh++) {
            HostPipe& pipe = p->pipes[(size_t)sh];
            if (!pipe.streams_ready) continue;
            st = set_device(sh);
            if (st != CPLB_OK) return bail(st);
            for (int t = 0; t < kHostStreams; t++) {
                cudaError_t e = cudaStreamSynchronize(pipe.streams[t]);
                if (e != cudaSuccess) return bail(cuda_fail(e, "cudaStreamSynchronize"));
            }
        }
        return CPLB_OK;
    }
    const int slot = p->next_ticket;
    p->next_ticket = (slot + 1) % kHostTickets;
    // the slot's previous use must be over before its events are re-recorded (the caller waited for it or never will)
    for (int sh = 0; sh < shards; sh++) {
        HostPipe& pipe = p->pipes[(size_t)sh];
        if (!pipe.host_done_ready) continue;
        st = set_device(sh);
        if (st != CPLB_OK) return bail(st);
        for (int t = 0; t < kHostStreams; t++) {
            cudaError_t e = cudaEventRecord(pipe.host_done[slot][t], pipe.streams[t]);
            if (e != cudaSuccess) return bail(cuda_fail(e, "cudaEventRecord"));
        }
    }
    *ticket = slot;
    return CPLB_OK;
}

cplb_status cplb_eval_host(cplb_problem* p, const cplb_eval_args* args) { return eval_host_impl(p, args, nullptr); }

cplb_status cplb_eval_host_begin(cplb_problem* p, const cplb_eval_args* args, int32_t* ticket)
{
    CPLB_REQUIRE(ticket);
    return eval_host_impl(p, args, ticket);
}

cplb_status cplb_eval_host_wait(cplb_problem* p, int32_t ticket)
{
    CPLB_REQUIRE(p);
    if (ticket == -1) return CPLB_OK;  // an empty call (no instances / no outputs) completed at once
    bool any_ready = false;
    for (const auto& pipe : p->pipes) any_ready = any_ready || pipe.host_done_ready;
    if (ticket < 0 || ticket >= kHostTickets || !any_ready) return fail(CPLB_INVALID_ARGUMENT, "unknown ticket %d", (int)ticket);
    DeviceGuard restore(p->pipes[0].device);
    if (!restore.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", p->pipes[0].device);
    for (auto& pipe : p->pipes) {
        if (!pipe.host_done_ready) continue;
        if (p->pipes.size() > 1) CPLB_CUDA(cudaSetDevice(pipe.device));
        for (int t = 0; t < kHostStreams; t++) CPLB_CUDA(cudaEventSynchronize(pipe.host_done[ticket][t]));
    }
    return CPLB_OK;
}

// ---- the caller side: N lock-step solves (SURVEY 8(f) rank 1) -----------------------------------------------------------------

void cplb_solver_default_options(cplb_solver_options* o)
{
    if (!o) return;
    o->tol = 1e-3;  // ifopt's IpoptSolver default (SURVEY Appendix B.8)
    o->mu_init = 0.1;
    o->bound_push = 1e-2;
    o->bound_frac = 1e-2;
    o->nlp_scaling_max_gradient = 100.0;
    o->constr_viol_tol = 1e-4;
    o->polish_viol_tol = 1e-9;
    o->bound_relax_factor = 1e-8;
    o->max_iter = 500;
    o->max_backtracks = 30;
    o->tail_instances = -1;
}

cplb_status cplb_solve_device(cplb_problem* p, int64_t num_instances, const double* x0, const cplb_instance_params* per_instance,
                              const cplb_solver_options* options, const cplb_solve_outputs* out, void* cuda_stream)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(out);
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (p->pipes.size() > 1) return fail(CPLB_INVALID_ARGUMENT, "cplb_solve_device needs a single-device problem (one solve batch per GPU)");
    if (num_instances == 0) return CPLB_OK;
    CPLB_REQUIRE(x0);
    CPLB_REQUIRE(out->x);
    CPLB_REQUIRE(out->status);
    CPLB_REQUIRE(out->iterations);
    CPLB_REQUIRE(out->cost);
    CPLB_REQUIRE(out->constr_viol);
    CPLB_REQUIRE(out->dual_inf);
    cplb_solver_options o;
    cplb_solver_default_options(&o);
    if (options) o = *options;
    if (!(o.tol > 0.0) || !(o.mu_init > 0.0) || o.max_iter < 0 || o.max_backtracks < 1)
        return fail(CPLB_INVALID_ARGUMENT, "solver options: tol and mu_init must be positive, max_iter >= 0, max_backtracks >= 1");
    if (cplb::solver::team_block_bytes(p->layout.n, p->layout.m, p->layout.nnz, nullptr) > cplb::solver::kMaxTeamBlockBytes) {
        // one instance's KKT system must fit one CTA's shared memory: name the largest contact count of this kind that does
        int limit = 0;
        for (int k = 1; k <= CPLB_MAX_CONTACTS; k++) {
            std::vector<std::string> names;
            for (int c = 0; c < k; c++) names.push_back("c" + std::to_string(c));
            cplb::Layout L;
            L.build(names, p->env != CPLB_ENV_NONE, p->env == CPLB_ENV_GROUND);
            if (cplb::solver::team_block_bytes(L.n, L.m, L.nnz, nullptr) > cplb::solver::kMaxTeamBlockBytes) break;
            limit = k;
        }
        return fail(CPLB_INVALID_ARGUMENT,
                    "cplb_solve_device: %d contacts need %zu bytes of shared memory per instance, more than the %zu a CTA has; "
                    "at most %d contacts can be solved with this environment",
                    (int)p->names.size(), cplb::solver::team_block_bytes(p->layout.n, p->layout.m, p->layout.nnz, nullptr),
                    cplb::solver::kMaxTeamBlockBytes, limit);
    }
    cplb_status st = bind_device(p);
    if (st != CPLB_OK) return st;
    DeviceGuard dg(p->device);
    if (!dg.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", p->device);
    std::lock_guard<std::mutex> lk(p->solver_mu);
    const cplb::Layout& L = p->layout;
    std::vector<double> cl(L.m), cu(L.m);
    cplb_get_constraint_bounds(p, cl.data(), cu.data());
    cplb::solver::ShapeHost SH;
    SH.build(L.n, L.m, L.nnz, L.iRow.data(), L.jCol.data(), p->x_lb.data(), p->x_ub.data(), cl.data(), cu.data(), o.bound_relax_factor);
    const cplb::solver::Options O{o.tol, o.mu_init, o.bound_push, o.bound_frac, o.nlp_scaling_max_gradient, o.constr_viol_tol, o.polish_viol_tol,
                                  o.bound_relax_factor, o.max_iter, o.max_backtracks, o.tail_instances};
    cplb::solver::SolveStats stats;
    const long long launches_per_round = 8;
    CplbInstParams q;
    const bool per_inst = instance_arrays(per_instance, &q);
    cudaError_t e = cplb::solver::solve_device(p->P, p->im_kernel, per_inst ? &q : nullptr, SH, O, num_instances, x0, out->x, out->status, out->iterations, out->cost,
                                               out->constr_viol, out->dual_inf, out->lam, &stats, &p->solver_ws, static_cast<cudaStream_t>(cuda_stream));
    if (e != cudaSuccess) return cuda_fail(e, "cplb_solve_device");
    p->launches.fetch_add(stats.evaluations + launches_per_round / 2 * stats.rounds + 3, std::memory_order_relaxed);
    if (out->rounds) *out->rounds = stats.rounds;
    if (out->evaluations) *out->evaluations = stats.evaluations;
    if (out->instance_evaluations) *out->instance_evaluations = stats.instance_evaluations;
    if (out->tail_instances) *out->tail_instances = stats.tail_instances;
    return CPLB_OK;
}

// ---- first-order derivative test (CentroidalPlanner.cpp:26) -------------------------------------------------------------------

void cplb_derivative_test_default_options(cplb_derivative_test_options* o)
{
    if (!o) return;
    o->perturbation = 1e-8;  // IPOPT's derivative_test_perturbation
    o->tol = 1e-4;           // derivative_test_tol
}

// The dense (row, col) -> slot table of the problem on its device, uploaded once.  The copy runs on a stream of its own and is
// waited for there, so the caller's stream is never synchronised.
static cplb_status derivtest_slot_table(cplb_problem* p)
{
    std::lock_guard<std::mutex> lk(p->derivtest_mu);
    if (p->slot_of) return CPLB_OK;
    const cplb::Layout& L = p->layout;
    std::vector<int32_t> table((size_t)L.m * L.n, -1);
    for (int s = 0; s < L.nnz; s++) table[(size_t)L.iRow[s] * L.n + L.jCol[s]] = s;
    const size_t bytes = table.size() * sizeof(int32_t);
    int32_t* d = nullptr;
    CPLB_CUDA(cudaMalloc(&d, bytes));
    cudaStream_t up = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&up, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        e = cudaMemcpyAsync(d, table.data(), bytes, cudaMemcpyHostToDevice, up);
        const cudaError_t e2 = cudaStreamSynchronize(up);
        if (e == cudaSuccess) e = e2;
        cudaStreamDestroy(up);
    }
    if (e != cudaSuccess) {
        cudaFree(d);
        return cuda_fail(e, "cplb_derivative_test_device: uploading the Jacobian structure");
    }
    p->slot_of = d;
    return CPLB_OK;
}

cplb_status cplb_derivative_test_device(cplb_problem* p, int64_t num_instances, const double* x, const cplb_instance_params* per_instance,
                                        const cplb_derivative_test_options* options, const cplb_derivative_test_outputs* out, void* cuda_stream)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(out);
    if (num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (num_instances > 0 && x == nullptr) return fail(CPLB_NULL_POINTER, "x is NULL");
    cplb_derivative_test_options o;
    cplb_derivative_test_default_options(&o);
    if (options) o = *options;
    if (!(std::isfinite(o.perturbation) && o.perturbation > 0.0))
        return fail(CPLB_INVALID_ARGUMENT, "derivative test options: perturbation must be finite and positive (got %g)", o.perturbation);
    if (!(o.tol > 0.0)) return fail(CPLB_INVALID_ARGUMENT, "derivative test options: tol must be positive (got %g)", o.tol);
    if (p->pipes.size() > 1)
        return fail(CPLB_INVALID_ARGUMENT, "cplb_derivative_test_device needs a single-device problem (one batch per GPU)");
    if (num_instances > INT32_MAX) return fail(CPLB_INVALID_ARGUMENT, "num_instances (%lld) must be below 2^31: one CTA per instance", (long long)num_instances);
    if (num_instances == 0) return CPLB_OK;
    cplb_status st = bind_device(p);
    if (st != CPLB_OK) return st;
    DeviceGuard dg(p->device);
    if (!dg.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", p->device);
    st = derivtest_slot_table(p);
    if (st != CPLB_OK) return st;
    CplbInstParams q;
    const bool per_inst = instance_arrays(per_instance, &q);
    const cplb::DerivTestOut dout{out->num_wrong, out->num_wrong_outside, out->max_rel_error, out->worst_row, out->worst_col, out->jac_fd, out->grad_fd};
    cudaError_t e = cplb::launch_derivative_test(p->P, per_inst ? &q : nullptr, x, num_instances, p->slot_of, o.perturbation, o.tol, dout,
                                                 static_cast<cudaStream_t>(cuda_stream));
    if (e != cudaSuccess) return cuda_fail(e, "cplb_derivative_test_device");
    p->launches.fetch_add(1, std::memory_order_relaxed);
    return CPLB_OK;
}

// ---- Jacobian products ---------------------------------------------------------------------------------------------------------

cplb_status cplb_jacobian_products_device(cplb_problem* p, const cplb_jacobian_products_args* args, void* cuda_stream)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(args);
    const cplb_jacobian_products_args& a = *args;
    if (a.num_instances < 0) return fail(CPLB_INVALID_ARGUMENT, "num_instances is negative");
    if (a.num_instances > 0 && a.x == nullptr) return fail(CPLB_NULL_POINTER, "x is NULL");
    if (a.x_bar && !a.lambda && !a.obj_factor)
        return fail(CPLB_INVALID_ARGUMENT, "x_bar is requested but lambda and obj_factor are both NULL: the reverse product has no term");
    if ((a.g_dot || a.f_dot) && a.v == nullptr) return fail(CPLB_NULL_POINTER, "v is NULL but g_dot or f_dot is requested");
    if (!a.x_bar && !a.g_dot && !a.f_dot) return fail(CPLB_INVALID_ARGUMENT, "no output requested: set x_bar, g_dot or f_dot");
    if (p->pipes.size() > 1)
        return fail(CPLB_INVALID_ARGUMENT, "cplb_jacobian_products_device needs a single-device problem (one batch per GPU)");
    if (a.num_instances > INT32_MAX) return fail(CPLB_INVALID_ARGUMENT, "num_instances (%lld) must be below 2^31", (long long)a.num_instances);
    if (a.num_instances == 0) return CPLB_OK;
    cplb_status st = bind_device(p);
    if (st != CPLB_OK) return st;
    DeviceGuard dg(p->device);
    if (!dg.ok) return fail(CPLB_CUDA_ERROR, "cudaSetDevice(%d) failed", p->device);
    CplbInstParams q;
    const bool per_inst = instance_arrays(a.per_instance, &q);
    const cplb::ProductArgs pa{a.x, a.lambda, a.obj_factor, a.x_bar, a.v, a.g_dot, a.f_dot, a.num_instances};
    cudaError_t e = cplb::launch_jacobian_products(p->P, per_inst ? &q : nullptr, pa, static_cast<cudaStream_t>(cuda_stream));
    if (e != cudaSuccess) return cuda_fail(e, "cplb_jacobian_products_device");
    p->launches.fetch_add(1, std::memory_order_relaxed);
    return CPLB_OK;
}

cplb_status cplb_host_alloc(size_t bytes, void** out)
{
    CPLB_REQUIRE(out);
    *out = nullptr;
    CPLB_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));  // pinned for every device of the process (sharded problems)
    return CPLB_OK;
}
cplb_status cplb_host_free(void* ptr)
{
    if (ptr) CPLB_CUDA(cudaFreeHost(ptr));
    return CPLB_OK;
}

cplb_status cplb_get_launch_count(const cplb_problem* p, int64_t* launches)
{
    CPLB_REQUIRE(p);
    CPLB_REQUIRE(launches);
    *launches = p->launches.load(std::memory_order_relaxed);
    return CPLB_OK;
}

cplb_status cplb_timing_begin(cplb_problem* p)
{
    CPLB_REQUIRE(p);
    std::lock_guard<std::mutex> lk(p->timing_mu);
    for (auto& ev : p->events) {
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    p->events.clear();
    p->timing = true;
    return CPLB_OK;
}

cplb_status cplb_timing_end(cplb_problem* p, double* avg_kernel_ms, int64_t* kernels)
{
    CPLB_REQUIRE(p);
    DeviceGuard dg(p->device >= 0 ? p->device : 0);
    std::lock_guard<std::mutex> lk(p->timing_mu);
    p->timing = false;
    double total = 0.0;
    long long cnt = 0;
    for (auto& ev : p->events) {
        CPLB_CUDA(cudaEventSynchronize(ev.second));
        float ms = 0.f;
        CPLB_CUDA(cudaEventElapsedTime(&ms, ev.first, ev.second));
        total += ms;
        cnt++;
        cudaEventDestroy(ev.first);
        cudaEventDestroy(ev.second);
    }
    p->events.clear();
    if (avg_kernel_ms) *avg_kernel_ms = cnt ? total / (double)cnt : 0.0;
    if (kernels) *kernels = cnt;
    return CPLB_OK;
}

}  // extern "C"
