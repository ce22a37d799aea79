// cplb_solver.cu -- the native lock-step solve round on the GPU: cplb_solve_device of include/cpl_batched.h.
//
// N instances of one problem are solved together by the interior-point scheme of cplb_solver_core.hpp.  A round is a fixed
// sequence of eight launches -- four batched evaluations of the hot path (the same kernels cplb_eval_device launches) and
// four solver kernels that run ONE CTA PER INSTANCE with the instance's KKT system in shared memory:
//
//   round_begin   kappa_sigma safeguard, convergence test, barrier update, the nf + 1 forward-difference points
//   [eval]        gradient + Jacobian at N (nf + 1) points
//   kkt           Lagrangian Hessian from the differences, assembly of the (n + m)^2 KKT matrix, pivoted LU and solve inside an
//                 inertia-free regularisation loop, feasibility-polish step, multiplier steps, fraction-to-the-boundary
//                 step lengths, merit-function set-up, 30 line-search candidates
//   [eval]        constraint values + cost at N x 30 candidates
//   ls_first      merit test of the full step; where it fails, second-order correction with the stored factors
//   [eval]        constraint values + cost at the corrected points
//   ls_select     first acceptable point in the order of a sequential backtracking search, iterate and multiplier update
//   [eval]        everything at the new iterate
//
// The host only counts the instances still running (one 4-byte read per round).  Nothing else leaves the device: what the
// previous driver (centroidalplanner_b200/lockstep_solver.py: ~1,500 small torch launches and cuBLAS' batched LU per round) did
// from Python happens inside these kernels.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <utility>
#include <vector>

#include "cplb_eval_inline.cuh"
#include "cplb_kernels.h"
#include "cplb_solver.h"
#include "cplb_solver_core.hpp"

namespace cplb {
namespace solver {

struct DeviceTeam {
    int rank, size;
    __device__ __forceinline__ void sync() const { __syncthreads(); }
    // the first warp of the CTA folds (cplb_solver_core.hpp: warp_fold, a __shfl_xor butterfly: every lane gets the result)
    __device__ __forceinline__ int lanes() const { return kWarp; }
};

constexpr int kThreads = 128;     // vector phases
constexpr int kThreadsLU = 256;   // phases that factor: a 16 x 16 thread grid on the trailing update

struct KernelArgs {
    Shape S;
    State T;
    Options O;
    int mats_in_global;  // dense Jacobian and Hessian of a slot in global memory (State::jd_slot / h0_slot) instead of the team's block
};

// Scratch::carve with the slot's external matrices where the launch uses them
__device__ __forceinline__ void carve_full(Scratch& q, double* smem, const KernelArgs& A, long long b)
{
    q.carve(smem, A.S.n, A.S.m, A.S.nnz, true, A.mats_in_global ? A.T.jd_slot + b * A.S.m * A.S.n : nullptr,
            A.mats_in_global ? A.T.h0_slot + b * A.S.n * A.S.n : nullptr);
}

__global__ void __launch_bounds__(kThreads) k_init_x(const __grid_constant__ KernelArgs A, const double* x0)
{
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    phase_init_x(team, A.S, A.T, A.O, (long long)blockIdx.x, x0);
}

__global__ void __launch_bounds__(kThreads) k_init_scale(const __grid_constant__ KernelArgs A)
{
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    phase_init_scale(team, A.S, A.T, A.O, (long long)blockIdx.x);
}

__global__ void __launch_bounds__(kThreads) k_round_begin(const __grid_constant__ KernelArgs A, int first, int last, int* n_active)
{
    extern __shared__ __align__(16) double smem[];
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    Scratch q;
    q.carve(smem, A.S.n, A.S.m, A.S.nnz, false);
    phase_round_begin(team, A.S, A.T, A.O, (long long)blockIdx.x, q, first, last, n_active);
}

__global__ void __launch_bounds__(kThreadsLU, 4) k_kkt(const __grid_constant__ KernelArgs A)
{
    extern __shared__ __align__(16) double smem[];
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    Scratch q;
    const long long b = (long long)blockIdx.x;
    carve_full(q, smem, A, b);
    phase_kkt(team, A.S, A.T, A.O, b, q);
}

__global__ void __launch_bounds__(kThreads) k_ls_first(const __grid_constant__ KernelArgs A)
{
    extern __shared__ __align__(16) double smem[];
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    Scratch q;
    const long long b = (long long)blockIdx.x;
    carve_full(q, smem, A, b);
    phase_ls_first(team, A.S, A.T, A.O, b, q);
}

__global__ void __launch_bounds__(kThreads) k_ls_select(const __grid_constant__ KernelArgs A)
{
    extern __shared__ __align__(16) double smem[];
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    Scratch q;
    q.carve(smem, A.S.n, A.S.m, A.S.nnz, false);
    phase_ls_select(team, A.S, A.T, A.O, (long long)blockIdx.x, q);
}

// The tail: one CTA carries one instance through ALL its remaining iterations, the four evaluations of an iteration done in
// place by eval_points (cplb_eval_inline.cuh: the batched kernels' arithmetic as a device function, spread over the team).  Entered
// once the working set no longer fills the GPU: from there a lock-step round costs its latency floor whatever the count, and
// every round would be paid by the slowest instance; here each instance pays only its own iterations and the host waits once.
__global__ void __launch_bounds__(kThreadsLU, 2) k_tail(const __grid_constant__ KernelArgs A, const __grid_constant__ CplbParams P,
                                                        const __grid_constant__ CplbInstParams Q, int per_instance, int it0,
                                                        unsigned long long* instance_rounds)
{
    extern __shared__ __align__(16) double smem[];
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    Scratch q;
    const long long b = (long long)blockIdx.x;
    carve_full(q, smem, A, b);
    const long long inst = A.T.list_cur[b];
    auto eval = [&](const double* x, int count, unsigned flags, double* g, double* jac, double* cost, double* grad) {
        eval_points(team.rank, team.size, P, per_instance ? &Q : nullptr, inst, x, count, g, jac, cost, grad, flags);
    };
    unsigned rounds = 0;
    for (int it = it0;;) {
        tail_iteration(team, A.S, A.T, A.O, b, q, eval);
        rounds++;
        it++;
        phase_round_begin(team, A.S, A.T, A.O, b, q, 0, it == A.O.max_iter, nullptr, true);
        team.sync();
        if (!A.T.active[inst]) break;
    }
    if (team.rank == 0) atomicAdd(instance_rounds, (unsigned long long)rounds);
}

// Per-instance parameter arrays (cplb_instance_params) in the order of the working set: the batched evaluations of a round run
// over slot-ordered buffers (one point per slot, nf + 1 difference points per slot, kCandidates line-search points per slot), so
// every round the parameters of the running instances are laid out the same way -- one row per evaluated point.
struct ParamGather {
    const double* src[CPLB_NUM_INST_ARRAYS];
    double* one[CPLB_NUM_INST_ARRAYS];  // [slots][len]
    double* fd[CPLB_NUM_INST_ARRAYS];   // [slots][reps_fd][len]
    double* ls[CPLB_NUM_INST_ARRAYS];   // [slots][reps_ls][len]
    int len[CPLB_NUM_INST_ARRAYS];
    int reps_fd, reps_ls;
};

__global__ void __launch_bounds__(kThreads) k_gather_params(const __grid_constant__ ParamGather G, const int32_t* list)
{
    const long long b = (long long)blockIdx.x, i = list[b];
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++) {
        if (G.src[a] == nullptr) continue;
        const int len = G.len[a], rows = 1 + G.reps_fd + G.reps_ls;
        for (int t = (int)threadIdx.x; t < rows * len; t += (int)blockDim.x) {
            const int row = t / len, e = t - row * len;
            const double v = G.src[a][i * len + e];
            if (row == 0) G.one[a][b * len + e] = v;
            else if (row <= G.reps_fd) G.fd[a][(b * G.reps_fd + (row - 1)) * (long long)len + e] = v;
            else G.ls[a][(b * G.reps_ls + (row - 1 - G.reps_fd)) * (long long)len + e] = v;
        }
    }
}

__global__ void __launch_bounds__(kThreads) k_finish(const __grid_constant__ KernelArgs A, double* x_out, double* lam_out)
{
    DeviceTeam team{(int)threadIdx.x, (int)blockDim.x};
    phase_finish(team, A.S, A.T, (long long)blockIdx.x, x_out, lam_out);
}

#define SOLVER_CUDA(call)                 \
    do {                                  \
        cudaError_t e__ = (call);         \
        if (e__ != cudaSuccess) return e__; \
    } while (0)

// device copies of the problem-level arrays + the per-instance state slab; owned by the problem handle, grown on demand
struct Workspace {
    void* shape_slab = nullptr;
    void* state_slab = nullptr;
    size_t state_bytes = 0, shape_bytes = 0;
    int* n_active = nullptr;
    int* n_active_host = nullptr;
    unsigned long long* tail_rounds = nullptr;  // device counter + its pinned mirror
    unsigned long long* tail_rounds_host = nullptr;
    void* param_slab = nullptr;  // slot-ordered copies of the per-instance parameter arrays
    size_t param_bytes = 0;
};

void workspace_free(Workspace* w)
{
    if (!w) return;
    if (w->shape_slab) cudaFree(w->shape_slab);
    if (w->state_slab) cudaFree(w->state_slab);
    if (w->n_active) cudaFree(w->n_active);
    if (w->n_active_host) cudaFreeHost(w->n_active_host);
    if (w->tail_rounds) cudaFree(w->tail_rounds);
    if (w->param_slab) cudaFree(w->param_slab);
    if (w->tail_rounds_host) cudaFreeHost(w->tail_rounds_host);
    delete w;
}

struct DeviceEngine {
    const CplbParams& P;
    int im_kernel;
    KernelArgs A;
    long long N;
    cudaStream_t st;
    Workspace* W;
    const double* x0;
    double *x_out, *lam_out;
    size_t smem, smem_small;
    long long tail_limit;
    const CplbInstParams* Qsrc;  // per-instance parameter arrays in instance order, or nullptr
    ParamGather G;
    CplbInstParams Q_one, Q_fd, Q_ls;
    bool gathered = false;
    cudaError_t err = cudaSuccess;

    void check(cudaError_t e)
    {
        if (err == cudaSuccess && e != cudaSuccess) err = e;
    }
    void eval(const double* x, double* g, double* jac, double* cost, double* grad, long long count, const CplbInstParams* Q)
    {
        if (err != cudaSuccess) return;
        unsigned flags = (g ? CPLB_WANT_G : 0u) | (jac ? CPLB_WANT_J : 0u) | (cost ? CPLB_WANT_COST : 0u) | (grad ? CPLB_WANT_GRAD : 0u);
        CplbIo io{x, g, jac, cost, grad, count, count};
        check(launch_instance_major(P, io, flags, Qsrc ? Q : nullptr, im_kernel, st));
    }
    // one CTA per slot of the working set (or per instance for the phases outside the rounds)
    template <class K, class... Args>
    void run(K kern, long long ctas, size_t shared, Args... args)
    {
        if (err != cudaSuccess || ctas <= 0) return;
        kern<<<(unsigned)ctas, (const void*)kern == (const void*)k_kkt ? kThreadsLU : kThreads, shared, st>>>(A, args...);
        check(cudaGetLastError());
    }
    void init_x() { run(k_init_x, N, 0, x0); }
    void init_scale() { run(k_init_scale, N, 0); }
    long long round_begin(bool first, bool last, long long slots)
    {
        if (err != cudaSuccess) return 0;
        check(cudaMemsetAsync(W->n_active, 0, sizeof(int), st));
        run(k_round_begin, slots, smem_small, (int)first, (int)last, W->n_active);
        check(cudaMemcpyAsync(W->n_active_host, W->n_active, sizeof(int), cudaMemcpyDeviceToHost, st));
        check(cudaStreamSynchronize(st));
        std::swap(A.T.list_cur, A.T.list_next);  // the instances still running, in the order their CTAs got there
        const long long running = err == cudaSuccess ? *W->n_active_host : 0;
        if (Qsrc && running > tail_limit) {  // the lock-step evaluations of this round read the parameters in slot order
            k_gather_params<<<(unsigned)running, kThreads, 0, st>>>(G, A.T.list_cur);
            check(cudaGetLastError());
            gathered = true;
        }
        return running;
    }
    void kkt(long long cnt) { run(k_kkt, cnt, smem); }
    void ls_first(long long cnt) { run(k_ls_first, cnt, smem); }
    void ls_select(long long cnt) { run(k_ls_select, cnt, smem_small); }
    long long tail_threshold() const { return tail_limit; }
    long long tail(long long running, int it0)
    {
        if (err != cudaSuccess) return 0;
        check(cudaMemsetAsync(W->tail_rounds, 0, sizeof(unsigned long long), st));
        k_tail<<<(unsigned)running, kThreadsLU, smem, st>>>(A, P, Qsrc ? *Qsrc : CplbInstParams{}, Qsrc ? 1 : 0, it0, W->tail_rounds);
        check(cudaGetLastError());
        check(cudaMemcpyAsync(W->tail_rounds_host, W->tail_rounds, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        check(cudaStreamSynchronize(st));
        return err == cudaSuccess ? (long long)*W->tail_rounds_host : 0;
    }
    void finish()
    {
        run(k_finish, N, 0, x_out, lam_out);
        check(cudaStreamSynchronize(st));
    }
    // (before the first round the slots are the instances: the caller's arrays serve as they are)
    void eval_full(long long cnt) { eval(A.T.xc, A.T.ev_c, A.T.ev_jv, A.T.ev_f, A.T.ev_df, cnt, gathered ? &Q_one : Qsrc); }
    void eval_fd(long long cnt) { eval(A.T.x_fd, nullptr, A.T.jac_fd, nullptr, A.T.grad_fd, cnt * (A.S.nf + 1), &Q_fd); }
    void eval_ls(long long cnt) { eval(A.T.x_ls, A.T.g_ls, nullptr, A.T.cost_ls, nullptr, cnt * kCandidates, &Q_ls); }
    void eval_soc(long long cnt) { eval(A.T.x_soc, A.T.g_soc, nullptr, A.T.cost_soc, nullptr, cnt, &Q_one); }
};

static size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

size_t team_block_bytes(int n, int m, int nnz, int* mats_in_global)
{
    // Four teams per SM are what the registers allow (256 threads x 64): where the full block is too large for that, the dense
    // Jacobian and the Hessian move to global memory (4 contacts: 71 KB -> 49 KB; 4,096 ground solves 0.0891 -> 0.0868 s); smaller
    // problems keep them in shared memory (CoMPlanner: 35 KB, and the global round trips would cost 10 %)
    Scratch probe;
    double dummy = 0.0;
    size_t bytes = probe.carve(nullptr, n, m, nnz, true) * sizeof(double);
    const int global = bytes > kMaxTeamBlockBytes / 4 - 1024 ? 1 : 0;
    if (global) bytes = probe.carve(nullptr, n, m, nnz, true, &dummy, &dummy) * sizeof(double);
    if (mats_in_global) *mats_in_global = global;
    return bytes;
}

cudaError_t solve_device(const CplbParams& P, int im_kernel, const CplbInstParams* per_instance, const ShapeHost& SH, const Options& O, long long N,
                         const double* x0, double* x_out,
                         int32_t* status, int32_t* iterations, double* cost, double* viol, double* dual, double* lam_out, SolveStats* stats,
                         Workspace** wsp, cudaStream_t st)
{
    if (!*wsp) *wsp = new Workspace();
    Workspace* W = *wsp;
    if (!W->n_active) {
        SOLVER_CUDA(cudaMalloc(&W->n_active, sizeof(int)));
        SOLVER_CUDA(cudaHostAlloc((void**)&W->n_active_host, sizeof(int), cudaHostAllocDefault));
        SOLVER_CUDA(cudaMalloc(&W->tail_rounds, sizeof(unsigned long long)));
        SOLVER_CUDA(cudaHostAlloc((void**)&W->tail_rounds_host, sizeof(unsigned long long), cudaHostAllocDefault));
    }
    KernelArgs A{};
    A.O = O;
    Shape& S = A.S;
    S.n = SH.n;
    S.m = SH.m;
    S.nnz = SH.nnz;
    S.nf = SH.nf;
    S.nk = SH.n + SH.m;
    // ---- problem-level arrays: one slab, uploaded per call (a few KB; setters may have changed the bounds) ----
    struct Up { const void* src; size_t bytes; const void** dst; };
    std::vector<Up> ups;
    auto up = [&](const auto& vec, const auto*& dst) {
        ups.push_back({vec.data(), vec.size() * sizeof(vec[0]), reinterpret_cast<const void**>(&dst)});
    };
    up(SH.iRow, S.iRow); up(SH.jCol, S.jCol); up(SH.col_ptr, S.col_ptr); up(SH.col_slot, S.col_slot); up(SH.free_idx, S.free_idx);
    up(SH.xl, S.xl); up(SH.xu, S.xu); up(SH.xlo_orig, S.xlo_orig); up(SH.xhi_orig, S.xhi_orig);
    up(SH.cl, S.cl); up(SH.cu, S.cu); up(SH.cl_r, S.cl_r); up(SH.cu_r, S.cu_r);
    up(SH.fixed, S.fixed); up(SH.x_lo, S.x_lo); up(SH.x_hi, S.x_hi); up(SH.s_lo, S.s_lo); up(SH.s_hi, S.s_hi); up(SH.is_eq, S.is_eq);
    size_t shape_bytes = 0;
    for (auto& u : ups) shape_bytes += align_up(u.bytes ? u.bytes : 1);
    if (shape_bytes > W->shape_bytes) {
        if (W->shape_slab) SOLVER_CUDA(cudaFree(W->shape_slab));
        W->shape_slab = nullptr;
        W->shape_bytes = 0;
        SOLVER_CUDA(cudaMalloc(&W->shape_slab, shape_bytes));
        W->shape_bytes = shape_bytes;
    }
    {
        std::vector<unsigned char> host(shape_bytes, 0);
        size_t off = 0;
        for (auto& u : ups) {
            if (u.bytes) std::memcpy(host.data() + off, u.src, u.bytes);
            *u.dst = static_cast<unsigned char*>(W->shape_slab) + off;
            off += align_up(u.bytes ? u.bytes : 1);
        }
        SOLVER_CUDA(cudaMemcpyAsync(W->shape_slab, host.data(), shape_bytes, cudaMemcpyHostToDevice, st));
        SOLVER_CUDA(cudaStreamSynchronize(st));  // `host` goes out of scope
    }
    // ---- per-instance state: one slab ----
    std::vector<StateField> fields = state_fields(A.T, SH);
    size_t state_bytes = 0;
    for (auto& f : fields) state_bytes += align_up(f.per_instance * (size_t)N * (f.is_int ? sizeof(int32_t) : sizeof(double)));
    if (state_bytes > W->state_bytes) {
        if (W->state_slab) SOLVER_CUDA(cudaFree(W->state_slab));
        W->state_slab = nullptr;
        W->state_bytes = 0;
        SOLVER_CUDA(cudaMalloc(&W->state_slab, state_bytes));
        W->state_bytes = state_bytes;
    }
    {
        size_t off = 0;
        for (auto& f : fields) {
            *f.ptr = static_cast<unsigned char*>(W->state_slab) + off;
            off += align_up(f.per_instance * (size_t)N * (f.is_int ? sizeof(int32_t) : sizeof(double)));
        }
    }
    // the caller's result arrays replace the internal ones where they exist
    A.T.status = status;
    A.T.iters = iterations;
    A.T.out_cost = cost;
    A.T.out_viol = viol;
    A.T.out_dual = dual;

    Scratch probe;
    const size_t smem = team_block_bytes(S.n, S.m, S.nnz, &A.mats_in_global);
    const size_t smem_small = probe.carve(nullptr, S.n, S.m, S.nnz, false) * sizeof(double);
    if (smem > kMaxTeamBlockBytes) return cudaErrorInvalidConfiguration;  // (cplb_solve_device refuses such shapes up front)
    for (const void* k : {(const void*)k_round_begin, (const void*)k_kkt, (const void*)k_ls_first, (const void*)k_ls_select, (const void*)k_tail})
        SOLVER_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxTeamBlockBytes));

    // The tail takes over when the working set fits the GPU in one wave of its CTAs (one per instance; `tail_instances` of the
    // options: < 0 picks SMs x resident CTAs, 0 never).
    long long tail_limit = O.tail_instances;
    if (tail_limit < 0) {
        int dev = 0, sms = 0, per_sm = 0;
        SOLVER_CUDA(cudaGetDevice(&dev));
        SOLVER_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        SOLVER_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tail, kThreadsLU, smem));
        tail_limit = (long long)sms * (per_sm > 0 ? per_sm : 1);
    }
    // ---- per-instance parameters: slot-ordered copies, one row per evaluated point ----
    ParamGather G{};
    CplbInstParams Q_one{}, Q_fd{}, Q_ls{};
    if (per_instance) {
        const double* const src[CPLB_NUM_INST_ARRAYS] = {per_instance->mass, per_instance->wrench, per_instance->mu, per_instance->F_thr,
                                                         per_instance->ground_z, per_instance->com_ref, per_instance->W_com, per_instance->p_ref,
                                                         per_instance->F_ref, per_instance->W_p, per_instance->W_F};
        const int nc = P.nc, len[CPLB_NUM_INST_ARRAYS] = {1, 6, 1, nc, 1, 3, 1, 3 * nc, 3 * nc, nc, nc};
        G.reps_fd = S.nf + 1;
        G.reps_ls = kCandidates;
        const size_t rows = 1 + (size_t)G.reps_fd + (size_t)G.reps_ls;
        size_t param_bytes = 0;
        for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
            if (src[a]) param_bytes += 3 * 256 + rows * (size_t)len[a] * (size_t)N * sizeof(double);
        if (param_bytes > W->param_bytes) {
            if (W->param_slab) SOLVER_CUDA(cudaFree(W->param_slab));
            W->param_slab = nullptr;
            W->param_bytes = 0;
            SOLVER_CUDA(cudaMalloc(&W->param_slab, param_bytes));
            W->param_bytes = param_bytes;
        }
        unsigned char* base = static_cast<unsigned char*>(W->param_slab);
        auto carve = [&](size_t doubles) {
            double* p = reinterpret_cast<double*>(base);
            base += align_up(doubles * sizeof(double));
            return p;
        };
        const double** one[CPLB_NUM_INST_ARRAYS] = {&Q_one.mass, &Q_one.wrench, &Q_one.mu, &Q_one.F_thr, &Q_one.ground_z, &Q_one.com_ref, &Q_one.W_com,
                                                     &Q_one.p_ref, &Q_one.F_ref, &Q_one.W_p, &Q_one.W_F};
        const double** fd[CPLB_NUM_INST_ARRAYS] = {&Q_fd.mass, &Q_fd.wrench, &Q_fd.mu, &Q_fd.F_thr, &Q_fd.ground_z, &Q_fd.com_ref, &Q_fd.W_com,
                                                    &Q_fd.p_ref, &Q_fd.F_ref, &Q_fd.W_p, &Q_fd.W_F};
        const double** ls[CPLB_NUM_INST_ARRAYS] = {&Q_ls.mass, &Q_ls.wrench, &Q_ls.mu, &Q_ls.F_thr, &Q_ls.ground_z, &Q_ls.com_ref, &Q_ls.W_com,
                                                    &Q_ls.p_ref, &Q_ls.F_ref, &Q_ls.W_p, &Q_ls.W_F};
        for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++) {
            G.src[a] = src[a];
            G.len[a] = len[a];
            if (!src[a]) continue;
            G.one[a] = carve((size_t)N * len[a]);
            G.fd[a] = carve((size_t)N * G.reps_fd * len[a]);
            G.ls[a] = carve((size_t)N * G.reps_ls * len[a]);
            *one[a] = G.one[a];
            *fd[a] = G.fd[a];
            *ls[a] = G.ls[a];
        }
    }
    DeviceEngine E{P, im_kernel, A, N, st, W, x0, x_out, lam_out, smem, smem_small, tail_limit, per_instance, G, Q_one, Q_fd, Q_ls};
    const SolveStats s = solve_loop(E, O, N, SH.nf);
    if (stats) *stats = s;
    return E.err;
}

}  // namespace solver
}  // namespace cplb
