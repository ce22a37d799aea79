// cplb_derivtest.cu -- the batched first-order derivative test: cplb_derivative_test_device of include/cpl_batched.h.
//
// The reference turns on IPOPT's `derivative_test first-order` before every solve (src/CentroidalPlanner.cpp:26): the Jacobian
// and the cost gradient are compared with forward differences of the problem's own g and f at the starting point.  Here that
// check runs for N instances at once, ONE CTA PER INSTANCE, fused:
//
//   1. g, Jacobian, cost and gradient at x by eval_points (cplb_eval_inline.cuh), kept in shared memory: the batched evaluator's
//      bits, so the "exact" side of every comparison is what cplb_eval_device returns.
//   2. The n perturbed points x + h_j e_j, h_j = perturbation * (|x_j| > 1 ? |x_j| : 1), in chunks of K columns: K rows of x
//      materialised in shared memory and evaluated (g and cost) by one eval_points call.  K is what the shared-memory budget
//      leaves after the point's own outputs (derivtest_chunk): every shape up to CPLB_KMAX_CONTACTS contacts fits.
//   3. fd = (g(x + h_j e_j) - g(x)) / h_j and (f(x + h_j e_j) - f(x)) / h_j, divided by h_j (not by the rounded step), as IPOPT
//      does; compared with every gradient entry and every entry of the dense m x n Jacobian, structural or not (outside the
//      structure the exact value is 0):  rel = |fd - exact| / (|exact| > 1 ? |exact| : 1), wrong iff !(rel <= tol).
//   4. Per instance: the number of wrong entries, how many of them lie outside the structure, and the worst entry -- the FIRST
//      entry, in the order gradient columns 0..n-1 then the Jacobian row by row, column ascending, with the largest rel (NaN
//      counted as +inf).  "Largest key, then smallest index" is associative and commutative, so the result does not depend on
//      which thread saw which entry or on the order of the folds.
//
// Compiled with -fmad=false like everything else: each + - * / above is one IEEE operation, which the CPU replay of the tests
// (NumPy over the C oracle) writes the same way.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <climits>

#include "cplb_derivtest.h"
#include "cplb_eval_inline.cuh"

namespace cplb {
namespace {

constexpr int kThreads = 128;
constexpr int kWarps = kThreads / 32;
// Dynamic shared memory of one CTA: below the 48 KB a CTA gets without opting in, with room for the fold's static scratch.
constexpr size_t kSmemBudget = 47 * 1024;

struct DtArgs {
    const double* x;
    const int32_t* slot_of;
    double perturbation, tol;
    int k;  // columns per chunk
    DerivTestOut out;
};

struct Worst {
    double key;  // rel, NaN counted as +inf
    double rel;  // rel as computed
    int idx;     // position in the entry order: gradient column c -> c, Jacobian (r, c) -> n + r n + c
};

__device__ __forceinline__ bool worse(const Worst& a, const Worst& b) { return a.key > b.key || (a.key == b.key && a.idx < b.idx); }

__device__ __forceinline__ double step_of(double xj, double perturbation)
{
    const double a = fabs(xj);
    return perturbation * (a > 1.0 ? a : 1.0);  // a comparison, not fmax: NaN x_j takes the perturbation itself, as on the host
}

// ENV, PER_INSTANCE: the evaluation is eval_points' (cplb_eval_inline.cuh) with its environment switch and parameter source
// resolved at compile time, so it inlines here -- the same expressions in the same order, so the same bits.  Three CTAs per SM:
// at that register budget no variant spills (the Ground one does at the unconstrained default).
template <int ENV, bool PER_INSTANCE>
__global__ void __launch_bounds__(kThreads, 3) k_derivative_test(const __grid_constant__ CplbParams P, const __grid_constant__ CplbInstParams Q,
                                                              const __grid_constant__ DtArgs A)
{
    extern __shared__ __align__(16) double smem[];
    __shared__ int s_wrong[kWarps], s_outside[kWarps], s_idx[kWarps];  // the fold's per-warp results
    __shared__ double s_key[kWarps], s_rel[kWarps];
    const int n = P.n, m = P.m, nnz = P.nnz, K = A.k;
    const int rank = (int)threadIdx.x, size = (int)blockDim.x;
    const long long inst = (long long)blockIdx.x;
    double* xs = smem;         // [n]    x
    double* g0 = xs + n;       // [m]    g(x)
    double* j0 = g0 + m;       // [nnz]  Jacobian at x
    double* f0 = j0 + nnz;     // [1]    f(x)
    double* gr0 = f0 + 1;      // [n]    gradient at x
    double* xp = gr0 + n;      // [K n]  perturbed points of the chunk
    double* gp = xp + K * n;   // [K m]  g there
    double* fp = gp + K * m;   // [K]    f there

    const double* xi = A.x + inst * n;
    for (int c = rank; c < n; c += size) xs[c] = xi[c];
    __syncthreads();
    auto eval = [&](const double* x, int count, double* g, double* jac, double* cost, double* grad, unsigned flags) {
        if (PER_INSTANCE)
            eval_points_env<ENV>(rank, size, P, InstanceParams<false>{P, Q, inst, 0}, x, count, g, jac, cost, grad, flags);
        else
            eval_points_env<ENV>(rank, size, P, SharedParams{P}, x, count, g, jac, cost, grad, flags);
    };
    eval(xs, 1, g0, j0, f0, gr0, CPLB_WANT_G | CPLB_WANT_J | CPLB_WANT_COST | CPLB_WANT_GRAD);

    int wrong = 0, outside = 0;
    Worst w{-1.0, 0.0, INT_MAX};
    for (int c0 = 0; c0 < n; c0 += K) {
        const int kc = min(K, n - c0);
        for (int t = rank; t < kc * n; t += size) {  // (the previous chunk's evaluation, the only reader of xp, has been fenced)
            const int a = t / n, e = t - a * n;
            const double v = xs[e];
            xp[t] = e == c0 + a ? v + step_of(v, A.perturbation) : v;
        }
        __syncthreads();
        eval(xp, kc, gp, nullptr, fp, nullptr, CPLB_WANT_G | CPLB_WANT_COST);
        __syncthreads();
        for (int t = rank; t < kc * (m + 1); t += size) {
            const int a = t / (m + 1), r = t - a * (m + 1) - 1, c = c0 + a;
            const double h = step_of(xs[c], A.perturbation);
            double fd, exact;
            int slot = -1, idx;
            if (r < 0) {
                fd = (fp[a] - f0[0]) / h;
                exact = gr0[c];
                idx = c;
                if (A.out.grad_fd) A.out.grad_fd[inst * n + c] = fd;
            } else {
                fd = (gp[a * m + r] - g0[r]) / h;
                slot = A.slot_of[r * n + c];
                exact = slot >= 0 ? j0[slot] : 0.0;
                idx = n + r * n + c;
                if (slot >= 0 && A.out.jac_fd) A.out.jac_fd[inst * nnz + slot] = fd;
            }
            const double ae = fabs(exact);
            const double rel = fabs(fd - exact) / (ae > 1.0 ? ae : 1.0);
            if (!(rel <= A.tol)) {
                wrong++;
                if (r >= 0 && slot < 0) outside++;
            }
            const Worst cand{isnan(rel) ? CUDART_INF : rel, rel, idx};
            if (worse(cand, w)) w = cand;
        }
    }

    // fold: a butterfly inside each warp, then thread 0 over the warps (any order gives the same: sums of counts, largest key
    // then smallest index)
    const int lane = rank & 31, warp = rank >> 5;
    for (int off = 16; off > 0; off >>= 1) {
        wrong += __shfl_xor_sync(0xffffffffu, wrong, off);
        outside += __shfl_xor_sync(0xffffffffu, outside, off);
        const Worst o{__shfl_xor_sync(0xffffffffu, w.key, off), __shfl_xor_sync(0xffffffffu, w.rel, off), __shfl_xor_sync(0xffffffffu, w.idx, off)};
        if (worse(o, w)) w = o;
    }
    if (lane == 0) {
        s_wrong[warp] = wrong;
        s_outside[warp] = outside;
        s_key[warp] = w.key;
        s_rel[warp] = w.rel;
        s_idx[warp] = w.idx;
    }
    __syncthreads();
    if (rank == 0) {
        for (int v = 1; v < kWarps; v++) {
            wrong += s_wrong[v];
            outside += s_outside[v];
            const Worst o{s_key[v], s_rel[v], s_idx[v]};
            if (worse(o, w)) w = o;
        }
        const DerivTestOut& O = A.out;
        if (O.num_wrong) O.num_wrong[inst] = wrong;
        if (O.num_wrong_outside) O.num_wrong_outside[inst] = outside;
        if (O.max_rel_error) O.max_rel_error[inst] = w.rel;
        if (O.worst_row) O.worst_row[inst] = w.idx < n ? -1 : (w.idx - n) / n;
        if (O.worst_col) O.worst_col[inst] = w.idx < n ? w.idx : (w.idx - n) % n;
    }
}

}  // namespace

size_t derivtest_smem_bytes(int n, int m, int nnz, int k)
{
    return (size_t)(2 * n + m + nnz + 1 + (size_t)k * (n + m + 1)) * sizeof(double);
}

int derivtest_chunk(int n, int m, int nnz)
{
    const long long fixed = 2LL * n + m + nnz + 1, per_column = (long long)n + m + 1;
    const long long k = ((long long)(kSmemBudget / sizeof(double)) - fixed) / per_column;
    return (int)(k < 0 ? 0 : (k > n ? n : k));
}

cudaError_t launch_derivative_test(const CplbParams& P, const CplbInstParams* per_instance, const double* x, long long N,
                                   const int32_t* slot_of, double perturbation, double tol, const DerivTestOut& out, cudaStream_t st)
{
    const int k = derivtest_chunk(P.n, P.m, P.nnz);
    if (k < 1 || N > INT_MAX) return cudaErrorInvalidConfiguration;  // (neither happens: shapes up to 32 contacts, N checked by the caller)
    const DtArgs A{x, slot_of, perturbation, tol, k, out};
    const CplbInstParams Q = per_instance ? *per_instance : CplbInstParams{};
    const size_t smem = derivtest_smem_bytes(P.n, P.m, P.nnz, k);
    const unsigned grid = (unsigned)N;
    const bool pi = per_instance != nullptr;
    switch (P.env) {
    case CPLB_ENV_NONE_K:
        if (pi) k_derivative_test<CPLB_ENV_NONE_K, true><<<grid, kThreads, smem, st>>>(P, Q, A);
        else k_derivative_test<CPLB_ENV_NONE_K, false><<<grid, kThreads, smem, st>>>(P, Q, A);
        break;
    case CPLB_ENV_GROUND_K:
        if (pi) k_derivative_test<CPLB_ENV_GROUND_K, true><<<grid, kThreads, smem, st>>>(P, Q, A);
        else k_derivative_test<CPLB_ENV_GROUND_K, false><<<grid, kThreads, smem, st>>>(P, Q, A);
        break;
    default:
        if (pi) k_derivative_test<CPLB_ENV_SUPERQUADRIC_K, true><<<grid, kThreads, smem, st>>>(P, Q, A);
        else k_derivative_test<CPLB_ENV_SUPERQUADRIC_K, false><<<grid, kThreads, smem, st>>>(P, Q, A);
        break;
    }
    return cudaGetLastError();
}

}  // namespace cplb
