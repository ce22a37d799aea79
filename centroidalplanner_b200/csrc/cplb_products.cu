// cplb_products.cu -- the fused Jacobian products: cplb_jacobian_products_device of include/cpl_batched.h.
//
//   reverse  x_bar = obj_factor * grad f(x) + J(x)^T lambda
//   forward  g_dot = J(x) v,  f_dot = grad f(x) . v
//
// without the Jacobian ever leaving registers.  The header states the bit contract: the results are those of a caller that
// materialises J and the gradient with cplb_eval_device and multiplies them in slot order, one IEEE multiply and one IEEE add per
// structural slot (the library is built with -fmad=false).  The only multiplies dropped are by the 1.0 identity entries, where
// the product is the factor itself.
//
// Mapping: a CTA takes a tile of 128 / nc instances.
//   1. Thread (instance, contact) evaluates the contact's Jacobian entries with contact_rows (cplb_device.cuh) into a register
//      array, numbered as in a one-contact problem (nc = 1, j = k = 0: with only CPLB_WANT_J requested, contact_rows reads no
//      per-contact parameter, and the slot numbers become compile-time constants).  Every entry of the contact's 9 columns and of
//      its own constraint rows belongs to this thread, so it finishes those x_bar columns (rows ascending) and g_dot rows
//      (columns ascending) by itself.  It leaves the terms of the cross-contact sums in shared memory: its 12 products with v
//      of the moment rows 3..5 and its 9 gradient products of f_dot.
//   2. Thread (instance, chain) runs the ten cross-contact sums, each in the contract's order: x_bar of the three CoM columns,
//      g_dot rows 0..5 and f_dot, over the contacts in the caller's vector order (the columns' order).  The CoM Jacobian block
//      is formed as eval_points_env forms it (sorted-name order).
#include <cuda_runtime.h>

#include <climits>

#include "cplb_device.cuh"
#include "cplb_products.h"

namespace cplb {
namespace {

constexpr int kThreads = 128;
constexpr int kChains = 10;  // per instance: x_bar of the 3 CoM columns, g_dot rows 0..5, f_dot
constexpr int kTerms = 21;   // per contact in shared memory: g_dot rows 3..5 x [F c0, F c1, p c0, p c1], then f_dot's 9 products

// The Jacobian of a one-contact problem: slot s (the slot arithmetic at the top of cplb_device.cuh with nc = 1) lies in local
// row row(s) -- 0..5 CentroidalStatics, 6.. the contact's own rows -- and local column col(s): 0..2 CoM, 3..5 F, 6..8 p, 9..11 n.
// A contact of any problem has these entries in the same relative order.
template <int ENV>
struct OneContact {
    static constexpr bool kEnv = ENV != CPLB_ENV_NONE_K;
    static constexpr int kNnz = kEnv ? 48 : 33;
    static constexpr int kRows = kEnv ? 6 : 2;  // the contact's own constraint rows
    __host__ __device__ static constexpr int row(int s)
    {
        if (s < 3) return s;                        // force balance
        if (s < 21) return 3 + (s - 3) / 6;          // moment rows: [CoM CoM F F p p]
        const int d = s - 21;
        if (!kEnv) return 6 + d / 6;                 // FrictionCone [F F F n n n] x 2
        if (d < 3) return 6;                         // EnvironmentConstraint [p p p]
        if (d < 15) return 7 + (d - 3) / 4;          // EnvironmentNormal [p p p n] x 3
        return 10 + (d - 15) / 6;
    }
    __host__ __device__ static constexpr int col(int s)
    {
        if (s < 3) return 3 + s;
        if (s < 21) {
            const int q = (s - 3) / 6, e = (s - 3) % 6;
            return 3 * (e / 2) + (e % 2 == 0 ? (q == 0 ? 1 : 0) : (q == 2 ? 1 : 2));  // the two columns != q of CoM, F, p
        }
        const int d = s - 21;
        if (kEnv && d < 3) return 6 + d;
        if (kEnv && d < 15) return (d - 3) % 4 < 3 ? 6 + (d - 3) % 4 : 9 + (d - 3) / 4;
        const int e = (kEnv ? d - 15 : d) % 6;
        return e < 3 ? 3 + e : 6 + e;
    }
};

// contact_rows' outputs into registers: Jacobian entries by one-contact slot, cost-gradient entries by column - col0.
struct LocalEmitter {
    double* J;
    double* gr;
    int col0;
    __device__ __forceinline__ void g(int, double) const {}
    __device__ __forceinline__ void j(int slot, double v) const { J[slot] = v; }
    __device__ __forceinline__ void grad(int col, double v) const { gr[col - col0] = v; }
};

// Phase 1: contact k (sorted rank j) of instance i.  terms: this contact's kTerms doubles in shared memory.
template <int ENV, class PS>
__device__ __forceinline__ void contact_products(const CplbParams& P, const PS& ps, const ProductArgs& A, long long i, int j, int k, double* terms)
{
    using L = OneContact<ENV>;
    const int nc = P.nc, n = P.n, m = P.m;
    const double* xi = A.x + i * n;
    const double* xk = xi + 3 + 9 * k;
    const double c[3] = {__ldg(xi + 0), __ldg(xi + 1), __ldg(xi + 2)};
    const double F[3] = {__ldg(xk + 0), __ldg(xk + 1), __ldg(xk + 2)};
    const double p[3] = {__ldg(xk + 3), __ldg(xk + 4), __ldg(xk + 5)};
    const double nn[3] = {__ldg(xk + 6), __ldg(xk + 7), __ldg(xk + 8)};
    double J[L::kNnz], gr[9];
    LocalEmitter em{J, gr, 3 + 9 * k};
    if (A.lambda || A.g_dot) contact_rows<ENV>(P, ps, em, 1, 0, 0, c, F, p, nn, CPLB_WANT_J);
    if (A.obj_factor || A.f_dot) contact_rows<ENV, true, 0, kPartStatics>(P, ps, em, nc, j, k, c, F, p, nn, CPLB_WANT_GRAD);
    const long long crow = 6 + L::kRows * j;  // the contact's first constraint row

    if (A.x_bar) {
        double xb[9];
        const double of = A.obj_factor ? __ldg(A.obj_factor + i) : 0.0;
#pragma unroll
        for (int q = 0; q < 9; q++) xb[q] = A.obj_factor ? of * gr[q] : 0.0;
        if (A.lambda) {
            const double* lam = A.lambda + i * m;
            double lr[6 + L::kRows];  // multipliers of the local rows
#pragma unroll
            for (int r = 0; r < 6; r++) lr[r] = __ldg(lam + r);
#pragma unroll
            for (int r = 0; r < L::kRows; r++) lr[6 + r] = __ldg(lam + crow + r);
#pragma unroll
            for (int s = 0; s < L::kNnz; s++) {  // slot order: per column, rows ascending
                const int cc = L::col(s);
                if (cc >= 3) xb[cc - 3] = xb[cc - 3] + J[s] * lr[L::row(s)];
            }
        }
        double* out = A.x_bar + i * n + 3 + 9 * k;
#pragma unroll
        for (int q = 0; q < 9; q++) out[q] = xb[q];
    }

    if (A.g_dot || A.f_dot) {
        const double* vk = A.v + i * n + 3 + 9 * k;
        double vl[12];  // v by local column (the CoM entries are not read here)
#pragma unroll
        for (int q = 0; q < 9; q++) vl[3 + q] = __ldg(vk + q);
        if (A.g_dot) {
            double gd[L::kRows];
#pragma unroll
            for (int r = 0; r < L::kRows; r++) gd[r] = 0.0;
#pragma unroll
            for (int s = 0; s < L::kNnz; s++) {  // slot order: per row, columns ascending
                const int cc = L::col(s), r = L::row(s);
                if (cc < 3 || r < 3) continue;  // the CoM block and the force-balance identities are the chains' (1.0 * v is v)
                const double t = J[s] * vl[cc];
                if (r >= 6) gd[r - 6] = gd[r - 6] + t;
                else terms[4 * (r - 3) + (s - 3) % 6 - 2] = t;
            }
            double* out = A.g_dot + i * m + crow;
#pragma unroll
            for (int r = 0; r < L::kRows; r++) out[r] = gd[r];
        }
        if (A.f_dot) {
#pragma unroll
            for (int q = 0; q < 9; q++) terms[12 + q] = gr[q] * vl[3 + q];
        }
    }
}

// CentroidalStatics' CoM block of row r (3..5) at x: the entries of its two CoM columns, summed over the contacts in sorted-name
// order as eval_points_env sums them (CentroidalStatics.cpp:128-133).
__device__ __forceinline__ void com_block(const CplbParams& P, const double* xi, int r, double& va, double& vb)
{
    const int ia = r == 3 ? 2 : (r == 4 ? 2 : 1), ib = r == 3 ? 1 : 0;
    const bool nega = (r == 4), negb = (r != 4);
    va = 0.0;
    vb = 0.0;
    for (int jj = 0; jj < P.nc; jj++) {
        const double* Fj = xi + 3 + 9 * P.perm[jj];
        const double fa = __ldg(Fj + ia), fb = __ldg(Fj + ib);
        va -= nega ? -fa : fa;
        vb -= negb ? -fb : fb;
    }
}

// Phase 2: chain ch of instance i.  terms: the instance's [nc][kTerms] products, contact index = vector order.
template <class PS>
__device__ __forceinline__ void instance_chain(const CplbParams& P, const PS& ps, const ProductArgs& A, long long i, int ch, const double* terms)
{
    const int nc = P.nc, n = P.n, m = P.m;
    const double* xi = A.x + i * n;
    if (ch < 3) {  // x_bar of CoM column ch: gradient, then rows 3..5 other than 3 + ch
        if (!A.x_bar) return;
        double acc = A.obj_factor ? __ldg(A.obj_factor + i) * (ps.W_com() * (__ldg(xi + ch) - ps.com_ref(ch))) : 0.0;
        if (A.lambda) {
            for (int r = 3; r < 6; r++) {
                if (r == 3 + ch) continue;
                double va, vb;
                com_block(P, xi, r, va, vb);
                acc = acc + (ch == (r == 3 ? 1 : 0) ? va : vb) * __ldg(A.lambda + i * m + r);
            }
        }
        A.x_bar[i * n + ch] = acc;
    } else if (ch < 9) {  // g_dot row r = 0..5
        if (!A.g_dot) return;
        const int r = ch - 3;
        const double* vi = A.v + i * n;
        double acc = 0.0;
        if (r < 3) {
            for (int k = 0; k < nc; k++) acc = acc + __ldg(vi + 3 + 9 * k + r);
        } else {
            double va, vb;
            com_block(P, xi, r, va, vb);
            const int q = r - 3, c0 = q == 0 ? 1 : 0, c1 = q == 2 ? 1 : 2;
            acc = acc + va * __ldg(vi + c0);
            acc = acc + vb * __ldg(vi + c1);
            for (int k = 0; k < nc; k++)
#pragma unroll
                for (int e = 0; e < 4; e++) acc = acc + terms[k * kTerms + 4 * q + e];
        }
        A.g_dot[i * m + r] = acc;
    } else {  // f_dot: the CoM gradient (eval_points_env's expression), then every contact column
        if (!A.f_dot) return;
        const double* vi = A.v + i * n;
        double acc = 0.0;
#pragma unroll
        for (int q = 0; q < 3; q++) acc = acc + (ps.W_com() * (__ldg(xi + q) - ps.com_ref(q))) * __ldg(vi + q);
        for (int k = 0; k < nc; k++)
#pragma unroll
            for (int q = 0; q < 9; q++) acc = acc + terms[k * kTerms + 12 + q];
        A.f_dot[i] = acc;
    }
}

template <int ENV, bool PER_INSTANCE>
__global__ void __launch_bounds__(kThreads, 4) k_jacobian_products(const __grid_constant__ CplbParams P, const __grid_constant__ CplbInstParams Q,
                                                                const __grid_constant__ ProductArgs A)
{
    extern __shared__ double terms[];  // [tile][nc][kTerms]
    const int nc = P.nc, tile = kThreads / nc, t = (int)threadIdx.x;
    const long long i0 = (long long)blockIdx.x * tile;
    {
        const int a = t / nc, j = t - a * nc;
        const long long i = i0 + a;
        if (a < tile && i < A.N) {
            const int k = P.perm[j];
            double* tk = terms + (a * nc + k) * kTerms;
            if (PER_INSTANCE) contact_products<ENV>(P, InstanceParams<false>{P, Q, i, 0}, A, i, j, k, tk);
            else contact_products<ENV>(P, SharedParams{P}, A, i, j, k, tk);
        }
    }
    __syncthreads();
    for (int u = t; u < tile * kChains; u += kThreads) {
        const int a = u / kChains, ch = u - a * kChains;
        const long long i = i0 + a;
        if (i >= A.N) continue;
        const double* ta = terms + a * nc * kTerms;
        if (PER_INSTANCE) instance_chain(P, InstanceParams<false>{P, Q, i, 0}, A, i, ch, ta);
        else instance_chain(P, SharedParams{P}, A, i, ch, ta);
    }
}

template <int ENV>
void launch_env(const CplbParams& P, const CplbInstParams* per_instance, const ProductArgs& A, unsigned grid, size_t smem, cudaStream_t st)
{
    const CplbInstParams Q = per_instance ? *per_instance : CplbInstParams{};
    if (per_instance) k_jacobian_products<ENV, true><<<grid, kThreads, smem, st>>>(P, Q, A);
    else k_jacobian_products<ENV, false><<<grid, kThreads, smem, st>>>(P, Q, A);
}

}  // namespace

cudaError_t launch_jacobian_products(const CplbParams& P, const CplbInstParams* per_instance, const ProductArgs& A, cudaStream_t st)
{
    const int tile = kThreads / P.nc;
    const long long blocks = (A.N + tile - 1) / tile;
    if (P.nc < 1 || P.nc > CPLB_KMAX_CONTACTS || blocks > INT_MAX) return cudaErrorInvalidConfiguration;  // (checked by the caller)
    const size_t smem = (size_t)tile * P.nc * kTerms * sizeof(double);  // at most 21 KB
    switch (P.env) {
    case CPLB_ENV_NONE_K: launch_env<CPLB_ENV_NONE_K>(P, per_instance, A, (unsigned)blocks, smem, st); break;
    case CPLB_ENV_GROUND_K: launch_env<CPLB_ENV_GROUND_K>(P, per_instance, A, (unsigned)blocks, smem, st); break;
    default: launch_env<CPLB_ENV_SUPERQUADRIC_K>(P, per_instance, A, (unsigned)blocks, smem, st); break;
    }
    return cudaGetLastError();
}

}  // namespace cplb
