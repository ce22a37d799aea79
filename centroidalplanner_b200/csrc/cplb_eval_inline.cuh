// cplb_eval_inline.cuh -- the evaluation as a device function: `count` points of ONE instance by one thread team.
//
// Same arithmetic, same order as the batched kernels (contact_rows per contact, CentroidalStatics sums and CoM block in sorted-name
// order, cost in sorted order; plain pointers instead of tiles), so its outputs are the batched evaluator's bit for bit.  Used by
// the solve round's tail kernel (cplb_solver.cu), where a handful of straggling instances iterate on their own and a kernel launch
// per evaluation would cost more than the evaluation.
#ifndef CPLB_EVAL_INLINE_CUH
#define CPLB_EVAL_INLINE_CUH

#include "cplb_device.cuh"

namespace cplb {

struct PointerEmitter {
    double* gp;
    double* jp;
    double* gradp;
    __device__ __forceinline__ void g(int row, double v) const { gp[row] = v; }
    __device__ __forceinline__ void j(int slot, double v) const { jp[slot] = v; }
    __device__ __forceinline__ void grad(int col, double v) const { gradp[col] = v; }
};

// (point, contact) pairs take the contacts' rows, (point, CentroidalStatics row) pairs the six sums and the CoM block -- each with
// the loop over contacts in sorted-name order and the expressions of the batched kernels (the row threads recompute the moment terms
// from x instead of exchanging them: the same products and differences, so the same bits) -- and one thread per point the cost.
// No thread reads what another wrote: the caller synchronises once afterwards.  x: [count][n]; outputs [count][m / nnz / 1 / n].
template <int ENV, class PS>
__device__ __forceinline__ void eval_points_env(int rank, int size, const CplbParams& P, const PS& ps, const double* x, int count, double* g,
                                                double* jac, double* cost, double* grad, unsigned flags)
{
    const int nc = P.nc, n = P.n, m = P.m, nnz = P.nnz;
    for (int t = rank; t < count * nc; t += size) {
        const int a = t / nc, j = t - a * nc, k = P.perm[j];
        const double* xa = x + (long long)a * n;
        const double* xk = xa + 3 + 9 * k;
        const double c[3] = {xa[0], xa[1], xa[2]};
        const double F[3] = {xk[0], xk[1], xk[2]}, p[3] = {xk[3], xk[4], xk[5]}, nn[3] = {xk[6], xk[7], xk[8]};
        PointerEmitter em{g ? g + (long long)a * m : nullptr, jac ? jac + (long long)a * nnz : nullptr, grad ? grad + (long long)a * n : nullptr};
        contact_rows<ENV>(P, ps, em, nc, j, k, c, F, p, nn, flags);
    }
    if (flags & (CPLB_WANT_G | CPLB_WANT_J)) {
        for (int t = rank; t < count * 6; t += size) {
            const int a = t / 6, r = t - a * 6;
            const double* xa = x + (long long)a * n;
            const double c[3] = {xa[0], xa[1], xa[2]};
            double v = 0.0;
            for (int jj = 0; jj < nc; jj++) {  // sorted-name order (CentroidalStatics.cpp:44-54)
                const double* xk = xa + 3 + 9 * P.perm[jj];
                if (r < 3) {
                    v += xk[r];
                } else {
                    const double d0 = xk[3] - c[0], d1 = xk[4] - c[1], d2 = xk[5] - c[2];
                    v += r == 3 ? d1 * xk[2] - d2 * xk[1] : (r == 4 ? d2 * xk[0] - d0 * xk[2] : d0 * xk[1] - d1 * xk[0]);  // :53
                }
            }
            if (flags & CPLB_WANT_G) g[(long long)a * m + r] = r < 3 ? (v - ps.wrench(r)) + ps.mg(r) : v - ps.wrench(r);  // :56-57
            if ((flags & CPLB_WANT_J) && r >= 3) {
                // CoM block (:128-133): row 3 <- (Fz, -Fy), row 4 <- (-Fz, Fx), row 5 <- (Fy, -Fx), each "acc -= term"
                const int ia = r == 3 ? 2 : (r == 4 ? 2 : 1), ib = r == 3 ? 1 : 0;
                const bool nega = (r == 4), negb = (r != 4);
                double va = 0.0, vb = 0.0;
                for (int jj = 0; jj < nc; jj++) {
                    const double* Fj = xa + 3 + 9 * P.perm[jj];
                    const double fa = Fj[ia], fb = Fj[ib];
                    va -= nega ? -fa : fa;
                    vb -= negb ? -fb : fb;
                }
                double* jr = jac + (long long)a * nnz + 3 * nc + (r - 3) * jac_moment_row_len(nc);
                jr[0] = va;
                jr[1] = vb;
            }
        }
    }
    if (flags & (CPLB_WANT_COST | CPLB_WANT_GRAD)) {
        for (int a = rank; a < count; a += size) {
            const double* xa = x + (long long)a * n;
            const double c[3] = {xa[0], xa[1], xa[2]};
            if (flags & CPLB_WANT_COST) {  // MinimizeCentroidalVariables.cpp:126-147: contacts in sorted order, then the CoM term
                double acc = 0.0;
                for (int jj = 0; jj < nc; jj++) {
                    const int k = P.perm[jj];
                    const double* xk = xa + 3 + 9 * k;
                    const double F[3] = {xk[0], xk[1], xk[2]}, p[3] = {xk[3], xk[4], xk[5]};
                    acc += contact_cost(ps, P.reduction_order, k, F, p);
                }
                acc += com_cost(ps, P.reduction_order, c);
                cost[a] = acc;
            }
            if (flags & CPLB_WANT_GRAD)
                for (int q = 0; q < 3; q++) grad[(long long)a * n + q] = ps.W_com() * (c[q] - ps.com_ref(q));
        }
    }
}

template <class PS>
__device__ __forceinline__ void eval_points_ps(int rank, int size, const CplbParams& P, const PS& ps, const double* x, int count, double* g,
                                               double* jac, double* cost, double* grad, unsigned flags)
{
    switch (P.env) {
    case CPLB_ENV_NONE_K: eval_points_env<CPLB_ENV_NONE_K>(rank, size, P, ps, x, count, g, jac, cost, grad, flags); break;
    case CPLB_ENV_GROUND_K: eval_points_env<CPLB_ENV_GROUND_K>(rank, size, P, ps, x, count, g, jac, cost, grad, flags); break;
    default: eval_points_env<CPLB_ENV_SUPERQUADRIC_K>(rank, size, P, ps, x, count, g, jac, cost, grad, flags); break;
    }
}

__device__ __noinline__ inline void eval_points(int rank, int size, const CplbParams& P, const CplbInstParams* Q, long long inst, const double* x, int count,
                                         double* g, double* jac, double* cost, double* grad, unsigned flags)
{
    if (Q == nullptr) {
        eval_points_ps(rank, size, P, SharedParams{P}, x, count, g, jac, cost, grad, flags);
    } else {
        eval_points_ps(rank, size, P, InstanceParams<false>{P, *Q, inst, 0}, x, count, g, jac, cost, grad, flags);
    }
}

}  // namespace cplb
#endif
