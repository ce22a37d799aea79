// cplb_solver_core.hpp -- per-instance arithmetic of the native batched solve round (SURVEY 8(f) rank 1: the caller of the
// hot path, cpl::CentroidalPlanner::Solve, src/CentroidalPlanner.cpp:22-34, for N instances in lock step).
//
// The algorithm is the primal-dual interior-point scheme of centroidalplanner_b200/lockstep_solver.py (IPOPT's method,
// Waechter & Biegler 2006: slack reformulation, log barrier, fraction to the boundary, monotone barrier update, gradient-based
// scaling, bound push / relaxation, kappa_sigma safeguard, second-order correction, l1 merit backtracking, Levenberg-Marquardt
// damping, feasibility polish; Lagrangian Hessian by forward differences of the batched gradient + Jacobian), written so that
// one THREAD TEAM works on one instance: a CTA on the GPU (cplb_solver.cu), a single thread on the host (the CPU replay of
// tests/native/solver_host_check.cpp, which puts the oracle behind the same code).  Everything an instance needs between two
// batched evaluations happens inside one team call, in shared memory: no per-operation kernel launches, no host round trips.
//
// Pattern: parallel over outputs, sequential within an output (sizes are <= 69), `team.sync()` between dependent phases.
#ifndef CPLB_SOLVER_CORE_HPP
#define CPLB_SOLVER_CORE_HPP

#include <math.h>
#include <stdint.h>
#include <string.h>

#include <vector>

#if defined(__CUDACC__)
#define CPLB_HD __host__ __device__ __forceinline__
#else
#define CPLB_HD inline
#endif

namespace cplb {
namespace solver {

constexpr int kStatusRunning = -1, kSuccess = 0, kMaxIter = 1, kInvalidNumber = 2;
constexpr int kCandidates = 30;  // line-search candidates alpha0 * 2^-k evaluated per round in one widened launch
constexpr int kMaxReg = 14;      // inertia-free regularisation attempts
constexpr double kInfBound = 1.0e19;

struct Options {
    double tol, mu_init, bound_push, bound_frac, max_gradient, constr_viol_tol, polish_viol_tol, bound_relax;
    int max_iter, max_backtracks;
    int tail_instances;  // working-set size at which the tail takes over (-1: what the GPU holds at once, 0: never)
};

// Problem-level data shared by all instances (variable / constraint bounds and the Jacobian structure are the problem's).
struct Shape {
    int n, m, nnz, nf, nk;          // nk = n + m
    const int32_t* iRow;            // [nnz]
    const int32_t* jCol;            // [nnz]
    const int32_t* col_ptr;         // [n + 1]  slots of column j: col_slot[col_ptr[j] .. col_ptr[j+1]), ascending
    const int32_t* col_slot;        // [nnz]
    const int32_t* free_idx;        // [nf]     non-fixed variables
    const double *xl, *xu;          // [n] relaxed variable bounds
    const double *xlo_orig, *xhi_orig;
    const double *cl, *cu;          // [m] original constraint bounds
    const double *cl_r, *cu_r;      // [m] relaxed
    const uint8_t *fixed, *x_lo, *x_hi;  // [n]
    const uint8_t *s_lo, *s_hi, *is_eq;  // [m]
};

// Per-instance state, instance-major arrays (element e of instance i at base[i * len + e]).
struct State {
    double *x, *s, *lam, *vxl, *vxu, *vsl, *vsu;              // iterate and multipliers
    double *mu, *tau, *delta_last, *delta_lm;                  // [N]
    int32_t *status, *iters, *polish, *active;                 // [N]
    double *f, *df, *c, *jv;                                   // raw evaluator outputs at x: cost [N], grad [N n], g [N m], jac [N nnz]
    // Working set: only the instances still running take part in a round.  list_cur[b] = instance of slot b in the current round;
    // every per-round buffer below (and xc / ev_*: the iterate handed to the evaluator and what it returned) is indexed by SLOT.
    int32_t *list_cur, *list_next;                             // [N]
    double *xc, *ev_f, *ev_df, *ev_c, *ev_jv;                  // [N n], [N], [N n], [N m], [N nnz]
    double *dc, *dobj, *sl, *su, *cu_s, *cl_s;                 // scaling and scaled slack bounds
    // step of the current round
    double *dx, *ds, *dlam, *dvxl, *dvxu, *dvsl, *dvsu, *h, *r_x, *r_s, *D;
    double *a_p, *a_d, *merit0, *Dm, *nu, *R0, *quad;
    int32_t *tiny, *pol, *okK, *accepted0;
    double *lu, *lu_dinv;                                      // [N nk nk], [N nk]: factors kept for the second-order correction
    double *jd_slot, *h0_slot;                                 // [N m n], [N n n]: dense Jacobian / Hessian of a slot (GPU: Scratch::carve)
    int32_t* piv;                                              // [N nk]
    // widened evaluation buffers
    double *x_fd, *grad_fd, *jac_fd;                           // [N (nf+1) n], [N (nf+1) n], [N (nf+1) nnz]
    double *x_ls, *g_ls, *cost_ls;                             // [N KC n], [N KC m], [N KC]
    double *x_soc, *g_soc, *cost_soc, *dx_soc, *ds_soc, *dlam_soc, *a_soc;
    int32_t* soc_valid;
    // results
    double *out_cost, *out_viol, *out_dual;
};

// A team is the set of threads that carry one instance through a phase.  rank / size / sync() as usual; the first lanes() threads
// form the team's "first warp", which folds team-shared term arrays with warp_fold (every lane gets the result; a fixed tree, so
// the result does not depend on timing).  On the host a team is one thread, and warp_fold replays the warp's tree.
struct HostTeam {
    int rank = 0, size = 1;
    void sync() const {}
    int lanes() const { return 1; }
};

constexpr int kWarp = 32;  // lanes of the GPU team's first warp (DeviceTeam::lanes)

// Fold of up to two strided index ranges by the first warp: lane l folds step1 over e = l, l + 32, ... < n1, then step2 over
// e = l, l + 32, ... < n2, from `init`; the 32 partials combine in the __shfl_xor butterfly v[l] = op(v[l], v[l ^ o]),
// o = 16, 8, 4, 2, 1.  The host (one thread) computes the same 32 partials and the same tree, so both sides return the same
// bits, signed zeros included (op's operand order is the device's).
template <class Team, class Op, class Step1, class Step2>
CPLB_HD double warp_fold(const Team& team, double init, Op op, int n1, Step1 step1, int n2, Step2 step2)
{
#if defined(__CUDA_ARCH__)
    double v = init;
    for (int e = team.rank; e < n1; e += kWarp) v = step1(v, e);
    for (int e = team.rank; e < n2; e += kWarp) v = step2(v, e);
#pragma unroll
    for (int o = kWarp / 2; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
#else
    (void)team;
    double v[kWarp], w[kWarp];
    for (int l = 0; l < kWarp; l++) {
        v[l] = init;
        for (int e = l; e < n1; e += kWarp) v[l] = step1(v[l], e);
        for (int e = l; e < n2; e += kWarp) v[l] = step2(v[l], e);
    }
    for (int o = kWarp / 2; o > 0; o >>= 1) {
        for (int l = 0; l < kWarp; l++) w[l] = op(v[l], v[l ^ o]);
        for (int l = 0; l < kWarp; l++) v[l] = w[l];
    }
    return v[0];
#endif
}

CPLB_HD bool finite_d(double v) { return v == v && v - v == 0.0; }
CPLB_HD double dmax(double a, double b) { return a > b ? a : b; }   // NaN-free callers only (torch.maximum propagates NaN: handled where it matters)
CPLB_HD double dmin(double a, double b) { return a < b ? a : b; }
CPLB_HD double dabs(double a) { return a < 0 ? -a : a; }
// torch.maximum / amax semantics: NaN wins
CPLB_HD double nanmax(double a, double b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); }
CPLB_HD double nanmin(double a, double b) { return (a != a) ? a : ((b != b) ? b : (a < b ? a : b)); }
CPLB_HD double clamp_min(double v, double lo) { return (v != v) ? v : (v < lo ? lo : v); }
CPLB_HD double clamp_max(double v, double hi) { return (v != v) ? v : (v > hi ? hi : v); }

CPLB_HD uint64_t bits_of(double v)
{
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double_as_longlong(v);
#else
    uint64_t u;
    memcpy(&u, &v, sizeof u);
    return u;
#endif
}
CPLB_HD double double_of(uint64_t u)
{
#if defined(__CUDA_ARCH__)
    return __longlong_as_double((long long)u);
#else
    double v;
    memcpy(&v, &u, sizeof v);
    return v;
#endif
}

// Natural logarithm from + - * / and exponent manipulation only, so that the GPU (-fmad=false) and the host (-ffp-contract=off)
// return the same bits; CUDA's and the C library's log are different algorithms, and the barrier terms of the merit function
// would part the two solves.  fdlibm's __ieee754_log (Sun Microsystems, 1993): x = 2^k (1 + f) with 1 + f in [sqrt(2)/2, sqrt(2)),
// log(1 + f) = 2 atanh(s), s = f / (2 + f), as a minimax polynomial in s^2, plus k ln2 as a hi/lo pair.  Error < 1 ulp;
// log(1) = 0, log(+-0) = -inf, log(x < 0) = NaN, log(inf) = inf, NaN -> NaN; subnormals are scaled by 2^54 first.
CPLB_HD double log_hd(double x)
{
    const double ln2_hi = double_of(0x3fe62e42fee00000ull), ln2_lo = double_of(0x3dea39ef35793c76ull);
    const double Lg1 = double_of(0x3fe5555555555593ull), Lg2 = double_of(0x3fd999999997fa04ull), Lg3 = double_of(0x3fd2492494229359ull),
                 Lg4 = double_of(0x3fcc71c51d8e78afull), Lg5 = double_of(0x3fc7466496cb03deull), Lg6 = double_of(0x3fc39a09d078c69full),
                 Lg7 = double_of(0x3fc2f112df3e5244ull);
    uint64_t u = bits_of(x);
    int32_t hx = (int32_t)(u >> 32);
    const uint32_t lx = (uint32_t)u;
    int k = 0;
    if (hx < 0x00100000) {                                               // x < 2^-1022
        if (((hx & 0x7fffffff) | lx) == 0) return double_of(0xfff0000000000000ull);  // log(+-0) = -inf
        if (hx < 0) return double_of(0x7ff8000000000000ull);               // log(negative) = NaN
        k -= 54;                                                           // subnormal: scale up
        x *= 18014398509481984.0;                                          // 2^54
        u = bits_of(x);
        hx = (int32_t)(u >> 32);
    }
    if (hx >= 0x7ff00000) return x + x;                                    // inf or NaN
    k += (hx >> 20) - 1023;
    hx &= 0x000fffff;
    const int32_t i = (hx + 0x95f64) & 0x100000;                           // mantissa >= sqrt(2): halve it, k + 1
    x = double_of(((uint64_t)(uint32_t)(hx | (i ^ 0x3ff00000)) << 32) | (u & 0xffffffffull));
    k += i >> 20;
    const double f = x - 1.0, dk = (double)k;
    if ((0x000fffff & (2 + hx)) < 3) {                                     // |f| < 2^-20
        if (f == 0.0) return k == 0 ? 0.0 : dk * ln2_hi + dk * ln2_lo;
        const double R = f * f * (0.5 - 0.33333333333333333 * f);
        return k == 0 ? f - R : dk * ln2_hi - ((R - dk * ln2_lo) - f);
    }
    const double s = f / (2.0 + f), z = s * s, w = z * z;
    const double t1 = w * (Lg2 + w * (Lg4 + w * Lg6)), t2 = z * (Lg1 + w * (Lg3 + w * (Lg5 + w * Lg7))), R = t2 + t1;
    if (((hx - 0x6147a) | (0x6b851 - hx)) > 0) {
        const double hfsq = 0.5 * f * f;
        return k == 0 ? f - (hfsq - s * (hfsq + R)) : dk * ln2_hi - ((hfsq - (s * (hfsq + R) + dk * ln2_lo)) - f);
    }
    return k == 0 ? f - s * (f - R) : dk * ln2_hi - ((s * (f - R) - dk * ln2_lo) - f);
}

// IPOPT's starting-point projection (Waechter & Biegler 2006, section 3.6)
CPLB_HD double push_inside(double v, double lo, double hi, bool has_lo, bool has_hi, double k1, double k2)
{
    const double span = (has_lo && has_hi) ? hi - lo : INFINITY;
    const double pl = dmin(k1 * dmax(dabs(lo), 1.0), k2 * span);
    const double pu = dmin(k1 * dmax(dabs(hi), 1.0), k2 * span);
    if (has_lo) v = nanmax(v, lo + pl);
    if (has_hi) v = nanmin(v, hi - pu);
    return v;
}

// ---- dense LU with partial pivoting of an nk x nk matrix held in team-shared memory (row-major, leading dimension ld) -------
// piv[k] = row swapped with row k at step k (LAPACK convention); dinv[k] = 1 / u_kk.  Zero pivots are not special-cased: the
// reciprocal is then inf, the factors and the solution non-finite, and the caller's regularisation loop takes over (as with
// torch's lu_factor).  Multipliers are formed as a_ik * (1 / a_kk).  Three barriers per step: pivot search (on the GPU one
// warp, strided rows + a shuffle reduction; NaN never wins, ties go to the lowest row), row swap, trailing update on a 2-D
// thread grid.  `cand` needs 64 doubles.
template <class Team>
CPLB_HD void lu_factor(const Team& team, double* A, int ld, int nk, int32_t* piv, double* dinv, double* cand)
{
    const int ntx = team.size >= 16 ? 16 : team.size, nty = team.size / ntx;
    const int tx = team.rank % ntx, ty = team.rank / ntx;
    for (int k = 0; k < nk; k++) {
#if defined(__CUDA_ARCH__)
        if (team.rank < 32) {
            int p = k;
            double best = -1.0;
            for (int r = k + team.rank; r < nk; r += 32) {
                const double v = dabs(A[r * ld + k]);
                if (v > best) {
                    best = v;
                    p = r;
                }
            }
            for (int off = 16; off > 0; off >>= 1) {
                const double ob = __shfl_down_sync(0xffffffffu, best, off);
                const int op = __shfl_down_sync(0xffffffffu, p, off);
                if (ob > best || (ob == best && op < p)) {
                    best = ob;
                    p = op;
                }
            }
            if (team.rank == 0) {
                piv[k] = p;
                dinv[k] = 1.0 / A[p * ld + k];
            }
        }
#else
        (void)cand;
        if (team.rank == 0) {
            int p = k;
            double best = -1.0;
            for (int r = k; r < nk; r++) {
                const double v = dabs(A[r * ld + k]);
                if (v > best) {
                    best = v;
                    p = r;
                }
            }
            piv[k] = p;
            dinv[k] = 1.0 / A[p * ld + k];
        }
#endif
        team.sync();
        const int p = piv[k];
        if (p != k)
            for (int c = team.rank; c < nk; c += team.size) {
                const double t = A[k * ld + c];
                A[k * ld + c] = A[p * ld + c];
                A[p * ld + c] = t;
            }
        team.sync();
        const double rp = dinv[k];
        if (ty < nty)
            for (int r = k + 1 + ty; r < nk; r += nty) {
                const double lik = A[r * ld + k] * rp;
                for (int c = k + 1 + tx; c < nk; c += ntx) A[r * ld + c] = A[r * ld + c] - lik * A[k * ld + c];
            }
        team.sync();
        // the multipliers themselves (column k below the diagonal), after every reader of a_ik is done; the two barriers of the
        // next step's pivot search and swap order these writes before any later access to column k
        for (int r = k + 1 + team.rank; r < nk; r += team.size) A[r * ld + k] = A[r * ld + k] * rp;
    }
    team.sync();
}

// solves A y = b in place (b -> y) with the factors of lu_factor; one barrier per substitution step
template <class Team>
CPLB_HD void lu_solve(const Team& team, const double* A, int ld, int nk, const int32_t* piv, const double* dinv, double* b)
{
    if (team.rank == 0)
        for (int k = 0; k < nk; k++) {
            const int p = piv[k];
            if (p != k) {
                const double t = b[k];
                b[k] = b[p];
                b[p] = t;
            }
        }
    team.sync();
    for (int k = 0; k < nk; k++) {  // L y = P b (unit lower triangle)
        const double yk = b[k];
        for (int r = k + 1 + team.rank; r < nk; r += team.size) b[r] = b[r] - A[r * ld + k] * yk;
        team.sync();
    }
    for (int k = nk - 1; k >= 0; k--) {  // U x = y: every thread forms x_k itself, thread 0 stores it
        const double xk = b[k] * dinv[k];
        for (int r = team.rank; r < k; r += team.size) b[r] = b[r] - A[r * ld + k] * xk;
        team.sync();
        if (team.rank == 0) b[k] = xk;
    }
    team.sync();
}

// shared scratch of one team, carved out of one block of doubles (shared memory on the GPU).  `full` = with the KKT matrix, the
// dense Jacobian and the Hessian (phase_kkt, phase_ls_first); the other phases only need the vectors.
struct Scratch {
    double *K, *rhs, *sol, *Jd, *H0, *w, *glb;                       // full only
    double *gxl, *gxu, *gsl, *gsu, *sigx, *sigs, *dx, *ds, *dl, *e, *red, *dinv;
    int32_t* piv;
    int ld;
    static constexpr int kTerms = 8;  // per-element term arrays in `e` (kTerms x nk)
    // returns the number of doubles used; base may be nullptr (size query)
    // jd_ext / h0_ext: where the dense Jacobian and the Hessian live when not in the team's own block (the GPU keeps them in
    // global memory, per slot: they are written once per iteration and only re-read to rebuild K, and without them a team's
    // shared memory drops from 71 KB to 49 KB at four contacts -- four teams per SM instead of three)
    CPLB_HD size_t carve(double* base, int n, int m, int nnz, bool full, double* jd_ext = nullptr, double* h0_ext = nullptr)
    {
        const int nk = n + m;
        ld = nk | 1;
        size_t o = 0;
        auto take = [&](size_t count) {
            double* p = base ? base + o : nullptr;
            o += count;
            return p;
        };
        gxl = take(n);
        gxu = take(n);
        sigx = take(n);
        dx = take(n);
        gsl = take(m);
        gsu = take(m);
        sigs = take(m);
        ds = take(m);
        dl = take(m);
        e = take((size_t)kTerms * nk);
        red = take(96);
        dinv = take(nk);
        piv = reinterpret_cast<int32_t*>(take(((size_t)nk + 1) / 2));
        K = rhs = sol = Jd = H0 = w = glb = nullptr;
        if (full) {
            K = take((size_t)nk * ld);
            rhs = take(nk);
            sol = take(nk);
            Jd = jd_ext ? jd_ext : take((size_t)m * n);
            H0 = h0_ext ? h0_ext : take((size_t)n * n);
            w = take(nnz);
            glb = take(n);
        }
        return o;
    }
    CPLB_HD double* term(int t, int nk) const { return e + (size_t)t * nk; }
};

// gaps to the bounds at (x, s) (1.0 where there is no bound)
template <class Team>
CPLB_HD void compute_gaps(const Team& team, const Shape& S, const double* x, const double* s, const double* sl, const double* su, Scratch& q)
{
    for (int j = team.rank; j < S.n; j += team.size) {
        q.gxl[j] = S.x_lo[j] ? x[j] - S.xl[j] : 1.0;
        q.gxu[j] = S.x_hi[j] ? S.xu[j] - x[j] : 1.0;
    }
    for (int r = team.rank; r < S.m; r += team.size) {
        q.gsl[r] = S.s_lo[r] ? s[r] - sl[r] : 1.0;
        q.gsu[r] = S.s_hi[r] ? su[r] - s[r] : 1.0;
    }
}

// dense scaled Jacobian with the fixed columns zeroed: Jd[r][j] = dc[r] * jac[slot]
template <class Team>
CPLB_HD void dense_jacobian(const Team& team, const Shape& S, const double* jv, const double* dc, double* Jd)
{
    for (int e = team.rank; e < S.m * S.n; e += team.size) Jd[e] = 0.0;
    team.sync();
    for (int sl_ = team.rank; sl_ < S.nnz; sl_ += team.size) {
        const int r = S.iRow[sl_], j = S.jCol[sl_];
        if (!S.fixed[j]) Jd[r * S.n + j] = dc[r] * jv[sl_];
    }
}

// ---- per-instance pointers ---------------------------------------------------------------------------------------------------
struct Inst {
    const Shape& S;
    const State& T;
    long long i;
    CPLB_HD double* vn(double* base) const { return base + i * S.n; }
    CPLB_HD double* vm(double* base) const { return base + i * S.m; }
};

CPLB_HD double scaled_df(const Inst& I, int j) { return I.S.fixed[j] ? 0.0 : I.T.dobj[I.i] * I.T.df[I.i * I.S.n + j]; }

// (J^T lam)_j with the scaled Jacobian; fixed columns contribute nothing
CPLB_HD double jt_lam(const Inst& I, int j, const double* lam)
{
    const Shape& S = I.S;
    if (S.fixed[j]) return 0.0;
    const double* jv = I.T.jv + I.i * S.nnz;
    const double* dc = I.T.dc + I.i * S.m;
    double acc = 0.0;
    for (int e = S.col_ptr[j]; e < S.col_ptr[j + 1]; e++) {
        const int sl = S.col_slot[e], r = S.iRow[sl];
        acc += (dc[r] * jv[sl]) * lam[r];
    }
    return acc;
}

// Folds over team-shared term arrays by the team's first warp (callers: threads with rank < lanes() only, all of them): each lane
// folds a strided share, the lanes combine in a fixed tree.  One thread doing these alone costs ~100 cycles per element (dependent
// fp64 compares behind shared-memory loads) -- the serial blocks were a tenth of an iteration's latency.
struct OpSum {
    CPLB_HD double operator()(double a, double b) const { return a + b; }
};
struct OpNanmax {
    CPLB_HD double operator()(double a, double b) const { return nanmax(a, b); }
};
struct OpNanmin {
    CPLB_HD double operator()(double a, double b) const { return nanmin(a, b); }
};
struct NoStep {
    CPLB_HD double operator()(double v, int) const { return v; }
};
template <class Team>
CPLB_HD double arr_nanmax(const Team& team, const double* a, int count, double init)
{
    return warp_fold(team, init, OpNanmax{}, count, [&](double v, int e) { return nanmax(v, a[e]); }, 0, NoStep{});
}
template <class Team>
CPLB_HD double arr_nanmin(const Team& team, const double* a, int count, double init)
{
    return warp_fold(team, init, OpNanmin{}, count, [&](double v, int e) { return nanmin(v, a[e]); }, 0, NoStep{});
}
template <class Team>
CPLB_HD double arr_sum(const Team& team, const double* a, int count)
{
    return warp_fold(team, 0.0, OpSum{}, count, [&](double v, int e) { return v + a[e]; }, 0, NoStep{});
}

// ---- phase 0a: project the starting point (before the first evaluation) ------------------------------------------------------
template <class Team>
CPLB_HD void phase_init_x(const Team& team, const Shape& S, const State& T, const Options& O, long long i, const double* x0)
{
    double* x = T.x + i * S.n;
    for (int j = team.rank; j < S.n; j += team.size) {
        double v = S.fixed[j] ? S.xl[j] : x0[i * S.n + j];
        v = push_inside(v, S.xl[j], S.xu[j], S.x_lo[j], S.x_hi[j], O.bound_push, O.bound_frac);
        x[j] = v;
        T.xc[i * S.n + j] = v;  // slot = instance before the first round
    }
    if (team.rank == 0) T.list_cur[i] = (int32_t)i;
}

// evaluator outputs of slot b -> the instance's own arrays
template <class Team>
CPLB_HD void fetch_evaluation(const Team& team, const Shape& S, const State& T, long long i, long long b)
{
    for (int j = team.rank; j < S.n; j += team.size) T.df[i * S.n + j] = T.ev_df[b * S.n + j];
    for (int r = team.rank; r < S.m; r += team.size) T.c[i * S.m + r] = T.ev_c[b * S.m + r];
    for (int e = team.rank; e < S.nnz; e += team.size) T.jv[i * S.nnz + e] = T.ev_jv[b * S.nnz + e];
    if (team.rank == 0) T.f[i] = T.ev_f[b];
    team.sync();
}

// ---- phase 0b: scaling, slacks, multipliers (after the first evaluation at x) -------------------------------------------------
template <class Team>
CPLB_HD void phase_init_scale(const Team& team, const Shape& S, const State& T, const Options& O, long long i)
{
    Inst I{S, T, i};
    fetch_evaluation(team, S, T, i, i);
    const double *df = I.vn(T.df), *c = I.vm(T.c), *jv = T.jv + i * S.nnz;
    double *dc = I.vm(T.dc), *sl = I.vm(T.sl), *su = I.vm(T.su), *s = I.vm(T.s);
    // gradient-based scaling at the starting point (nlp_scaling_method = gradient-based, nlp_scaling_max_gradient)
    for (int r = team.rank; r < S.m; r += team.size) dc[r] = 0.0;  // row maxima first
    team.sync();
    if (team.rank == 0) {
        bool bad = !finite_d(T.f[i]);
        double gmax = 0.0;
        for (int j = 0; j < S.n; j++) {
            if (S.fixed[j]) continue;
            if (!finite_d(df[j])) bad = true;
            else gmax = dmax(gmax, dabs(df[j]));
        }
        for (int sl_ = 0; sl_ < S.nnz; sl_++) {
            if (S.fixed[S.jCol[sl_]]) continue;
            const double v = jv[sl_];
            if (!finite_d(v)) bad = true;
            else dc[S.iRow[sl_]] = dmax(dc[S.iRow[sl_]], dabs(v));
        }
        for (int r = 0; r < S.m; r++) {
            if (!finite_d(c[r])) bad = true;
            dc[r] = dmin(O.max_gradient / dmax(dc[r], 1e-300), 1.0);
        }
        T.dobj[i] = dmin(O.max_gradient / dmax(gmax, 1e-300), 1.0);
        T.status[i] = bad ? kInvalidNumber : kStatusRunning;
        if (bad) {  // no round measures a rejected start: its residuals are NaN (include/cpl_batched.h)
            T.out_viol[i] = double_of(0x7ff8000000000000ull);
            T.out_dual[i] = double_of(0x7ff8000000000000ull);
        }
        T.iters[i] = 0;
        T.polish[i] = 0;
        T.active[i] = bad ? 0 : 1;
        T.mu[i] = O.mu_init;
        T.tau[i] = 0.99;
        T.delta_last[i] = 0.0;
        T.delta_lm[i] = 0.0;
    }
    team.sync();
    for (int r = team.rank; r < S.m; r += team.size) {
        sl[r] = dc[r] * S.cl_r[r];
        su[r] = dc[r] * S.cu_r[r];
        I.vm(T.cu_s)[r] = dc[r] * S.cu[r];
        I.vm(T.cl_s)[r] = dc[r] * S.cl[r];
        const double cs = dc[r] * c[r];
        s[r] = S.is_eq[r] ? sl[r] : push_inside(cs, sl[r], su[r], S.s_lo[r], S.s_hi[r], O.bound_push, O.bound_frac);
        I.vm(T.lam)[r] = 0.0;
        I.vm(T.vsl)[r] = S.s_lo[r] ? 1.0 : 0.0;
        I.vm(T.vsu)[r] = S.s_hi[r] ? 1.0 : 0.0;
    }
    for (int j = team.rank; j < S.n; j += team.size) {
        I.vn(T.vxl)[j] = S.x_lo[j] ? 1.0 : 0.0;
        I.vn(T.vxu)[j] = S.x_hi[j] ? 1.0 : 0.0;
    }
}

// ---- phase 1: start of a round -------------------------------------------------------------------------------------------------
// (after the evaluation at the new x) kappa_sigma safeguard of the bound multipliers, convergence test, barrier update, and the
// forward-difference points of the Hessian.  Returns through T.active[i]; *n_active counts the instances still running.
template <class Team>
CPLB_HD void phase_round_begin(const Team& team, const Shape& S, const State& T, const Options& O, long long b_prev, Scratch& q, int first_round,
                               int last_round, int* n_active, bool fixed_slot = false)
{
    const long long i = T.list_cur[b_prev];  // the working set of the previous round, in its slot order
    Inst I{S, T, i};
    const int n = S.n, m = S.m, nk = S.nk;
    if (T.status[i] >= 0) {  // finished earlier (only before the first round: a bad starting point)
        if (team.rank == 0) T.active[i] = 0;
        return;
    }
    if (!first_round) fetch_evaluation(team, S, T, i, b_prev);  // (the first round's evaluation was fetched by phase_init_scale)
    double *x = I.vn(T.x), *s = I.vm(T.s);
    double *vxl = I.vn(T.vxl), *vxu = I.vn(T.vxu), *vsl = I.vm(T.vsl), *vsu = I.vm(T.vsu);
    const double *lam = I.vm(T.lam), *c = I.vm(T.c), *dc = I.vm(T.dc), *sl = I.vm(T.sl), *su = I.vm(T.su);
    compute_gaps(team, S, x, s, sl, su, q);
    team.sync();
    // term arrays: 0 |residual|, 1 multiplier sums, 2 primal infeasibility / row violation, 3..6 gap x multiplier products
    double *t_res = q.term(0, nk), *t_sum = q.term(1, nk), *t_prim = q.term(2, nk), *t_viol = q.term(3, nk);
    double *p_xl = q.term(4, nk), *p_xu = q.term(5, nk), *p_sl = q.term(6, nk), *p_su = q.term(7, nk);
    const double mu_old = T.mu[i], ks = 1e10;
    for (int j = team.rank; j < n; j += team.size) {
        double a = vxl[j], b = vxu[j];
        if (!first_round) {  // kappa_sigma safeguard (Waechter & Biegler eq. 16) with the gaps at the new point
            a = S.x_lo[j] ? nanmin(nanmax(a, mu_old / (ks * q.gxl[j])), ks * mu_old / q.gxl[j]) : 0.0;
            b = S.x_hi[j] ? nanmin(nanmax(b, mu_old / (ks * q.gxu[j])), ks * mu_old / q.gxu[j]) : 0.0;
            vxl[j] = a;
            vxu[j] = b;
        }
        const double rx = S.fixed[j] ? 0.0 : (scaled_df(I, j) + jt_lam(I, j, lam) - a + b);
        t_res[j] = dabs(rx);
        t_sum[j] = a + b;
        p_xl[j] = S.x_lo[j] ? q.gxl[j] * a : -1.0;  // -1: no bound (products are >= 0 otherwise)
        p_xu[j] = S.x_hi[j] ? q.gxu[j] * b : -1.0;
    }
    for (int r = team.rank; r < m; r += team.size) {
        double a = vsl[r], b = vsu[r];
        if (!first_round) {
            a = S.s_lo[r] ? nanmin(nanmax(a, mu_old / (ks * q.gsl[r])), ks * mu_old / q.gsl[r]) : 0.0;
            b = S.s_hi[r] ? nanmin(nanmax(b, mu_old / (ks * q.gsu[r])), ks * mu_old / q.gsu[r]) : 0.0;
            vsl[r] = a;
            vsu[r] = b;
        }
        const double rs = S.is_eq[r] ? 0.0 : (-lam[r] - a + b);
        const double cs = dc[r] * c[r];
        t_res[n + r] = dabs(rs);
        t_sum[n + r] = dabs(lam[r]) + a + b;
        t_prim[r] = dabs(cs - s[r]);
        t_viol[r] = (clamp_min(sl[r] - cs, 0.0) + clamp_min(cs - su[r], 0.0)) / dc[r];
        p_sl[r] = S.s_lo[r] ? q.gsl[r] * a : -1.0;
        p_su[r] = S.s_hi[r] ? q.gsu[r] * b : -1.0;
    }
    team.sync();
    if (team.rank < team.lanes()) {  // the first warp folds; its lane 0 decides
        const double sd = clamp_min(arr_sum(team, t_sum, nk) / (double)(m + 2 * n + 2 * m), 100.0) / 100.0;
        const double dual = arr_nanmax(team, t_res, nk, 0.0) / sd, prim = arr_nanmax(team, t_prim, m, 0.0);
        auto comp = [&](double mu) {  // max |gap x multiplier - mu| over the bounded components, / sd
            const auto xs = [&](double e, int j) {
                if (p_xl[j] != -1.0) e = nanmax(e, dabs(p_xl[j] - mu));
                if (p_xu[j] != -1.0) e = nanmax(e, dabs(p_xu[j] - mu));
                return e;
            };
            const auto ss = [&](double e, int r) {
                if (p_sl[r] != -1.0) e = nanmax(e, dabs(p_sl[r] - mu));
                if (p_su[r] != -1.0) e = nanmax(e, dabs(p_su[r] - mu));
                return e;
            };
            return warp_fold(team, 0.0, OpNanmax{}, n, xs, m, ss) / sd;
        };
        const double E0 = nanmax(nanmax(dual, prim), comp(0.0));
        const double vmax = arr_nanmax(team, t_viol, m, 0.0);
        // barrier update candidates need comp(mu) from every lane: evaluate the (uniform) recursion on all lanes
        double mu_next = mu_old;
        {
            const double dp0 = nanmax(dual, prim);
            for (int rep = 0; rep < 4; rep++) {
                const double Emu = nanmax(dp0, comp(mu_next));
                if (Emu <= 10.0 * mu_next && mu_next > O.tol / 10.0) mu_next = dmax(dmin(0.2 * mu_next, mu_next * sqrt(mu_next)), O.tol / 10.0);  // mu^1.5
            }
        }
      if (team.rank == 0) {
        // IPOPT's test (scaled error <= tol, unscaled violation <= constr_viol_tol) switches the instance to the feasibility
        // polish; it is done when the constraints hold to polish_viol_tol as well.  The polish moves x with the multipliers
        // frozen, so the test must still hold where it ends: a polished iterate that lost it (the scaled error grew past tol)
        // leaves the polish and takes Newton steps again, undamped (the polish's line searches raise the Levenberg-Marquardt
        // damping; kept, it stalls the Newton steps of a degenerate problem) -- SUCCEEDED always means E0 <= tol at the returned
        // iterate.
        if (E0 <= O.tol && vmax <= O.constr_viol_tol) T.polish[i] = 1;
        else if (T.polish[i] && vmax <= O.polish_viol_tol) { T.polish[i] = 0; T.delta_lm[i] = 0.0; }
        if (T.polish[i] && vmax <= O.polish_viol_tol) T.status[i] = kSuccess;
        else if (!finite_d(E0)) T.status[i] = kInvalidNumber;
        T.out_dual[i] = dual;
        T.out_viol[i] = vmax;
        int active = T.status[i] < 0;
        if (active && last_round) {
            T.status[i] = kMaxIter;
            active = 0;
        }
        if (active) {
            T.iters[i] += 1;
            // monotone barrier update (Waechter & Biegler eq. 7): computed above by the whole warp
            const double mu = mu_next;
            T.mu[i] = mu;
            T.tau[i] = dmax(1.0 - mu, 0.99);
            // slot in the working set of this round (the tail kernel keeps an instance in its slot: nobody else is waiting)
            int slot = (int)b_prev;
            if (!fixed_slot) {
#if defined(__CUDA_ARCH__)
                slot = atomicAdd(n_active, 1);
#else
                slot = (*n_active)++;
#endif
                T.list_next[slot] = (int32_t)i;
            }
            q.red[1] = (double)slot;
        }
        T.active[i] = active;
        q.red[0] = (double)active;
      }
    }
    team.sync();
    // forward-difference points of the Lagrangian Hessian: point a < nf perturbs free variable a, point nf is x itself
    if (q.red[0] != 0.0) {
        double* X = T.x_fd + (long long)q.red[1] * (S.nf + 1) * n;
        for (int a = 0; a <= S.nf; a++)
            for (int j = team.rank; j < n; j += team.size) {
                double v = x[j];
                if (a < S.nf && S.free_idx[a] == j) v += 1e-7 * dmax(dabs(v), 1.0);
                X[a * n + j] = v;
            }
    }
}

// ---- phase 2: Hessian, KKT system, regularised Newton step, line-search set-up ------------------------------------------------
template <class Team>
CPLB_HD void phase_kkt(const Team& team, const Shape& S, const State& T, const Options& O, long long b, Scratch& q)
{
    const long long i = T.list_cur[b];
    Inst I{S, T, i};
    const int n = S.n, m = S.m, nk = S.nk, ld = q.ld;
    double* Xls = T.x_ls + b * (long long)kCandidates * n;
    double *x = I.vn(T.x), *s = I.vm(T.s);
    const double *lam = I.vm(T.lam), *dc = I.vm(T.dc), *sl = I.vm(T.sl), *su = I.vm(T.su);
    const double *vxl = I.vn(T.vxl), *vxu = I.vn(T.vxu), *vsl = I.vm(T.vsl), *vsu = I.vm(T.vsu), *c = I.vm(T.c);
    const double mu = T.mu[i], tau = T.tau[i], dobj = T.dobj[i];
    double *h = I.vm(T.h), *r_x = I.vn(T.r_x), *r_s = I.vm(T.r_s), *D = I.vm(T.D);
    // shared copies of what the dense phases read repeatedly: term arrays 0 = r_x | r_s (nk), 1 = h (m) | D (m at +m... separate), see below
    double *s_rx = q.term(0, nk), *s_rs = s_rx + n, *s_h = q.term(1, nk), *s_D = q.term(2, nk);

    compute_gaps(team, S, x, s, sl, su, q);
    dense_jacobian(team, S, T.jv + i * S.nnz, dc, q.Jd);
    for (int sl_ = team.rank; sl_ < S.nnz; sl_ += team.size) q.w[sl_] = dc[S.iRow[sl_]] * lam[S.iRow[sl_]];
    team.sync();

    // Lagrangian Hessian by forward differences: grad L at point a = dobj * grad f + sum_slots jac[slot] * (dc lam)[row(slot)]
    const double* gfd = T.grad_fd + b * (long long)(S.nf + 1) * n;
    const double* jfd = T.jac_fd + b * (long long)(S.nf + 1) * S.nnz;
    auto grad_lagrangian = [&](int a, int j) -> double {
        if (S.fixed[j]) return 0.0;
        double acc = dobj * gfd[(long long)a * n + j];
        const double* ja = jfd + (long long)a * S.nnz;
        for (int e = S.col_ptr[j]; e < S.col_ptr[j + 1]; e++) acc += ja[S.col_slot[e]] * q.w[S.col_slot[e]];
        return acc;
    };
    for (int j = team.rank; j < n; j += team.size) q.glb[j] = grad_lagrangian(S.nf, j);
    team.sync();
    {
        // thread grid (rows a, columns j): K's top-left block is the staging area for Hc
        const int ntx = team.size >= 32 ? 32 : team.size, nty = team.size / ntx;
        const int tx = team.rank % ntx, ty = team.rank / ntx;
        if (ty < nty)
            for (int a = ty; a < S.nf; a += nty) {
                const int row = S.free_idx[a];
                const double eps = 1e-7 * dmax(dabs(x[row]), 1.0);
                for (int j = tx; j < n; j += ntx) q.K[row * ld + j] = S.fixed[j] ? 0.0 : (grad_lagrangian(a, j) - q.glb[j]) / eps;
            }
    }
    for (int j = team.rank; j < n; j += team.size) q.sigx[j] = (S.x_lo[j] ? vxl[j] / q.gxl[j] : 0.0) + (S.x_hi[j] ? vxu[j] / q.gxu[j] : 0.0);
    for (int r = team.rank; r < m; r += team.size) q.sigs[r] = (S.s_lo[r] ? vsl[r] / q.gsl[r] : 0.0) + (S.s_hi[r] ? vsu[r] / q.gsu[r] : 0.0);
    team.sync();
    // W = (Hc + Hc^T) / 2 on the free variables;  H0 = W + diag(sigma_x on the free ones, 1 on the fixed ones)
    for (int a = 0; a < n; a++)
        for (int b = team.rank; b < n; b += team.size) {
            double v = 0.0;
            if (!S.fixed[a] && !S.fixed[b]) v = 0.5 * (q.K[a * ld + b] + q.K[b * ld + a]);
            if (a == b) v += S.fixed[a] ? 1.0 : q.sigx[a];
            q.H0[a * n + b] = v;
        }
    // residuals of the barrier problem
    for (int j = team.rank; j < n; j += team.size)
        s_rx[j] = S.fixed[j] ? 0.0
                             : (scaled_df(I, j) + jt_lam(I, j, lam) - (S.x_lo[j] ? mu / q.gxl[j] : 0.0) + (S.x_hi[j] ? mu / q.gxu[j] : 0.0));
    for (int r = team.rank; r < m; r += team.size) {
        s_rs[r] = S.is_eq[r] ? 0.0 : (-lam[r] - (S.s_lo[r] ? mu / q.gsl[r] : 0.0) + (S.s_hi[r] ? mu / q.gsu[r] : 0.0));
        s_h[r] = dc[r] * c[r] - s[r];
        s_D[r] = S.is_eq[r] ? 0.0 : 1.0 / clamp_min(q.sigs[r], 1e-300);
    }
    team.sync();
    for (int j = team.rank; j < n; j += team.size) r_x[j] = s_rx[j];  // kept for the second-order correction
    for (int r = team.rank; r < m; r += team.size) {
        r_s[r] = s_rs[r];
        h[r] = s_h[r];
        D[r] = s_D[r];
    }
    const double delta_c = 1e-8 * sqrt(sqrt(mu));  // mu^0.25 (IEEE sqrt: the same bits on both sides, unlike pow)
    double* t_dx = q.term(3, nk);   // candidate step [dx | ds]
    double* t_hdx = q.term(4, nk);  // H dx

    // inertia-free regularisation (Chiang & Zavala 2016): raise delta_w until the step sees positive curvature
    double delta = T.delta_lm[i];
    for (int reg = 0; reg < kMaxReg; reg++) {
        // K = [[H0 + delta I_free, Jf^T], [Jf, -(D + delta_c)]],  rhs = [-r_x, -h - D r_s]
        if (team.rank == 0) q.red[0] = 1.0;
        team.sync();
        bool fin = true;
        for (int a = 0; a < nk; a++)
            for (int b = team.rank; b < nk; b += team.size) {
                double v;
                if (a < n && b < n) v = q.H0[a * n + b] + ((a == b && !S.fixed[a]) ? delta : 0.0);
                else if (a < n) v = q.Jd[(b - n) * n + a];
                else if (b < n) v = q.Jd[(a - n) * n + b];
                else v = (a == b) ? -(s_D[a - n] + delta_c) : 0.0;
                q.K[a * ld + b] = v;
                fin = fin && finite_d(v);
            }
        for (int a = team.rank; a < nk; a += team.size) {
            const double v = a < n ? -s_rx[a] : -s_h[a - n] - s_D[a - n] * s_rs[a - n];
            q.rhs[a] = v;
            fin = fin && finite_d(v);
        }
        if (!fin) q.red[0] = 0.0;
        team.sync();
        const bool okK = q.red[0] != 0.0;
        if (!okK) {  // identity system, zero right-hand side: a zero step (the Python driver's eyeK)
            for (int a = 0; a < nk; a++)
                for (int b = team.rank; b < nk; b += team.size) q.K[a * ld + b] = (a == b) ? 1.0 : 0.0;
            for (int a = team.rank; a < nk; a += team.size) q.rhs[a] = 0.0;
            team.sync();
        }
        lu_factor(team, q.K, ld, nk, q.piv, q.dinv, q.red + 16);
        for (int a = team.rank; a < nk; a += team.size) q.sol[a] = q.rhs[a];
        team.sync();
        lu_solve(team, q.K, ld, nk, q.piv, q.dinv, q.sol);
        // candidate step and the curvature it sees
        for (int j = team.rank; j < n; j += team.size) t_dx[j] = S.fixed[j] ? 0.0 : q.sol[j];
        for (int r = team.rank; r < m; r += team.size) t_dx[n + r] = S.is_eq[r] ? 0.0 : s_D[r] * (q.sol[n + r] - s_rs[r]);
        team.sync();
        for (int j = team.rank; j < n; j += team.size) {  // (H dx)_j, H = H0 + delta on the free diagonal
            double acc = 0.0;
            for (int b = 0; b < n; b++) acc += (q.H0[j * n + b] + ((j == b && !S.fixed[j]) ? delta : 0.0)) * t_dx[b];
            t_hdx[j] = acc;
        }
        team.sync();
        if (team.rank == 0) {
            bool sfin = true;
            double quad = 0.0, nrm = 0.0;
            for (int a = 0; a < nk; a++) sfin = sfin && finite_d(q.sol[a]);
            for (int j = 0; j < n; j++) {
                quad += t_dx[j] * t_hdx[j];
                nrm += t_dx[j] * t_dx[j];
            }
            for (int r = 0; r < m; r++) {
                quad += q.sigs[r] * t_dx[n + r] * t_dx[n + r];
                nrm += t_dx[n + r] * t_dx[n + r];
            }
            const bool good = sfin && quad >= 1e-8 * nrm;
            q.red[1] = (good || reg == kMaxReg - 1) ? 1.0 : 0.0;
            q.red[2] = quad;
        }
        team.sync();
        if (q.red[1] != 0.0) {
            for (int j = team.rank; j < n; j += team.size) q.dx[j] = t_dx[j];
            for (int r = team.rank; r < m; r += team.size) {
                q.ds[r] = t_dx[n + r];
                q.dl[r] = q.sol[n + r];
            }
            if (team.rank == 0) {
                T.quad[i] = q.red[2];
                T.delta_last[i] = delta;
                T.okK[i] = okK ? 1 : 0;
            }
            break;
        }
        delta = dmax(delta * 8.0, 1e-4);
        team.sync();
    }
    team.sync();
    const double quad = q.red[2];
    // the factors stay for the second-order correction
    {
        double* LU = T.lu + i * (long long)nk * nk;
        for (int a = 0; a < nk; a++)
            for (int b = team.rank; b < nk; b += team.size) LU[a * nk + b] = q.K[a * ld + b];
        for (int a = team.rank; a < nk; a += team.size) {
            T.piv[i * nk + a] = q.piv[a];
            T.lu_dinv[i * nk + a] = q.dinv[a];
        }
    }
    if (team.rank == 0) {
        bool bad = false;
        for (int j = 0; j < n; j++) bad = bad || !finite_d(q.dx[j]);
        for (int r = 0; r < m; r++) bad = bad || !finite_d(q.dl[r]);
        q.red[3] = bad ? 1.0 : 0.0;
    }
    team.sync();
    if (q.red[3] != 0.0) {
        for (int j = team.rank; j < n; j += team.size) q.dx[j] = 0.0;
        for (int r = team.rank; r < m; r += team.size) q.ds[r] = q.dl[r] = 0.0;
        team.sync();
    }

    // multiplier steps and the fraction-to-the-boundary limit of the dual step (with the Newton step, also for polishing instances:
    // their dual step length is zero anyway); merit-function quantities of the Newton step
    double *dvxl = I.vn(T.dvxl), *dvxu = I.vn(T.dvxu), *dvsl = I.vm(T.dvsl), *dvsu = I.vm(T.dvsu);
    double *t_ad = q.term(3, nk), *t_lb = q.term(4, nk), *t_dphi = q.term(5, nk), *t_h1 = q.term(6, nk), *t_lmax = q.term(7, nk);
    auto ms = [&](double val, double dval, bool mask, double cur) {  // largest a with val + a dval >= (1 - tau) val
        if (mask && dval < 0) cur = nanmin(cur, -tau * val / dval);
        return cur;
    };
    for (int j = team.rank; j < n; j += team.size) {
        const double a = S.x_lo[j] ? (mu / q.gxl[j] - vxl[j] - vxl[j] / q.gxl[j] * q.dx[j]) : 0.0;
        const double b = S.x_hi[j] ? (mu / q.gxu[j] - vxu[j] + vxu[j] / q.gxu[j] * q.dx[j]) : 0.0;
        dvxl[j] = a;
        dvxu[j] = b;
        t_ad[j] = ms(vxu[j], b, S.x_hi[j], ms(vxl[j], a, S.x_lo[j], INFINITY));
        t_lb[j] = (S.x_lo[j] ? log_hd(q.gxl[j]) : 0.0) + (S.x_hi[j] ? log_hd(q.gxu[j]) : 0.0);
        const double gphi = S.fixed[j] ? 0.0 : (scaled_df(I, j) - (S.x_lo[j] ? mu / q.gxl[j] : 0.0) + (S.x_hi[j] ? mu / q.gxu[j] : 0.0));
        t_dphi[j] = gphi * q.dx[j];
    }
    for (int r = team.rank; r < m; r += team.size) {
        const double a = S.s_lo[r] ? (mu / q.gsl[r] - vsl[r] - vsl[r] / q.gsl[r] * q.ds[r]) : 0.0;
        const double b = S.s_hi[r] ? (mu / q.gsu[r] - vsu[r] + vsu[r] / q.gsu[r] * q.ds[r]) : 0.0;
        dvsl[r] = a;
        dvsu[r] = b;
        t_ad[n + r] = ms(vsu[r], b, S.s_hi[r], ms(vsl[r], a, S.s_lo[r], INFINITY));
        t_lb[n + r] = (S.s_lo[r] ? log_hd(q.gsl[r]) : 0.0) + (S.s_hi[r] ? log_hd(q.gsu[r]) : 0.0);
        const double gphi = S.is_eq[r] ? 0.0 : (-(S.s_lo[r] ? mu / q.gsl[r] : 0.0) + (S.s_hi[r] ? mu / q.gsu[r] : 0.0));
        t_dphi[n + r] = gphi * q.ds[r];
        t_h1[r] = dabs(s_h[r]);
        t_lmax[r] = dabs(lam[r] + q.dl[r]);
    }
    team.sync();
    const bool pol = T.polish[i] != 0;
    if (team.rank < team.lanes()) {
        const double h1 = arr_sum(team, t_h1, m), dphi = arr_sum(team, t_dphi, nk), lb = arr_sum(team, t_lb, nk), lmax = arr_nanmax(team, t_lmax, m, 0.0);
        const double a_d_min = arr_nanmin(team, t_ad, nk, INFINITY);
      if (team.rank == 0) {
        const double phi0 = dobj * T.f[i] - mu * lb;
        const double nu_need = (dphi + 0.5 * clamp_min(quad, 0.0)) / (0.9 * clamp_min(h1, 1e-300));
        const double nu = nanmax(clamp_min(nu_need, 0.0), lmax) * 1.1 + 1e-3;
        T.nu[i] = nu;
        T.Dm[i] = dphi - nu * h1;
        T.merit0[i] = phi0 + nu * h1;
        T.a_d[i] = pol ? 0.0 : clamp_max(a_d_min, 1.0);
        T.pol[i] = pol ? 1 : 0;
      }
    }
    team.sync();

    // feasibility polish: minimum-norm Newton step on x only (multipliers stay), on the equality rows and on the inequality
    // rows that sit beyond their ORIGINAL bound
    if (pol) {
        const double *cu_s = I.vm(T.cu_s), *cl_s = I.vm(T.cl_s);
        double* act = q.term(3, nk);  // [m]
        double* r_p = q.term(4, nk);  // [m]
        for (int r = team.rank; r < m; r += team.size) {
            const double cs = dc[r] * c[r];
            const bool over = !S.is_eq[r] && S.s_hi[r] && cs > cu_s[r], under = !S.is_eq[r] && S.s_lo[r] && cs < cl_s[r];
            act[r] = (S.is_eq[r] || over || under) ? 1.0 : 0.0;
            r_p[r] = over ? cs - cu_s[r] : (under ? cs - cl_s[r] : (S.is_eq[r] ? cs - sl[r] : 0.0));
        }
        if (team.rank == 0) q.red[4] = 1.0;
        team.sync();
        bool fin = true;
        for (int a = 0; a < m; a++)
            for (int b = team.rank; b < m; b += team.size) {  // M = Je Je^T + diag((1 - act) + 1e-14)
                double acc = 0.0;
                if (act[a] != 0.0 && act[b] != 0.0)
                    for (int j = 0; j < n; j++) acc += q.Jd[a * n + j] * q.Jd[b * n + j];
                if (a == b) acc += (1.0 - act[a]) + 1e-14;
                q.K[a * ld + b] = acc;
                fin = fin && finite_d(acc);
            }
        if (!fin) q.red[4] = 0.0;
        team.sync();
        if (q.red[4] == 0.0) {
            for (int a = 0; a < m; a++)
                for (int b = team.rank; b < m; b += team.size) q.K[a * ld + b] = (a == b) ? 1.0 : 0.0;
            team.sync();
        }
        for (int r = team.rank; r < m; r += team.size) q.sol[r] = r_p[r];
        lu_factor(team, q.K, ld, m, q.piv, q.dinv, q.red + 16);
        lu_solve(team, q.K, ld, m, q.piv, q.dinv, q.sol);
        for (int j = team.rank; j < n; j += team.size) {
            double acc = 0.0;
            for (int r = 0; r < m; r++)
                if (act[r] != 0.0) acc += q.Jd[r * n + j] * q.sol[r];
            q.rhs[j] = S.fixed[j] ? 0.0 : -acc;
        }
        team.sync();
        if (team.rank == 0) {
            bool f2 = true;
            for (int j = 0; j < n; j++) f2 = f2 && finite_d(q.rhs[j]);
            q.red[5] = f2 ? 1.0 : 0.0;
        }
        team.sync();
        for (int j = team.rank; j < n; j += team.size) q.dx[j] = q.red[5] != 0.0 ? q.rhs[j] : 0.0;
        for (int r = team.rank; r < m; r += team.size) q.ds[r] = q.dl[r] = 0.0;
        team.sync();
    }

    // primal fraction-to-the-boundary step length, tiny-step flag, polish residual; the step goes to global memory
    double *dx = I.vn(T.dx), *ds = I.vm(T.ds), *dlam = I.vm(T.dlam);
    double *t_ap = q.term(3, nk), *t_tiny = q.term(4, nk), *t_R0 = q.term(5, nk);
    const double *cu_s = I.vm(T.cu_s), *cl_s = I.vm(T.cl_s);
    for (int j = team.rank; j < n; j += team.size) {
        dx[j] = q.dx[j];
        t_ap[j] = ms(q.gxu[j], -q.dx[j], S.x_hi[j], ms(q.gxl[j], q.dx[j], S.x_lo[j], INFINITY));
        t_tiny[j] = dabs(q.dx[j]) / (1.0 + dabs(x[j]));
    }
    for (int r = team.rank; r < m; r += team.size) {
        ds[r] = q.ds[r];
        dlam[r] = q.dl[r];
        t_ap[n + r] = pol ? INFINITY : ms(q.gsu[r], -q.ds[r], S.s_hi[r], ms(q.gsl[r], q.ds[r], S.s_lo[r], INFINITY));
        const double cs = dc[r] * c[r];
        t_R0[r] = S.is_eq[r] ? dabs(cs - sl[r]) : ((S.s_hi[r] ? clamp_min(cs - cu_s[r], 0.0) : 0.0) + (S.s_lo[r] ? clamp_min(cl_s[r] - cs, 0.0) : 0.0));
    }
    team.sync();
    if (team.rank < team.lanes()) {
        const double a_p = clamp_max(arr_nanmin(team, t_ap, nk, INFINITY), 1.0);
        const double tiny_max = arr_nanmax(team, t_tiny, n, 0.0), R0 = arr_nanmax(team, t_R0, m, 0.0);
        if (team.rank == 0) {
            T.a_p[i] = a_p;
            T.tiny[i] = tiny_max < 1e-13 ? 1 : 0;
            T.R0[i] = R0;
            q.red[6] = a_p;
        }
    }
    team.sync();
    // line-search candidates x + alpha0 2^-k dx, k = 0 .. kCandidates - 1
    const double a0 = q.red[6];
    for (int k = 0; k < kCandidates; k++) {
        const double al = a0 * ldexp(1.0, -k);
        for (int j = team.rank; j < n; j += team.size) Xls[k * n + j] = x[j] + al * q.dx[j];
    }
}

// Merit test of one trial point by the whole team: row values ct (scaled), slacks by the reset rule.  Writes the trial slacks to
// st_out (team-shared, m) and returns (to every thread) ok / ct_finite.  Needs term arrays 0..2 of q.
struct Trial {
    bool ok, ct_finite;
};
template <class Team>
CPLB_HD Trial merit_test(const Team& team, const Inst& I, Scratch& q, const double* X, const double* g_raw, double cost_raw, const double* S_lin,
                         double AL, double* st_out)
{
    const Shape& S = I.S;
    const State& T = I.T;
    const long long i = I.i;
    const int n = S.n, m = S.m, nk = S.nk;
    const double *dc = I.vm(T.dc), *sl = I.vm(T.sl), *su = I.vm(T.su), *s = I.vm(T.s), *cu_s = I.vm(T.cu_s), *cl_s = I.vm(T.cl_s);
    const double mu = T.mu[i], nu = T.nu[i], keep = mu / nu;
    const bool pol = T.pol[i] != 0;
    double *t_lb = q.term(0, nk), *t_viol = q.term(1, nk), *t_bad = q.term(2, nk);
    for (int j = team.rank; j < n; j += team.size) t_lb[j] = (S.x_lo[j] ? log_hd(X[j] - S.xl[j]) : 0.0) + (S.x_hi[j] ? log_hd(S.xu[j] - X[j]) : 0.0);
    for (int r = team.rank; r < m; r += team.size) {
        const double ct = dc[r] * g_raw[r];
        t_bad[r] = finite_d(ct) ? 0.0 : 1.0;
        double st = S_lin[r], lbr = 0.0, vr = 0.0;
        // slack reset (Nocedal & Wright 2006, section 19.3): the row value itself, mu / nu inside its bound
        if (S.s_hi[r] && !S.s_lo[r]) st = nanmin(ct, su[r] - keep);
        if (S.s_lo[r] && !S.s_hi[r]) st = nanmax(ct, sl[r] + keep);
        if (pol) {
            // polishing instances: the slack of a strictly satisfied inequality row is the row value; the merit is the residual
            const bool inside = (!S.s_lo[r] || ct > sl[r]) && (!S.s_hi[r] || ct < su[r]);
            st = (!S.is_eq[r] && inside) ? ct : s[r];
            vr = S.is_eq[r] ? dabs(ct - sl[r]) : ((S.s_hi[r] ? clamp_min(ct - cu_s[r], 0.0) : 0.0) + (S.s_lo[r] ? clamp_min(cl_s[r] - ct, 0.0) : 0.0));
        } else {
            lbr = (S.s_lo[r] ? log_hd(st - sl[r]) : 0.0) + (S.s_hi[r] ? log_hd(su[r] - st) : 0.0);
            vr = dabs(ct - st);
        }
        t_lb[n + r] = lbr;
        t_viol[r] = vr;
        st_out[r] = st;
    }
    team.sync();
    if (team.rank < team.lanes()) {
        const bool ct_fin = arr_sum(team, t_bad, m) == 0.0;
        bool ok;
        if (pol) {
            ok = ct_fin && arr_nanmax(team, t_viol, m, 0.0) < T.R0[i];
        } else {
            const double mt = (T.dobj[i] * cost_raw - mu * arr_sum(team, t_lb, nk)) + nu * arr_sum(team, t_viol, m);
            const double m0 = T.merit0[i];
            ok = finite_d(mt) && mt <= (m0 + 10.0 * 2.2e-16 * dabs(m0)) + 1e-4 * AL * T.Dm[i];
        }
        if (team.rank == 0) {
            q.red[90] = ok ? 1.0 : 0.0;
            q.red[91] = ct_fin ? 1.0 : 0.0;
        }
    }
    team.sync();
    Trial t;
    t.ok = q.red[90] != 0.0;
    t.ct_finite = q.red[91] != 0.0;
    team.sync();
    return t;
}

// ---- phase 3: the full step, else the second-order correction ------------------------------------------------------------------
// Tests candidate 0; when it fails, solves the same KKT matrix with the constraint residual of the rejected point added to
// the right-hand side (Waechter & Biegler 2006, section 2.4) and emits the corrected trial point for one more evaluation.
template <class Team>
CPLB_HD void phase_ls_first(const Team& team, const Shape& S, const State& T, const Options& O, long long b, Scratch& q)
{
    const long long i = T.list_cur[b];
    Inst I{S, T, i};
    const int n = S.n, m = S.m, nk = S.nk;
    double* Xsoc = T.x_soc + b * n;
    const double* x = I.vn(T.x);
    if (team.rank == 0) {
        T.accepted0[i] = 0;
        T.soc_valid[i] = 0;
    }
    const double *s = I.vm(T.s), *ds = I.vm(T.ds), *dc = I.vm(T.dc);
    const double a0 = T.a_p[i];
    const double* X0 = T.x_ls + b * (long long)kCandidates * n;
    const double* g0 = T.g_ls + b * (long long)kCandidates * m;
    double *slin = q.term(3, nk), *st = q.term(4, nk);
    for (int r = team.rank; r < m; r += team.size) slin[r] = s[r] + a0 * ds[r];  // linearly stepped slacks of candidate 0
    team.sync();
    const Trial t0 = merit_test(team, I, q, X0, g0, T.cost_ls[b * kCandidates], slin, a0, st);
    const bool ok0 = (t0.ok || (T.tiny[i] && t0.ct_finite)) && O.max_backtracks >= 1;
    if (team.rank == 0) T.accepted0[i] = ok0 ? 1 : 0;
    if (ok0 || T.pol[i]) {
        for (int j = team.rank; j < n; j += team.size) Xsoc[j] = x[j];
        return;
    }
    // second-order correction with the stored factors
    const double *h = I.vm(T.h), *r_x = I.vn(T.r_x), *r_s = I.vm(T.r_s), *D = I.vm(T.D);
    const bool okK = T.okK[i] != 0;
    for (int a = team.rank; a < nk; a += team.size) {
        double v = 0.0;
        if (okK) {
            if (a < n) v = -r_x[a];
            else {
                const int r = a - n;
                const double h_soc = a0 * h[r] + (dc[r] * g0[r] - (s[r] + a0 * ds[r]));
                v = -h_soc - D[r] * r_s[r];
            }
        }
        q.sol[a] = v;
    }
    const double* LU = T.lu + i * (long long)nk * nk;
    for (int a = 0; a < nk; a++)
        for (int b = team.rank; b < nk; b += team.size) q.K[a * q.ld + b] = LU[a * nk + b];
    for (int a = team.rank; a < nk; a += team.size) {
        q.piv[a] = T.piv[i * nk + a];
        q.dinv[a] = T.lu_dinv[i * nk + a];
    }
    team.sync();
    lu_solve(team, q.K, q.ld, nk, q.piv, q.dinv, q.sol);
    compute_gaps(team, S, x, s, I.vm(T.sl), I.vm(T.su), q);
    team.sync();
    double *dxc = T.dx_soc + i * n, *dsc = T.ds_soc + i * m, *dlc = T.dlam_soc + i * m;
    const double tau = T.tau[i];
    auto ms = [&](double val, double dval, bool mask, double cur) {
        if (mask && dval < 0) cur = nanmin(cur, -tau * val / dval);
        return cur;
    };
    double *t_ac = q.term(5, nk), *t_bad = q.term(6, nk);
    for (int j = team.rank; j < n; j += team.size) {
        const double d = S.fixed[j] ? 0.0 : q.sol[j];
        dxc[j] = d;
        q.dx[j] = d;
        t_ac[j] = ms(q.gxu[j], -d, S.x_hi[j], ms(q.gxl[j], d, S.x_lo[j], INFINITY));
        t_bad[j] = finite_d(q.sol[j]) ? 0.0 : 1.0;
    }
    for (int r = team.rank; r < m; r += team.size) {
        const double dl = q.sol[n + r];
        const double d = S.is_eq[r] ? 0.0 : D[r] * (dl - r_s[r]);
        dlc[r] = dl;
        dsc[r] = d;
        t_ac[n + r] = ms(q.gsu[r], -d, S.s_hi[r], ms(q.gsl[r], d, S.s_lo[r], INFINITY));
        t_bad[n + r] = finite_d(dl) ? 0.0 : 1.0;
    }
    team.sync();
    if (team.rank < team.lanes()) {
        const double a_c = clamp_max(arr_nanmin(team, t_ac, nk, INFINITY), 1.0);
        const bool fin = arr_sum(team, t_bad, nk) == 0.0;
      if (team.rank == 0) {
        T.a_soc[i] = a_c;
        T.soc_valid[i] = fin ? 1 : 0;
        q.red[1] = a_c;
        q.red[2] = fin ? 1.0 : 0.0;
      }
    }
    team.sync();
    for (int j = team.rank; j < n; j += team.size) Xsoc[j] = q.red[2] != 0.0 ? x[j] + q.red[1] * q.dx[j] : x[j];
}

// ---- phase 4: accept a point, update the iterate and the multipliers ------------------------------------------------------------
template <class Team>
CPLB_HD void phase_ls_select(const Team& team, const Shape& S, const State& T, const Options& O, long long b, Scratch& q)
{
    const long long i = T.list_cur[b];
    Inst I{S, T, i};
    const int n = S.n, m = S.m, nk = S.nk;
    double *x = I.vn(T.x), *s = I.vm(T.s), *lam = I.vm(T.lam);
    const double *dx = I.vn(T.dx), *ds = I.vm(T.ds);
    const double a0 = T.a_p[i];
    const bool pol = T.pol[i] != 0;
    double *slin = q.term(3, nk), *st = q.term(4, nk);
    // order of a sequential backtracking search: full step, second-order correction, 1/2, 1/4, ...
    int choice = -1;  // candidate index; kCandidates = the corrected point
    double alpha = a0;
    if (T.accepted0[i]) {
        choice = 0;
        for (int r = team.rank; r < m; r += team.size) slin[r] = s[r] + a0 * ds[r];
        team.sync();
        merit_test(team, I, q, T.x_ls + b * (long long)kCandidates * n, T.g_ls + b * (long long)kCandidates * m, T.cost_ls[b * kCandidates], slin, a0, st);
    } else {
        if (T.soc_valid[i] && !pol) {
            const double a_c = T.a_soc[i];
            const double* dsc = T.ds_soc + i * m;
            for (int r = team.rank; r < m; r += team.size) slin[r] = s[r] + a_c * dsc[r];
            team.sync();
            const Trial t = merit_test(team, I, q, T.x_soc + b * n, T.g_soc + b * m, T.cost_soc[b], slin, a0, st);
            if (t.ok) choice = kCandidates;
        }
        const int kmax = O.max_backtracks < kCandidates ? O.max_backtracks : kCandidates;
        for (int k = 1; k < kmax && choice < 0; k++) {
            const double AL = a0 * ldexp(1.0, -k);
            for (int r = team.rank; r < m; r += team.size) slin[r] = s[r] + AL * ds[r];
            team.sync();
            const Trial t = merit_test(team, I, q, T.x_ls + (b * kCandidates + k) * (long long)n, T.g_ls + (b * kCandidates + k) * (long long)m,
                                       T.cost_ls[b * kCandidates + k], slin, AL, st);
            if (t.ok || (T.tiny[i] && t.ct_finite)) {
                choice = k;
                alpha = AL;
            }
        }
    }
    if (choice < 0) {  // search exhausted: take the last (tiny) step
        alpha = a0 * ldexp(1.0, -O.max_backtracks);
        for (int r = team.rank; r < m; r += team.size) st[r] = s[r] + alpha * ds[r];
        team.sync();
    }
    if (team.rank == 0) {
        // Levenberg-Marquardt damping of the next step: a search that had to backtrack asks for a shorter step next time
        double n_back = rint(log2(clamp_min(a0 / clamp_min(alpha, 1e-300), 1.0)));
        if (pol) n_back = 1.0;
        const double dl = T.delta_last[i];
        double dlm = n_back >= 2 ? dmax(dl * 8.0, 1e-6) : (n_back >= 1 ? dmax(dl * 2.0, 1e-6) : dl / 4.0);
        if (dlm < 1e-12) dlm = 0.0;
        T.delta_lm[i] = dmin(dlm, 1.0);
    }
    const double a_d = T.a_d[i];
    const double* dlam_used = (choice == kCandidates) ? T.dlam_soc + i * m : I.vm(T.dlam);
    const double* xnew = choice == kCandidates ? T.x_soc + b * n : (choice >= 0 ? T.x_ls + (b * kCandidates + choice) * (long long)n : nullptr);
    for (int j = team.rank; j < n; j += team.size) {
        const double v = xnew ? xnew[j] : x[j] + alpha * dx[j];
        x[j] = v;
        T.xc[b * n + j] = v;  // what the evaluator sees next, in slot order
        I.vn(T.vxl)[j] += a_d * I.vn(T.dvxl)[j];
        I.vn(T.vxu)[j] += a_d * I.vn(T.dvxu)[j];
    }
    for (int r = team.rank; r < m; r += team.size) {
        s[r] = st[r];
        lam[r] += alpha * dlam_used[r];
        I.vm(T.vsl)[r] += a_d * I.vm(T.dvsl)[r];
        I.vm(T.vsu)[r] += a_d * I.vm(T.dvsu)[r];
    }
}

// ---- results: honor_original_bounds, unscaled cost and multipliers -------------------------------------------------------------
template <class Team>
CPLB_HD void phase_finish(const Team& team, const Shape& S, const State& T, long long i, double* x_out, double* lam_out)
{
    Inst I{S, T, i};
    const double* x = I.vn(T.x);
    for (int j = team.rank; j < S.n; j += team.size) x_out[i * S.n + j] = nanmin(nanmax(x[j], S.xlo_orig[j]), S.xhi_orig[j]);
    if (lam_out)
        for (int r = team.rank; r < S.m; r += team.size) lam_out[i * S.m + r] = I.vm(T.lam)[r] * I.vm(T.dc)[r] / T.dobj[i];
    if (team.rank == 0) T.out_cost[i] = T.f[i];
}

// ==== host side shared by the GPU driver (cplb_solver.cu) and the CPU replay (tests/native/solver_host_check.cpp) ================

// Owner of the problem-level arrays of a Shape (host copies; the GPU driver uploads them).
struct ShapeHost {
    int n = 0, m = 0, nnz = 0, nf = 0;
    std::vector<int32_t> iRow, jCol, col_ptr, col_slot, free_idx;
    std::vector<double> xl, xu, xlo_orig, xhi_orig, cl, cu, cl_r, cu_r;
    std::vector<uint8_t> fixed, x_lo, x_hi, s_lo, s_hi, is_eq;

    // bounds as Problem::GetBoundsOnOptimizationVariables / GetBoundsOnConstraints report them (ifopt inf = 1e20);
    // fixed_variable_treatment = make_parameter, bound_relax_factor as in IPOPT
    void build(int n_, int m_, int nnz_, const int32_t* iRow_, const int32_t* jCol_, const double* xlb, const double* xub, const double* clb,
               const double* cub, double bound_relax)
    {
        n = n_;
        m = m_;
        nnz = nnz_;
        iRow.assign(iRow_, iRow_ + nnz);
        jCol.assign(jCol_, jCol_ + nnz);
        xlo_orig.assign(xlb, xlb + n);
        xhi_orig.assign(xub, xub + n);
        cl.assign(clb, clb + m);
        cu.assign(cub, cub + m);
        xl = xlo_orig;
        xu = xhi_orig;
        fixed.assign(n, 0);
        x_lo.assign(n, 0);
        x_hi.assign(n, 0);
        free_idx.clear();
        for (int j = 0; j < n; j++) {
            fixed[j] = xl[j] == xu[j];
            if (!fixed[j]) {
                xl[j] = xl[j] - bound_relax * dmax(dabs(xl[j]), 1.0);
                xu[j] = xu[j] + bound_relax * dmax(dabs(xu[j]), 1.0);
                free_idx.push_back(j);
            }
            x_lo[j] = !fixed[j] && xl[j] > -kInfBound;
            x_hi[j] = !fixed[j] && xu[j] < kInfBound;
        }
        nf = (int)free_idx.size();
        cl_r = cl;
        cu_r = cu;
        s_lo.assign(m, 0);
        s_hi.assign(m, 0);
        is_eq.assign(m, 0);
        for (int r = 0; r < m; r++) {
            is_eq[r] = cl[r] == cu[r];
            if (!is_eq[r]) {
                cl_r[r] = cl[r] - bound_relax * dmax(dabs(cl[r]), 1.0);
                cu_r[r] = cu[r] + bound_relax * dmax(dabs(cu[r]), 1.0);
            }
            s_lo[r] = !is_eq[r] && cl[r] > -kInfBound;
            s_hi[r] = !is_eq[r] && cu[r] < kInfBound;
        }
        col_ptr.assign(n + 1, 0);
        for (int e = 0; e < nnz; e++) col_ptr[jCol[e] + 1]++;
        for (int j = 0; j < n; j++) col_ptr[j + 1] += col_ptr[j];
        col_slot.assign(nnz, 0);
        std::vector<int32_t> fill(col_ptr.begin(), col_ptr.end() - 1);
        for (int e = 0; e < nnz; e++) col_slot[fill[jCol[e]]++] = e;  // ascending slot order within a column
    }
};

// Every per-instance array of a State with its element count per instance: lets both engines allocate generically.
struct StateField {
    void** ptr;
    size_t per_instance;  // elements per instance
    bool is_int;
};
inline std::vector<StateField> state_fields(State& T, const ShapeHost& S)
{
    const size_t n = S.n, m = S.m, nnz = S.nnz, nk = S.n + S.m, P = S.nf + 1, KC = kCandidates;
    std::vector<StateField> f;
    auto D = [&](double*& p, size_t c) { f.push_back({reinterpret_cast<void**>(&p), c, false}); };
    auto I = [&](int32_t*& p, size_t c) { f.push_back({reinterpret_cast<void**>(&p), c, true}); };
    D(T.x, n); D(T.s, m); D(T.lam, m); D(T.vxl, n); D(T.vxu, n); D(T.vsl, m); D(T.vsu, m);
    D(T.mu, 1); D(T.tau, 1); D(T.delta_last, 1); D(T.delta_lm, 1);
    I(T.status, 1); I(T.iters, 1); I(T.polish, 1); I(T.active, 1);
    D(T.f, 1); D(T.df, n); D(T.c, m); D(T.jv, nnz);
    I(T.list_cur, 1); I(T.list_next, 1); D(T.xc, n); D(T.ev_f, 1); D(T.ev_df, n); D(T.ev_c, m); D(T.ev_jv, nnz);
    D(T.dc, m); D(T.dobj, 1); D(T.sl, m); D(T.su, m); D(T.cu_s, m); D(T.cl_s, m);
    D(T.dx, n); D(T.ds, m); D(T.dlam, m); D(T.dvxl, n); D(T.dvxu, n); D(T.dvsl, m); D(T.dvsu, m); D(T.h, m); D(T.r_x, n); D(T.r_s, m); D(T.D, m);
    D(T.a_p, 1); D(T.a_d, 1); D(T.merit0, 1); D(T.Dm, 1); D(T.nu, 1); D(T.R0, 1); D(T.quad, 1);
    I(T.tiny, 1); I(T.pol, 1); I(T.okK, 1); I(T.accepted0, 1);
    D(T.lu, nk * nk); D(T.lu_dinv, nk); I(T.piv, nk);
    D(T.jd_slot, m * n); D(T.h0_slot, n * n);
    D(T.x_fd, P * n); D(T.grad_fd, P * n); D(T.jac_fd, P * nnz);
    D(T.x_ls, KC * n); D(T.g_ls, KC * m); D(T.cost_ls, KC);
    D(T.x_soc, n); D(T.g_soc, m); D(T.cost_soc, 1); D(T.dx_soc, n); D(T.ds_soc, m); D(T.dlam_soc, m); D(T.a_soc, 1);
    I(T.soc_valid, 1);
    D(T.out_cost, 1); D(T.out_viol, 1); D(T.out_dual, 1);
    return f;
}

struct SolveStats {
    int rounds = 0;                 // lock-step rounds
    long long evaluations = 0, instance_evaluations = 0;
    long long tail_instances = 0;   // instances that finished in the tail (on their own, after the lock-step rounds)
};

// One full iteration of a single instance between two phase_round_begin calls, with the four evaluations done by `eval(x, count,
// flags, g, jac, cost, grad)` on the instance's slot buffers: what the tail runs.  Returns when the iteration is complete (the
// new iterate evaluated into ev_*).
template <class Team, class Eval>
CPLB_HD void tail_iteration(const Team& team, const Shape& S, const State& T, const Options& O, long long b, Scratch& q, Eval&& eval)
{
    const int n = S.n, m = S.m, nnz = S.nnz, P = S.nf + 1;
    eval(T.x_fd + b * (long long)P * n, P, 2u | 8u, nullptr, T.jac_fd + b * (long long)P * nnz, nullptr, T.grad_fd + b * (long long)P * n);
    team.sync();
    phase_kkt(team, S, T, O, b, q);
    team.sync();
    eval(T.x_ls + b * (long long)kCandidates * n, kCandidates, 1u | 4u, T.g_ls + b * (long long)kCandidates * m, nullptr,
         T.cost_ls + b * (long long)kCandidates, nullptr);
    team.sync();
    phase_ls_first(team, S, T, O, b, q);
    team.sync();
    eval(T.x_soc + b * n, 1, 1u | 4u, T.g_soc + b * m, nullptr, T.cost_soc + b, nullptr);
    team.sync();
    phase_ls_select(team, S, T, O, b, q);
    team.sync();
    eval(T.xc + b * n, 1, 15u, T.ev_c + b * m, T.ev_jv + b * nnz, T.ev_f + b, T.ev_df + b * n);
    team.sync();
}

// The lock-step round, engine-independent.  Engine: init_x(), init_scale(), round_begin(first, last, slots) -> instances still
// running (the new working set; finished instances leave it: a round costs what its running instances cost), kkt(count),
// ls_first(count), ls_select(count), finish(), and the four batched evaluations eval_full / eval_fd / eval_ls / eval_soc (count).
template <class Engine>
SolveStats solve_loop(Engine& E, const Options& O, long long N, int nf)
{
    SolveStats st;
    E.init_x();
    E.eval_full(N);
    st.evaluations++;
    st.instance_evaluations += N;
    E.init_scale();
    long long working = N;  // slots of the previous round's working set
    for (int it = 0; it <= O.max_iter; it++) {
        const long long running = E.round_begin(it == 0, it == O.max_iter, working);  // also swaps the working-set lists
        if (running == 0) break;
        if (running <= E.tail_threshold()) {
            // The few instances left iterate on their own from here (one thread team each, evaluations inline): a straggler no
            // longer costs the whole batch a round trip per iteration, and its iterations cost no host round trip at all.
            const long long tail_rounds = E.tail(running, it);  // instance-rounds executed
            st.tail_instances += running;
            st.instance_evaluations += tail_rounds * (long long)(nf + 1 + kCandidates + 2);
            break;
        }
        st.rounds++;
        E.eval_fd(running);   // gradient + Jacobian at the nf + 1 difference points of every running instance
        E.kkt(running);
        E.eval_ls(running);   // constraint values + cost at the line-search candidates
        E.ls_first(running);
        E.eval_soc(running);  // ... and at the second-order-corrected points
        E.ls_select(running);
        E.eval_full(running);
        st.evaluations += 4;
        st.instance_evaluations += running * (long long)(nf + 1 + kCandidates + 2);
        working = running;
    }
    E.finish();
    return st;
}

}  // namespace solver
}  // namespace cplb
#endif
