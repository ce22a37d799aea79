// C entry to the CPU replay of the native solve round (solver_host_engine.hpp), for tests/test_gpu_solver_replay.py: solves N
// starts of the problem an oracle handle describes with the per-instance code of csrc/cplb_solver_core.hpp, one thread per
// instance, the oracle behind the evaluations.  Link against the oracle/libcpl_oracle.so the ctypes wrapper loads, so that the
// wrapper's handle (cpl_oracle_py.Oracle._h) is valid here.  A second entry takes one oracle per instance (per-instance
// parameter sweeps).  TEST INFRASTRUCTURE.
#include <cstdint>
#include <cstring>

#include "cpl_batched.h"
#include "solver_host_engine.hpp"

using namespace cplb::solver;

// stats (may be NULL): [rounds, evaluations, instance_evaluations, tail_instances].  tail_instances < 0 counts as 0 (lock-step
// rounds to the end): the host has no GPU to fill, and where the tail takes over does not change any instance's result.
// per (may be NULL): N oracle handles, per[i] the problem of instance i (same shape and bounds as o); o = per[0] then.
// Returns 0, or -1 on bad arguments.
static int replay(cpl_oracle* o, cpl_oracle* const* per, int64_t N, const double* x0, const cplb_solver_options* opt, double* x, double* lam,
                  int32_t* status, int32_t* iterations, double* cost, double* constr_viol, double* dual_inf, int64_t* stats, int threads)
{
    if (!o || N <= 0 || !x0 || !opt || !x || !status || !iterations || !cost || !constr_viol || !dual_inf) return -1;
    int n, m, nnz;
    cpl_oracle_dims(o, &n, &m, &nnz);
    std::vector<int> iRow(nnz), jCol(nnz);
    cpl_oracle_structure(o, iRow.data(), jCol.data());
    std::vector<double> xl(n), xu(n), cl(m), cu(m);
    cpl_oracle_var_bounds(o, xl.data(), xu.data());
    cpl_oracle_con_bounds(o, cl.data(), cu.data());

    HostEngine E;
    E.o = o;
    if (per) {
        for (int64_t i = 0; i < N; i++) {
            int ni, mi, nnzi;
            if (!per[i]) return -1;
            cpl_oracle_dims(per[i], &ni, &mi, &nnzi);
            if (ni != n || mi != m || nnzi != nnz) return -1;
        }
        E.per.assign(per, per + N);
    }
    E.N = N;
    E.threads = threads > 0 ? threads : 1;
    E.O = Options{opt->tol, opt->mu_init, opt->bound_push, opt->bound_frac, opt->nlp_scaling_max_gradient, opt->constr_viol_tol,
                  opt->polish_viol_tol, opt->bound_relax_factor, opt->max_iter, opt->max_backtracks, opt->tail_instances};
    E.tail_limit = opt->tail_instances > 0 ? opt->tail_instances : 0;
    E.SH.build(n, m, nnz, iRow.data(), jCol.data(), xl.data(), xu.data(), cl.data(), cu.data(), E.O.bound_relax);
    E.setup();
    E.x0.assign(x0, x0 + N * n);
    const SolveStats st = solve_loop(E, E.O, N, E.SH.nf);

    std::memcpy(x, E.x_out.data(), sizeof(double) * N * n);
    if (lam) std::memcpy(lam, E.lam_out.data(), sizeof(double) * N * m);
    std::memcpy(status, E.T.status, sizeof(int32_t) * N);
    std::memcpy(iterations, E.T.iters, sizeof(int32_t) * N);
    std::memcpy(cost, E.T.out_cost, sizeof(double) * N);
    std::memcpy(constr_viol, E.T.out_viol, sizeof(double) * N);
    std::memcpy(dual_inf, E.T.out_dual, sizeof(double) * N);
    if (stats) {
        stats[0] = st.rounds;
        stats[1] = st.evaluations;
        stats[2] = st.instance_evaluations;
        stats[3] = st.tail_instances;
    }
    return 0;
}

extern "C" int cplb_replay_solve(cpl_oracle* o, int64_t N, const double* x0, const cplb_solver_options* opt, double* x, double* lam,
                                 int32_t* status, int32_t* iterations, double* cost, double* constr_viol, double* dual_inf, int64_t* stats,
                                 int threads)
{
    return replay(o, nullptr, N, x0, opt, x, lam, status, iterations, cost, constr_viol, dual_inf, stats, threads);
}

// The replay of a sweep: instance i solves the problem of oracle o[i] (its own cplb_instance_params, set on that oracle).  Every
// evaluated point goes to the oracle of its instance; the variable / constraint bounds are o[0]'s (the bounds stay the problem's).
extern "C" int cplb_replay_solve_per_instance(cpl_oracle* const* o, int64_t N, const double* x0, const cplb_solver_options* opt, double* x,
                                              double* lam, int32_t* status, int32_t* iterations, double* cost, double* constr_viol,
                                              double* dual_inf, int64_t* stats, int threads)
{
    if (!o || N <= 0) return -1;
    return replay(o[0], o, N, x0, opt, x, lam, status, iterations, cost, constr_viol, dual_inf, stats, threads);
}
