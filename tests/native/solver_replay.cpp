// C entry to the CPU replay of the native solve round (solver_host_engine.hpp), for tests/test_gpu_solver_replay.py: solves N
// starts of the problem an oracle handle describes with the per-instance code of csrc/cplb_solver_core.hpp, one thread per
// instance, the oracle behind the evaluations.  Link against the oracle/libcpl_oracle.so the ctypes wrapper loads, so that the
// wrapper's handle (cpl_oracle_py.Oracle._h) is valid here.  TEST INFRASTRUCTURE.
#include <cstdint>
#include <cstring>

#include "cpl_batched.h"
#include "solver_host_engine.hpp"

using namespace cplb::solver;

// stats (may be NULL): [rounds, evaluations, instance_evaluations, tail_instances].  tail_instances < 0 counts as 0 (lock-step
// rounds to the end): the host has no GPU to fill, and where the tail takes over does not change any instance's result.
// Returns 0, or -1 on bad arguments.
extern "C" int cplb_replay_solve(cpl_oracle* o, int64_t N, const double* x0, const cplb_solver_options* opt, double* x, double* lam,
                                 int32_t* status, int32_t* iterations, double* cost, double* constr_viol, double* dual_inf, int64_t* stats,
                                 int threads)
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
