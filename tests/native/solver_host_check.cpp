// CPU replay of the native solve round (csrc/cplb_solver_core.hpp): the SAME per-instance code the GPU runs one CTA per
// instance, here one thread per instance, with the oracle behind the four batched evaluations.  TEST INFRASTRUCTURE.
// Replays the parameter sets of the reference's tests (tests/TestBasic.cpp:64-135 testGroundEnv, :138-222 testSuperquadricEnv,
// :225-292 testCoMPlanner) from a batch of perturbed starting points and checks the reference's EXPECT lines on every instance.
//   usage: solver_host_check [ground|superquadric|complanner|simple] [N]
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <utility>
#include <string>
#include <vector>

#include "solver_host_engine.hpp"

using namespace cplb::solver;

// lockstep_solver.default_start
static std::vector<double> default_start(const std::vector<double>& lb, const std::vector<double>& ub, int n)
{
    const int nc = (n - 3) / 9;
    std::vector<double> lo(n), hi(n), mid(n), half(n), x(n);
    for (int j = 0; j < n; j++) {
        lo[j] = std::fmax(lb[j], -1.0);
        hi[j] = std::fmin(ub[j], 1.0);
        mid[j] = 0.5 * (lo[j] + hi[j]);
        half[j] = 0.5 * (hi[j] - lo[j]);
        x[j] = mid[j];
    }
    const double corners[4][2] = {{1, 1}, {-1, 1}, {-1, -1}, {1, -1}};
    auto clip = [](double v, double a, double b) { return v < a ? a : (v > b ? b : v); };
    for (int k = 0; k < nc; k++) {
        const int b = 3 + 9 * k;
        const double shrink = 0.8 / (1 + k / 4);
        const double F[3] = {1.0 + 0.5 * k, -1.0 + 0.25 * k, 981.0 / nc};
        for (int c = 0; c < 3; c++) x[b + c] = clip(F[c], lb[b + c], ub[b + c]);
        x[b + 3] = mid[b + 3] + corners[k % 4][0] * shrink * half[b + 3];
        x[b + 4] = mid[b + 4] + corners[k % 4][1] * shrink * half[b + 4];
        const double nn[3] = {0, 0, 1};
        for (int c = 0; c < 3; c++) x[b + 6 + c] = clip(nn[c], lb[b + 6 + c], ub[b + 6 + c]);
    }
    return x;
}

int main(int argc, char** argv)
{
    const std::string which = argc > 1 ? argv[1] : "ground";
    const long long N = argc > 2 ? atoll(argv[2]) : 16;
    // (ground8: config 4's shape -- 8 contacts, names given r_* first so that vector order != sorted order; a 129 x 129 KKT matrix)
    const char* names4[4] = {"contact1", "contact2", "contact3", "contact4"};
    const char* names8[8] = {"r_hand_b", "r_hand_a", "l_hand_b", "l_hand_a", "r_foot_b", "r_foot_a", "l_foot_b", "l_foot_a"};
    const int nc = which == "simple" ? 1 : (which == "ground8" ? 8 : 4);
    const char** names = nc == 8 ? names8 : names4;
    const int env = which == "superquadric" ? CPL_ORACLE_ENV_SUPERQUADRIC : (which == "complanner" ? CPL_ORACLE_ENV_NONE : CPL_ORACLE_ENV_GROUND);
    cpl_oracle* o = cpl_oracle_new(nc, names, env, 100.0);
    const double wrench[6] = {100, 0, 0, 0, 0, 100};
    if (which == "ground" || which == "ground8") {
        cpl_oracle_set_ground_z(o, 0.1);
        cpl_oracle_set_mu(o, 0.5);
        cpl_oracle_set_com_weight(o, 2.0);
        for (int k = 0; k < nc; k++) {
            cpl_oracle_set_force_weight(o, k, 0.0);
            const double lb[3] = {-0.3, -0.3, 0.0}, ub[3] = {0.3, 0.3, 1.0};
            cpl_oracle_set_var_bounds(o, 2, k, lb, ub);
        }
        cpl_oracle_set_wrench(o, wrench);
    } else if (which == "superquadric") {
        cpl_oracle_set_mu(o, 0.5);
        const double C[3] = {0, 0, 1}, R[3] = {0.3, 0.3, 10}, P[3] = {10, 10, 10};
        cpl_oracle_set_superquadric(o, C, R, P);
        for (int k = 0; k < 4; k++) {
            cpl_oracle_set_force_weight(o, k, 0.0);
            const double lb[3] = {-0.5, -0.5, 0.5}, ub[3] = {0.5, 0.5, 1.5};
            cpl_oracle_set_var_bounds(o, 2, k, lb, ub);
        }
        cpl_oracle_set_wrench(o, wrench);
    } else if (which == "complanner") {
        cpl_oracle_set_mu(o, 0.5);
        const double pts[4][3] = {{1, 1, 0}, {-1, 1, 0}, {-1, -1, 0}, {1, -1, 0}};
        for (int k = 0; k < 4; k++) {
            cpl_oracle_set_pos_weight(o, k, 0.0);
            cpl_oracle_set_force_weight(o, k, 0.0);
            const double nl[3] = {0, 0, 1};
            cpl_oracle_set_var_bounds(o, 3, k, nl, nl);
            cpl_oracle_set_var_bounds(o, 2, k, pts[k], pts[k]);
            cpl_oracle_set_force_threshold(o, k, 20.0);
        }
        const double z[3] = {0, 0, 0};
        cpl_oracle_set_var_bounds(o, 1, 3, z, z);
        cpl_oracle_set_force_threshold(o, 3, 0.0);
    } else {
        cpl_oracle_set_ground_z(o, 0.1);
    }
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
    E.O = Options{1e-3, 0.1, 1e-2, 1e-2, 100.0, 1e-4, 1e-9, 1e-8, 500, 30, 0};
    if (getenv("SOLVER_TOL")) E.O.tol = atof(getenv("SOLVER_TOL"));
    if (getenv("SOLVER_TAIL")) E.tail_limit = atoll(getenv("SOLVER_TAIL"));
    if (getenv("SOLVER_TRACE")) E.trace = atoll(getenv("SOLVER_TRACE"));
    if (getenv("SOLVER_FORCE_WEIGHT"))
        for (int k = 0; k < nc; k++) cpl_oracle_set_force_weight(o, k, atof(getenv("SOLVER_FORCE_WEIGHT")));
    E.SH.build(n, m, nnz, iRow.data(), jCol.data(), xl.data(), xu.data(), cl.data(), cu.data(), E.O.bound_relax);
    E.setup();
    const std::vector<double> xs = default_start(xl, xu, n);
    std::mt19937_64 rng(7);
    std::normal_distribution<double> nd(0.0, 0.05);
    E.x0.resize(N * n);
    for (long long i = 0; i < N; i++)
        for (int j = 0; j < n; j++) E.x0[i * n + j] = xs[j] + (i == 0 ? 0.0 : nd(rng));
    const SolveStats st = solve_loop(E, E.O, N, E.SH.nf);

    int failures = 0, max_it = 0;
    double worst_viol = 0.0;
    std::vector<double> g(m);
    for (long long i = 0; i < N; i++) {
        const double* x = E.x_out.data() + i * n;
        if (E.T.status[i] != kSuccess) {
            failures++;
            printf("instance %lld: status %d after %d iterations (viol %.2e dual %.2e)\n", i, E.T.status[i], E.T.iters[i], E.T.out_viol[i], E.T.out_dual[i]);
            continue;
        }
        max_it = E.T.iters[i] > max_it ? E.T.iters[i] : max_it;
        cpl_oracle_eval(o, x, g.data(), nullptr, nullptr, nullptr);
        // TestBasic: sum F = w[0:3] - m g, sum tau = w[3:6] (rows 0..5 of CentroidalStatics are those residuals)
        for (int r = 0; r < 6; r++) {
            const double tol = r < 3 ? 1e-6 : 1e-4;
            if (std::fabs(g[r]) > tol) {
                failures++;
                printf("instance %lld: statics row %d = %.3e\n", i, r, g[r]);
            }
            worst_viol = std::fmax(worst_viol, std::fabs(g[r]));
        }
        const int per = env == CPL_ORACLE_ENV_NONE ? 2 : 6;
        for (int j = 0; j < nc; j++) {
            const int row = 6 + per * j + (per == 6 ? 4 : 0);
            if (g[row] > 1e-6 || g[row + 1] > 1e-6) {  // friction rows <= 0 up to the bound relaxation
                failures++;
                printf("instance %lld: friction rows of contact %d: %.3e %.3e\n", i, j, g[row], g[row + 1]);
            }
            if (per == 6)
                for (int r = 0; r < 4; r++)
                    if (std::fabs(g[6 + per * j + r]) > (env == CPL_ORACLE_ENV_SUPERQUADRIC ? 1e-4 : 1e-6)) {
                        failures++;
                        printf("instance %lld: environment row %d of contact %d = %.3e\n", i, r, j, g[6 + per * j + r]);
                    }
        }
    }
    if (getenv("SOLVER_HIST")) {
        std::vector<int> hist(20, 0);
        for (long long i = 0; i < N; i++) hist[std::min(19, E.T.iters[i] / 10)]++;
        printf("iterations histogram (bins of 10):");
        for (int h : hist) printf(" %d", h);
        printf("\nslowest:");
        std::vector<long long> idx(N);
        for (long long i = 0; i < N; i++) idx[i] = i;
        std::sort(idx.begin(), idx.end(), [&](long long a, long long b) { return E.T.iters[a] > E.T.iters[b]; });
        for (int k = 0; k < 8 && k < N; k++) printf(" %lld(%d)", idx[k], E.T.iters[idx[k]]);
        printf("\n");
    }
    printf("%s: N %lld, %d rounds, %lld batched evaluations (%lld instance evaluations), max iterations %d, worst statics residual %.2e -> %d failures\n",
           which.c_str(), N, st.rounds, st.evaluations, st.instance_evaluations, max_it, worst_viol, failures);
    cpl_oracle_free(o);
    return failures ? 1 : 0;
}
