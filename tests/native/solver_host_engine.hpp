// HostEngine: the CPU replay of the native solve round (csrc/cplb_solver_core.hpp) -- the SAME per-instance code the GPU runs one
// CTA per instance, here one thread per instance, with the oracle behind the four batched evaluations.  TEST INFRASTRUCTURE,
// shared by solver_host_check.cpp (a CLI over the reference's TEST_F set-ups) and solver_replay.cpp (a C entry for Python).
#ifndef SOLVER_HOST_ENGINE_HPP
#define SOLVER_HOST_ENGINE_HPP

#include <cmath>
#include <cstdio>
#include <utility>
#include <vector>

#include "cpl_oracle.h"
#include "cplb_solver_core.hpp"

namespace cplb {
namespace solver {

struct HostEngine {
    cpl_oracle* o;
    ShapeHost SH;
    Shape S;
    State T{};
    Options O;
    long long N;
    std::vector<std::vector<double>> dstore;
    std::vector<std::vector<int32_t>> istore;
    std::vector<double> x0, x_out, lam_out, scratch;
    Scratch q;
    int threads = 8;

    void setup()
    {
        S.n = SH.n; S.m = SH.m; S.nnz = SH.nnz; S.nf = SH.nf; S.nk = SH.n + SH.m;
        S.iRow = SH.iRow.data(); S.jCol = SH.jCol.data(); S.col_ptr = SH.col_ptr.data(); S.col_slot = SH.col_slot.data();
        S.free_idx = SH.free_idx.data();
        S.xl = SH.xl.data(); S.xu = SH.xu.data(); S.xlo_orig = SH.xlo_orig.data(); S.xhi_orig = SH.xhi_orig.data();
        S.cl = SH.cl.data(); S.cu = SH.cu.data(); S.cl_r = SH.cl_r.data(); S.cu_r = SH.cu_r.data();
        S.fixed = SH.fixed.data(); S.x_lo = SH.x_lo.data(); S.x_hi = SH.x_hi.data();
        S.s_lo = SH.s_lo.data(); S.s_hi = SH.s_hi.data(); S.is_eq = SH.is_eq.data();
        for (auto& f : state_fields(T, SH)) {
            if (f.is_int) {
                istore.emplace_back(f.per_instance * N, 0);
                *f.ptr = istore.back().data();
            } else {
                dstore.emplace_back(f.per_instance * N, 0.0);
                *f.ptr = dstore.back().data();
            }
        }
        Scratch probe;
        scratch.assign(probe.carve(nullptr, S.n, S.m, S.nnz, true), 0.0);
        q.carve(scratch.data(), S.n, S.m, S.nnz, true);
        x_out.assign(N * S.n, 0.0);
        lam_out.assign(N * S.m, 0.0);
    }
    HostTeam team;
    void init_x() { for (long long i = 0; i < N; i++) phase_init_x(team, S, T, O, i, x0.data()); }
    void init_scale() { for (long long i = 0; i < N; i++) phase_init_scale(team, S, T, O, i); }
    long long round_begin(bool first, bool last, long long slots)
    {
        int running = 0;
        for (long long b = 0; b < slots; b++) phase_round_begin(team, S, T, O, b, q, first, last, &running);
        std::swap(T.list_cur, T.list_next);
        return running;
    }
    void kkt(long long cnt) { for (long long b = 0; b < cnt; b++) phase_kkt(team, S, T, O, b, q); }
    void ls_first(long long cnt) { for (long long b = 0; b < cnt; b++) phase_ls_first(team, S, T, O, b, q); }
    long long trace = -1;  // SOLVER_TRACE=<instance>: one line per iteration of that instance
    void ls_select(long long cnt)
    {
        for (long long b = 0; b < cnt; b++) {
            const long long i = T.list_cur[b];
            double alpha_sel = 0.0;
            if (i == trace) {
                double viol = 0.0;
                for (int r = 0; r < S.m; r++) {
                    const double c = T.c[i * S.m + r] * T.dc[i * S.m + r];
                    (void)c;
                }
                printf("  it %3d mu %.2e a_p %.3e a_d %.3e tiny %d pol %d okK %d acc0 %d delta %.2e |dx| ", T.iters[i], T.mu[i], T.a_p[i], T.a_d[i], T.tiny[i],
                       T.pol[i], T.okK[i], T.accepted0[i], T.delta_last[i]);
                double nd = 0.0;
                for (int j = 0; j < S.n; j++) nd = std::fmax(nd, std::fabs(T.dx[i * S.n + j]));
                printf("%.3e", nd);
                (void)viol;
                (void)alpha_sel;
            }
            const double f_before = T.f[i];
            std::vector<double> xb(T.x + i * S.n, T.x + (i + 1) * S.n);
            phase_ls_select(team, S, T, O, b, q);
            if (i == trace) {
                double step = 0.0;
                for (int j = 0; j < S.n; j++) step = std::fmax(step, std::fabs(T.x[i * S.n + j] - xb[j]));
                printf(" step %.3e f %.6e\n", step, f_before);
            }
        }
    }
    long long tail_limit = 0;
    long long tail_threshold() const { return tail_limit; }
    long long tail(long long running, int it0)
    {
        long long rounds = 0;
        auto eval = [&](const double* x, int count, unsigned flags, double* g, double* jac, double* cost, double* grad) {
            (void)flags;
            for (int a = 0; a < count; a++)
                cpl_oracle_eval(o, x + (long long)a * S.n, g ? g + (long long)a * S.m : nullptr, jac ? jac + (long long)a * S.nnz : nullptr,
                                cost ? cost + a : nullptr, grad ? grad + (long long)a * S.n : nullptr);
        };
        for (long long b = 0; b < running; b++) {
            for (int it = it0;;) {
                tail_iteration(team, S, T, O, b, q, eval);
                rounds++;
                it++;
                int dummy = 0;
                phase_round_begin(team, S, T, O, b, q, 0, it == O.max_iter, &dummy, true);
                if (!T.active[T.list_cur[b]]) break;
            }
        }
        return rounds;
    }
    void finish() { for (long long i = 0; i < N; i++) phase_finish(team, S, T, i, x_out.data(), lam_out.data()); }
    void eval_full(long long cnt) { cpl_oracle_eval_batch(o, cnt, T.xc, T.ev_c, T.ev_jv, T.ev_f, T.ev_df, threads); }
    void eval_fd(long long cnt) { cpl_oracle_eval_batch(o, cnt * (S.nf + 1), T.x_fd, nullptr, T.jac_fd, nullptr, T.grad_fd, threads); }
    void eval_ls(long long cnt) { cpl_oracle_eval_batch(o, cnt * kCandidates, T.x_ls, T.g_ls, nullptr, T.cost_ls, nullptr, threads); }
    void eval_soc(long long cnt) { cpl_oracle_eval_batch(o, cnt, T.x_soc, T.g_soc, nullptr, T.cost_soc, nullptr, threads); }
};

}  // namespace solver
}  // namespace cplb
#endif
