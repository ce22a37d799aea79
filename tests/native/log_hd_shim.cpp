// ctypes shim over cplb::solver::log_hd (cplb_solver_core.hpp), the host build of the logarithm the solve round shares between
// the GPU and the CPU replay; tests/test_gpu_solver_replay.py compares it with mpmath.  TEST INFRASTRUCTURE.
#include <cstdint>

#include "cplb_solver_core.hpp"

extern "C" void cplb_log_hd_batch(const double* x, double* y, int64_t n)
{
    for (int64_t i = 0; i < n; i++) y[i] = cplb::solver::log_hd(x[i]);
}
