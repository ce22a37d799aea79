// Stand-alone check (built by tests/test_gpu_solver_replay.py with nvcc -fmad=false, host side -ffp-contract=off): the
// elementary functions of the solve round that must give the same bits on the GPU and in the CPU replay --
// cplb::solver::log_hd (cplb_solver_core.hpp), mu^1.5 as mu * sqrt(mu) and mu^0.25 as sqrt(sqrt(mu)) -- evaluated by the
// device and by the host build of the same source on the same inputs.  NaN results are matched by position only.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "cplb_solver_core.hpp"

using cplb::solver::log_hd;

CPLB_HD double f_of(int which, double x)
{
    if (which == 0) return log_hd(x);
    if (which == 1) return x * sqrt(x);
    return sqrt(sqrt(x));
}

__global__ void eval(const double* x, double* y, int n, int which)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = f_of(which, x[i]);
}

static double from_bits(uint64_t u)
{
    double v;
    std::memcpy(&v, &u, 8);
    return v;
}

int main()
{
    const int n = 1 << 21;
    std::vector<double> x;
    x.reserve(n);
    const double specials[] = {0.0, -0.0, 1.0, -1.0, INFINITY, -INFINITY, NAN, -NAN, 4.9e-324, 2.2250738585072014e-308,
                               2.225073858507201e-308, 1.7976931348623157e308, 0.5, 2.0, 1e-300, 1e300, M_SQRT2, M_SQRT1_2};
    for (double s : specials) x.push_back(s);
    for (int e = -1074; e <= 1023; e++) {  // every power of two and its neighbours
        const double p = std::ldexp(1.0, e);
        x.push_back(p);
        x.push_back(std::nextafter(p, 0.0));
        x.push_back(std::nextafter(p, INFINITY));
    }
    for (int k = 1; k <= 4096; k++) {  // 1 +- k eps
        x.push_back(1.0 + k * 2.220446049250313e-16);
        x.push_back(1.0 - k * 1.1102230246251565e-16);
    }
    std::mt19937_64 rng(20261020);
    while ((int)x.size() < n) {
        const uint64_t u = rng();
        switch (x.size() % 4) {
            case 0: x.push_back(from_bits(u)); break;                                          // any bit pattern
            case 1: x.push_back(from_bits(u & 0x000fffffffffffffull)); break;                 // subnormals
            case 2: x.push_back(std::ldexp(1.0 + (double)(u >> 11) / 9007199254740992.0, (int)(u % 2000) - 1000)); break;
            default: x.push_back(std::exp(-40.0 + 50.0 * (double)(u >> 11) / 9007199254740992.0)); break;  // gaps, mu, slack magnitudes
        }
    }
    double *dx, *dy;
    if (cudaMalloc(&dx, n * 8) != cudaSuccess || cudaMalloc(&dy, n * 8) != cudaSuccess) {
        printf("CUDA error\n");
        return 2;
    }
    cudaMemcpy(dx, x.data(), n * 8, cudaMemcpyHostToDevice);
    const char* names[3] = {"log_hd", "x*sqrt(x)", "sqrt(sqrt(x))"};
    std::vector<double> y(n);
    long long total_bad = 0;
    for (int which = 0; which < 3; which++) {
        eval<<<(n + 255) / 256, 256>>>(dx, dy, n, which);
        if (cudaMemcpy(y.data(), dy, n * 8, cudaMemcpyDeviceToHost) != cudaSuccess) {
            printf("CUDA error\n");
            return 2;
        }
        long long bad = 0;
        for (int i = 0; i < n; i++) {
            const double h = f_of(which, x[i]), d = y[i];
            uint64_t hb, db;
            std::memcpy(&hb, &h, 8);
            std::memcpy(&db, &d, 8);
            const bool same = (h != h && d != d) || hb == db;
            if (!same && bad++ == 0) printf("%s: first mismatch x=%a device=%a host=%a\n", names[which], x[i], d, h);
        }
        printf("%s: checked %d inputs, mismatches %lld\n", names[which], n, bad);
        total_bad += bad;
    }
    cudaFree(dx);
    cudaFree(dy);
    return total_bad ? 1 : 0;
}
