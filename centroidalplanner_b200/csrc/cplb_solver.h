// cplb_solver.h -- entry point of the native lock-step solve round (cplb_solver.cu), called by cplb_solve_device (cplb_abi.cu).
#ifndef CPLB_SOLVER_H
#define CPLB_SOLVER_H

#include <cuda_runtime.h>

#include "cplb_params.h"
#include "cplb_solver_core.hpp"

namespace cplb {
namespace solver {

// Shared memory one CTA of the solver kernels may use (sm_100: 227 KB a block).
constexpr size_t kMaxTeamBlockBytes = 227 * 1024;
// Bytes of the full team block (Scratch::carve with the KKT matrix) of an n-variable, m-row problem, as the solve launches it;
// *mats_in_global (may be NULL) says whether the dense Jacobian and the Hessian go to global memory to keep four teams per SM.
// A problem whose block exceeds kMaxTeamBlockBytes cannot be solved.
size_t team_block_bytes(int n, int m, int nnz, int* mats_in_global);

struct Workspace;  // device slabs owned by a problem handle, grown on demand
void workspace_free(Workspace* w);

// All pointers are device pointers on the current device; synchronises `st` (the host counts the running instances once per
// round).  Returns the first CUDA error.
// per_instance: per-instance parameter arrays (device, instance-major, indexed by instance), or nullptr.
cudaError_t solve_device(const CplbParams& P, int im_kernel, const CplbInstParams* per_instance, const ShapeHost& SH, const Options& O, long long N,
                         const double* x0, double* x_out,
                         int32_t* status, int32_t* iterations, double* cost, double* viol, double* dual, double* lam_out, SolveStats* stats,
                         Workspace** wsp, cudaStream_t st);

}  // namespace solver
}  // namespace cplb
#endif
