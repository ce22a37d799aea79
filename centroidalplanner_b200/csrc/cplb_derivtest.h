// cplb_derivtest.h -- launcher of the batched first-order derivative test (cplb_derivtest.cu), called by
// cplb_derivative_test_device (cplb_abi.cu).
#ifndef CPLB_DERIVTEST_H
#define CPLB_DERIVTEST_H

#include <cuda_runtime.h>

#include <cstdint>

#include "cplb_params.h"

namespace cplb {

struct DerivTestOut {  // device arrays, instance-major; any may be nullptr
    int32_t* num_wrong;
    int32_t* num_wrong_outside;
    double* max_rel_error;
    int32_t* worst_row;
    int32_t* worst_col;
    double* jac_fd;   // [N nnz]
    double* grad_fd;  // [N n]
};

// Columns of x perturbed together in one chunk: as many as fit the kernel's shared-memory budget next to the point's own
// outputs, at most n.  At least 1 for every shape up to CPLB_KMAX_CONTACTS contacts in every environment.
int derivtest_chunk(int n, int m, int nnz);
// Dynamic shared memory of one CTA for chunks of k columns.
size_t derivtest_smem_bytes(int n, int m, int nnz, int k);

// slot_of[r*n + c]: the structural slot of Jacobian entry (r, c), -1 outside the structure (device, per problem).
// per_instance: per-instance parameter arrays (device, instance-major), or nullptr.  Asynchronous on st.
cudaError_t launch_derivative_test(const CplbParams& P, const CplbInstParams* per_instance, const double* x, long long N,
                                   const int32_t* slot_of, double perturbation, double tol, const DerivTestOut& out, cudaStream_t st);

}  // namespace cplb
#endif
