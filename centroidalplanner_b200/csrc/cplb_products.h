// cplb_products.h -- launcher of the fused Jacobian products (cplb_products.cu), called by cplb_jacobian_products_device
// (cplb_abi.cu).
#ifndef CPLB_PRODUCTS_H
#define CPLB_PRODUCTS_H

#include <cuda_runtime.h>

#include "cplb_params.h"

namespace cplb {

struct ProductArgs {  // device arrays, instance-major; see cplb_jacobian_products_args in include/cpl_batched.h
    const double* x;           // [N n]
    const double* lambda;      // [N m] or nullptr
    const double* obj_factor;  // [N]   or nullptr
    double* x_bar;             // [N n] or nullptr
    const double* v;           // [N n] (needed when g_dot or f_dot is set)
    double* g_dot;             // [N m] or nullptr
    double* f_dot;             // [N]   or nullptr
    long long N;
};

// per_instance: per-instance parameter arrays (device, instance-major), or nullptr.  One launch, asynchronous on st.
cudaError_t launch_jacobian_products(const CplbParams& P, const CplbInstParams* per_instance, const ProductArgs& A, cudaStream_t st);

}  // namespace cplb
#endif
