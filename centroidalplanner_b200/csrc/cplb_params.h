// cplb_params.h -- the read-only parameter block handed BY VALUE to every kernel launch
// (__grid_constant__, lives in the constant bank: one broadcast read per warp, no HBM traffic,
// no staleness between a setter and the next launch on any stream).
//
// It holds what the reference keeps scattered over its IFOPT objects: CentroidalStatics::_m/_g/
// _wrench_manip (CentroidalStatics.cpp:12-15), FrictionCone::_F_thr (FrictionCone.cpp:14),
// EnvironmentClass::_mu (Environment.h:46), Ground::_ground_z, Superquadric::_C/_R/_P, and the
// refs/weights of MinimizeCentroidalVariables (MinimizeCentroidalVariables.cpp:11-26).
#ifndef CPLB_PARAMS_H
#define CPLB_PARAMS_H

#include <stdint.h>

#define CPLB_KMAX_CONTACTS 32

#define CPLB_WANT_G 1u
#define CPLB_WANT_J 2u
#define CPLB_WANT_COST 4u
#define CPLB_WANT_GRAD 8u
#define CPLB_JAC_COMPUTED_K 64u  // instance-major: like PACKED, also without the slots that are copies +-x[col] (JacMap<ENV, 2>)
#define CPLB_JAC_PACKED_K 32u   // instance-major: the Jacobian slice holds only the x-dependent slots (JacMap<ENV, true>)
#define CPLB_INPUTS_READY 16u  // x / per-instance arrays are not outputs of the preceding kernel: read them before griddepcontrol.wait

struct CplbParams {
    int32_t nc;
    int32_t env;
    int32_t n, m, nnz;
    int32_t reduction_order;            // Eigen fixed-size 3-term reductions: 0 = (v0+v1)+v2, 1 = v0+(v1+v2)
    int32_t perm[CPLB_KMAX_CONTACTS];  // sorted-name rank -> index in the caller's vector
    double mg[3];                       // _m * _g, one IEEE multiply per component, done on the host
    double mass;                        // _m (per-instance mode recomputes _m * _g on the device)
    double wrench[6];
    double mu;
    double ground_z;
    // Superquadric: raw parameters plus the constant-argument pow() results the reference
    // recomputes on every call (host glibc pow on the same arguments gives the same bits).
    double sqC[3], sqR[3], sqP[3];
    double sqPoverRP[3];  // P / pow(R, P)          Superquadric.cpp:54-56
    double sqRmP[3];      // pow(R, -P)             :98,109,...
    double sqRm2P[3];     // pow(R, -(P*2.0))       :82,86,107,...
    double sqR2P[3];      // pow(R,  P*2.0)         :95,96,149,150,203,204
    int32_t sqIntP[3];    // P as an integer when all three curvatures are integers in [2, 63], else 0
    int32_t sqBits;       // chain length: bit length of max(P) - 2
    int32_t sqWindow;     // |binary exponent of d| <= window keeps d^(2P) a normal number
    int32_t pad1;
    double F_thr[CPLB_KMAX_CONTACTS];
    double com_ref[3];
    double W_com;
    double p_ref[CPLB_KMAX_CONTACTS][3];
    double F_ref[CPLB_KMAX_CONTACTS][3];
    double W_p[CPLB_KMAX_CONTACTS];
    double W_F[CPLB_KMAX_CONTACTS];
};

// The optional per-instance parameter arrays, in the member order of cplb_instance_params (include/cpl_batched.h;
// cplb_abi.cu pins the correspondence).  The arrays before CPLB_IA_COM_REF are the ones the constraint rows read; the
// rest only the cost and its gradient.
enum CplbInstArray {
    CPLB_IA_MASS,
    CPLB_IA_WRENCH,
    CPLB_IA_MU,
    CPLB_IA_F_THR,     // contact index = position in the caller's name vector
    CPLB_IA_GROUND_Z,
    CPLB_IA_COM_REF,
    CPLB_IA_W_COM,
    CPLB_IA_P_REF,     // x,y,z of contact 0, then contact 1, ...
    CPLB_IA_F_REF,
    CPLB_IA_W_P,
    CPLB_IA_W_F,
    CPLB_NUM_INST_ARRAYS
};

// doubles per instance of array a
__host__ __device__ constexpr int cplb_inst_len(int a, int nc)
{
    switch (a) {
    case CPLB_IA_WRENCH: return 6;
    case CPLB_IA_COM_REF: return 3;
    case CPLB_IA_F_THR: case CPLB_IA_W_P: case CPLB_IA_W_F: return nc;
    case CPLB_IA_P_REF: case CPLB_IA_F_REF: return 3 * nc;
    default: return 1;
    }
}

// The per-instance arrays of one call (device memory; NULL = use the shared value of CplbParams), indexed by CplbInstArray.
// Same layout rule as x: element e of instance i is arr[a][i*len + e] (instance-major) or arr[a][e*ld + i] (component-major),
// len = cplb_inst_len(a, nc).
struct CplbInstParams {
    const double* arr[CPLB_NUM_INST_ARRAYS];
};

// Instance-major kernel, per-instance parameter mode: where each staged parameter array's slice of a warp tile sits in the
// shared-memory parameter buffer (doubles from the buffer start; -1 = not staged: absent, or not needed by the requested
// outputs), indexed by CplbInstArray.
struct CplbParamTile {
    int off[CPLB_NUM_INST_ARRAYS];
    int len[CPLB_NUM_INST_ARRAYS];  // doubles per instance of each array
    int total;                      // doubles per buffer (one warp tile)
};

// Pointers of one evaluation (device memory), see cplb_eval_args in include/cpl_batched.h.
struct CplbIo {
    const double* x;
    double* g;
    double* jac;
    double* cost;
    double* grad;
    long long ld;  // COMPONENT_MAJOR row pitch (elements)
    long long N;
};

#endif
