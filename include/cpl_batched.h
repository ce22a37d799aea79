/*
 * cpl_batched.h -- C ABI of the B200 batched evaluator for CentroidalPlanner's IFOPT problem.
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types, no exceptions.
 * Every entry point names the reference interface it replaces (paths relative to the
 * ADVRHumanoids/CentroidalPlanner tree).  One `cplb_problem` describes ONE problem *shape*
 * (contact names, environment, parameters) -- what the reference holds in one
 * `cpl::solver::CplProblem` -- and evaluates it for N independent instances (N different x)
 * per call on one GPU.
 *
 * Layout contract (identical to the reference + ifopt, see DESIGN.md):
 *   columns  CoM -> 0..2; contact k (index in the CALLER'S name vector): F_k -> 3+9k+{0,1,2},
 *            p_k -> 3+9k+{3,4,5}, n_k -> 3+9k+{6,7,8}                 (src/CplProblem.cpp:17-34)
 *   rows     0..5 CentroidalStatics; contact of sorted-name rank j (std::map order):
 *            6+6j EnvironmentConstraint, 6+6j+{1,2,3} EnvironmentNormal, 6+6j+{4,5}
 *            FrictionCone; without environment 6+2j+{0,1} FrictionCone    (src/CplProblem.cpp:37-75)
 *   Jacobian values in the order ifopt's IpoptAdapter::eval_jac_g emits (iRow, jCol): row-major,
 *            column ascending, every coeffRef'd slot present even when its value is 0.0.
 *
 * Error convention: every function returns a cplb_status; on failure a message is kept in a
 * thread-local buffer (cplb_last_error).  The status says which C++ exception the reference
 * would have thrown at the same place.  Non-finite outputs are data, not errors (the reference
 * divides by the tangential force norm without a guard, src/Constraints/FrictionCone.cpp:85-87).
 *
 * Threading: setters must not run concurrently with evaluation on the same problem.  Evaluation
 * calls take x as an argument (not problem state, unlike Variable3D::SetVariables,
 * src/Variable3D.cpp:18-25) so several host threads may evaluate disjoint instance ranges of the
 * same problem on different streams at once.
 */
#ifndef CPL_BATCHED_H
#define CPL_BATCHED_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPLB_ABI_VERSION 3
#define CPLB_MAX_CONTACTS 32
#define CPLB_MAX_SHARDS 64

typedef enum cplb_status {
    CPLB_OK = 0,
    CPLB_INVALID_ARGUMENT = 1, /* reference throws std::invalid_argument */
    CPLB_OUT_OF_RANGE = 2,     /* reference throws std::out_of_range (std::map::at on an unknown contact) */
    CPLB_RUNTIME_ERROR = 3,    /* reference throws std::runtime_error */
    CPLB_CUDA_ERROR = 4,       /* CUDA runtime failure (no device, launch failure, out of memory) */
    CPLB_NULL_POINTER = 5      /* a required pointer argument was NULL */
} cplb_status;

/* cpl::env::EnvironmentClass::Ptr passed to CplProblem (src/CplProblem.cpp:8,44,63):
 * nullptr / Ground / Superquadric */
typedef enum cplb_env_kind {
    CPLB_ENV_NONE = 0,
    CPLB_ENV_GROUND = 1,
    CPLB_ENV_SUPERQUADRIC = 2
} cplb_env_kind;

/* How the N instances are laid out in the batched buffers.
 *  INSTANCE_MAJOR : buf[i*len + e]   -- instance i owns a contiguous slice; this is what one
 *                   IPOPT thread hands to / receives from eval_g / eval_jac_g (x[n], g[m], values[nnz]).
 *  COMPONENT_MAJOR: buf[e*ld + i]    -- struct-of-arrays, ld >= N is the row pitch in elements. */
typedef enum cplb_layout {
    CPLB_INSTANCE_MAJOR = 0,
    CPLB_COMPONENT_MAJOR = 1
} cplb_layout;

/* Which variable block a bound refers to (Variable3D objects of src/CplProblem.cpp:17-33). */
typedef enum cplb_block {
    CPLB_BLOCK_COM = 0,
    CPLB_BLOCK_FORCE = 1,
    CPLB_BLOCK_POSITION = 2,
    CPLB_BLOCK_NORMAL = 3
} cplb_block;

typedef struct cplb_problem cplb_problem; /* opaque */

/* ---- life cycle --------------------------------------------------------------------------- */

/* Replaces cpl::solver::CplProblem::CplProblem(contact_names, robot_mass, env)
 * (src/CplProblem.cpp:6-82) together with the robot_mass check of
 * cpl::CentroidalPlanner::CentroidalPlanner (src/CentroidalPlanner.cpp:12-15: mass <= 0 ->
 * CPLB_INVALID_ARGUMENT).  Parameters start at the reference's defaults (mass-g (0,0,-9.81),
 * zero wrench, mu 1, F_thr 0, ground z 0, superquadric C=(0,0,10) R=P=(10,10,10), CoM ref (0,0,1),
 * all weights 1, refs 0, variable bounds +-1000).  Duplicate or empty name lists are rejected
 * (CPLB_INVALID_ARGUMENT): the reference's std::map would silently merge them.
 * device: CUDA ordinal (validated now: CPLB_CUDA_ERROR when no CUDA device is usable), or -1 to bind to
 * the calling thread's current device at the first evaluation.  Creation, layout queries and the
 * parameter setters are host-only; evaluation on a machine without a GPU fails with
 * CPLB_CUDA_ERROR -- there is no CPU fallback. */
cplb_status cplb_create(int32_t num_contacts, const char *const *contact_names, cplb_env_kind env,
                        double robot_mass, int32_t device, cplb_problem **out);
void cplb_destroy(cplb_problem *p);

/* The same problem on SEVERAL GPUs of one box, driven from this one process: `devices` lists num_devices CUDA ordinals
 * (validated now; an ordinal listed twice simply gets two pipelines -- how a one-GPU box exercises the sharded path).  Instances shard by index with no collective anywhere (no cross-instance term exists in
 * the files under src/Constraints or src/MinimizeCentroidalVariables.cpp): a batch of N instances is cut into contiguous ranges, shard s of
 * G owning [s*per, (s+1)*per) with per = ceil(N / G) rounded up to a multiple of 32 (cplb_get_shard reports the exact range),
 * parameters are replicated (they travel as kernel arguments), and
 *   cplb_eval_host / cplb_eval_host_begin / _wait   take ONE set of host buffers for the whole batch and run every device's
 *       H2D / kernel / D2H pipeline at once (pinned buffers: all asynchronous, enqueued round robin over the devices by the
 *       calling thread; pageable buffers: one packing thread per device);
 *   cplb_eval_device_shard   evaluates device-resident buffers of one shard on that shard's device and stream
 *       (cplb_eval_device refuses a problem with more than one shard: a device pointer belongs to one device).
 * Everything else (setters, layout, bounds) is shared by the shards.  This is what a C++ caller in the position of
 * cpl::solver::CplProblem (src/CplProblem.cpp:6-82) uses to feed the solver threads of one process from all GPUs of the box;
 * a single-device problem (cplb_create) behaves as a problem with one shard. */
cplb_status cplb_create_sharded(int32_t num_contacts, const char *const *contact_names, cplb_env_kind env,
                                double robot_mass, int32_t num_devices, const int32_t *devices, cplb_problem **out);
cplb_status cplb_get_num_shards(const cplb_problem *p, int32_t *num_shards);
/* Device ordinal of a shard and its instance range [begin, end) in a batch of num_instances; each out-pointer may be NULL. */
cplb_status cplb_get_shard(const cplb_problem *p, int32_t shard, int64_t num_instances, int32_t *device, int64_t *begin,
                           int64_t *end);

/* Thread-local message of the last failing call on this thread ("" if none). */
const char *cplb_last_error(void);
int32_t cplb_abi_version(void);

/* ---- layout: what ifopt::Problem / IpoptAdapter report ------------------------------------- */

/* n = GetNumberOfOptimizationVariables, m = GetNumberOfConstraints,
 * nnz = GetJacobianOfConstraints().nonZeros() [ifopt; call sites src/CplProblem.cpp:19-80] */
cplb_status cplb_get_dims(const cplb_problem *p, int32_t *n, int32_t *m, int32_t *nnz);
/* IpoptAdapter::eval_jac_g(values == NULL): C-style (iRow, jCol), nnz entries each. */
cplb_status cplb_get_jacobian_structure(const cplb_problem *p, int32_t *iRow, int32_t *jCol);
/* sorted_to_vector[j] = index in the caller's name vector of the contact with sorted rank j
 * (iteration order of _contact_vars_map, src/CplProblem.cpp:42). */
cplb_status cplb_get_sorted_order(const cplb_problem *p, int32_t *sorted_to_vector);
/* First column of a block / first row of a contact's constraint rows (-1 rows for statics = 0). */
cplb_status cplb_get_block_column(const cplb_problem *p, cplb_block block, const char *contact_name, int32_t *col);
cplb_status cplb_get_contact_row(const cplb_problem *p, const char *contact_name, int32_t *row);
/* Problem::GetBoundsOnOptimizationVariables / GetBoundsOnConstraints
 * (Variable3D::GetBounds src/Variable3D.cpp:54-65; CentroidalStatics.cpp:64-73, FrictionCone.cpp:48-58,
 * EnvironmentConstraint.cpp:31-40, EnvironmentNormal.cpp:36-50; ifopt inf = 1e20). */
cplb_status cplb_get_variable_bounds(const cplb_problem *p, double *lower, double *upper);
cplb_status cplb_get_constraint_bounds(const cplb_problem *p, double *lower, double *upper);

/* ---- parameters: the CplProblem forwarders (src/CplProblem.cpp:109-316) --------------------- */

/* CentroidalStatics::SetMass (src/Constraints/CentroidalStatics.cpp:20-23); mass <= 0 rejected like the planner ctor. */
cplb_status cplb_set_mass(cplb_problem *p, double mass);
cplb_status cplb_get_mass(const cplb_problem *p, double *mass);
/* Association of the 3-term sums behind Eigen's Vector3d dot() / norm() / squaredNorm() (FrictionCone.cpp:39-40,71,
 * Superquadric.cpp:66-68, MinimizeCentroidalVariables.cpp:142,145): 0 = (v0+v1)+v2 (Eigen >= 3.3 with its default
 * vectorisation; the default here), 1 = v0+(v1+v2) (Eigen 3.2 / EIGEN_DONT_VECTORIZE).  The reference pins no Eigen
 * version; results differ by at most one rounding of the reduced quantity.  Anything else -> CPLB_INVALID_ARGUMENT. */
cplb_status cplb_set_reduction_order(cplb_problem *p, int32_t order);
/* CplProblem::Set/GetManipulationWrench (src/CplProblem.cpp:263-272) */
cplb_status cplb_set_manipulation_wrench(cplb_problem *p, const double wrench[6]);
cplb_status cplb_get_manipulation_wrench(const cplb_problem *p, double wrench[6]);
/* CplProblem::SetMu/GetMu (src/CplProblem.cpp:275-303) -> EnvironmentClass::SetMu
 * (include/CentroidalPlanner/Environment/Environment.h:19-26): mu <= 0 -> CPLB_INVALID_ARGUMENT */
cplb_status cplb_set_mu(cplb_problem *p, double mu);
cplb_status cplb_get_mu(const cplb_problem *p, double *mu);
/* Ground::SetGroundZ/GetGroundZ (src/Ground.cpp:11-20); CPLB_RUNTIME_ERROR if env is not GROUND */
cplb_status cplb_set_ground_z(cplb_problem *p, double ground_z);
cplb_status cplb_get_ground_z(const cplb_problem *p, double *ground_z);
/* Superquadric::SetParameters/GetParameters (src/Superquadric.cpp:12-37): any R <= 0 or any P < 2 ->
 * CPLB_INVALID_ARGUMENT; CPLB_RUNTIME_ERROR if env is not SUPERQUADRIC */
cplb_status cplb_set_superquadric(cplb_problem *p, const double C[3], const double R[3], const double P[3]);
cplb_status cplb_get_superquadric(const cplb_problem *p, double C[3], double R[3], double P[3]);
/* CplProblem::Set/GetForceThreshold (src/CplProblem.cpp:306-316) -> FrictionCone::SetForceThreshold
 * (src/Constraints/FrictionCone.cpp:18-27); unknown contact -> CPLB_OUT_OF_RANGE (map::at) */
cplb_status cplb_set_force_threshold(cplb_problem *p, const char *contact_name, double F_thr);
cplb_status cplb_get_force_threshold(const cplb_problem *p, const char *contact_name, double *F_thr);
/* CplProblem::Set*Bounds / Get*Bounds (src/CplProblem.cpp:109-172) -> Variable3D::SetBounds
 * (src/Variable3D.cpp:28-40): any upper < lower -> CPLB_INVALID_ARGUMENT ("Inconsistent bounds"; like the
 * reference the new bounds are stored BEFORE the check fires). contact_name ignored for CPLB_BLOCK_COM. */
cplb_status cplb_set_bounds(cplb_problem *p, cplb_block block, const char *contact_name, const double lower[3],
                            const double upper[3]);
cplb_status cplb_get_bounds(const cplb_problem *p, cplb_block block, const char *contact_name, double lower[3],
                            double upper[3]);
/* MinimizeCentroidalVariables setters/getters (src/MinimizeCentroidalVariables.cpp:30-121) */
cplb_status cplb_set_pos_ref(cplb_problem *p, const char *contact_name, const double ref[3]);
cplb_status cplb_get_pos_ref(const cplb_problem *p, const char *contact_name, double ref[3]);
cplb_status cplb_set_force_ref(cplb_problem *p, const char *contact_name, const double ref[3]);
cplb_status cplb_get_force_ref(const cplb_problem *p, const char *contact_name, double ref[3]);
cplb_status cplb_set_com_ref(cplb_problem *p, const double ref[3]);
cplb_status cplb_get_com_ref(const cplb_problem *p, double ref[3]);
cplb_status cplb_set_com_weight(cplb_problem *p, double W_CoM);
cplb_status cplb_get_com_weight(const cplb_problem *p, double *W_CoM);
cplb_status cplb_set_pos_weight(cplb_problem *p, double W_p);   /* all contacts (:80-86) */
cplb_status cplb_set_force_weight(cplb_problem *p, double W_F); /* all contacts (:102-108) */
cplb_status cplb_set_contact_pos_weight(cplb_problem *p, const char *contact_name, double W_p);
cplb_status cplb_get_contact_pos_weight(const cplb_problem *p, const char *contact_name, double *W_p);
cplb_status cplb_set_contact_force_weight(cplb_problem *p, const char *contact_name, double W_F);
cplb_status cplb_get_contact_force_weight(const cplb_problem *p, const char *contact_name, double *W_F);

/* ---- evaluation: the hot path -------------------------------------------------------------- */

/* One batched evaluation.  Replaces, for N instances at once, what ifopt does per instance on behalf
 * of IpoptAdapter (SetVariables(x) + ...):
 *   g        Problem::EvaluateConstraints       -> each ConstraintSet::GetValues
 *            (CentroidalStatics.cpp:37-61, FrictionCone.cpp:30-45, EnvironmentConstraint.cpp:16-28,
 *             EnvironmentNormal.cpp:16-33, Ground.cpp:23-43, Superquadric.cpp:40-69)
 *   jac      Problem::EvalNonzerosOfJacobian    -> each ConstraintSet::FillJacobianBlock
 *            (CentroidalStatics.cpp:75-138, FrictionCone.cpp:60-103, EnvironmentConstraint.cpp:42-62,
 *             EnvironmentNormal.cpp:52-87, Ground.cpp:30-50, Superquadric.cpp:51-210)
 *   cost     Problem::EvaluateCostFunction      -> MinimizeCentroidalVariables::GetCost (:124-148)
 *   grad     Problem::EvaluateCostFunctionGradient -> MinimizeCentroidalVariables::FillJacobianBlock (:151-193)
 * Any of g / jac / cost / grad may be NULL: that output is not computed and not written.
 * Element counts per instance: x n, g m, jac nnz, cost 1, grad n.  `layout`/`ld` apply to every buffer
 * (cost is always cost[i]); ld is ignored for INSTANCE_MAJOR and may be 0 (= num_instances) otherwise. */
/* Optional per-instance parameters.  The reference holds ONE parameter set per CplProblem; a batch whose instances are
 * different planning problems of the same shape (other wrench, mass, friction, references ...) passes arrays here.
 * Every pointer may be NULL (= the problem's shared value set with cplb_set_*).  Arrays live in the same memory space
 * as x and follow the same layout rule: element e of instance i is arr[i*len + e] (INSTANCE_MAJOR) or arr[e*ld + i]
 * (COMPONENT_MAJOR), with len = the count given below; contact index = position in the caller's name vector.
 * Values are used as they are (no validation: they never pass through the host).  The Superquadric shape (C, R, P) is
 * always shared. */
typedef struct cplb_instance_params {
    const double *mass;             /* 1    CentroidalStatics::_m          (src/Constraints/CentroidalStatics.cpp:14,57) */
    const double *wrench;           /* 6    CentroidalStatics::_wrench_manip (:25-28,56) */
    const double *mu;               /* 1    EnvironmentClass::_mu           (Environment.h:46) */
    const double *force_threshold;  /* nc   FrictionCone::_F_thr            (src/Constraints/FrictionCone.cpp:14,39) */
    const double *ground_z;         /* 1    Ground::_ground_z               (src/Ground.cpp:26) */
    const double *com_ref;          /* 3    MinimizeCentroidalVariables::_CoM_ref (src/MinimizeCentroidalVariables.cpp:11) */
    const double *com_weight;       /* 1    _W_CoM (:13) */
    const double *pos_ref;          /* 3*nc _contact_vars_ref_map[..].position_value (:30-34) */
    const double *force_ref;        /* 3*nc ...force_value (:43-47) */
    const double *pos_weight;       /* nc   _pos_weight_map (:80-93) */
    const double *force_weight;     /* nc   _force_weight_map (:102-115) */
} cplb_instance_params;

/* cplb_eval_args.host_flags (cplb_eval_host only) */
#define CPLB_HOST_JAC_CONSTANTS_PRESENT 1 /* the constant slots of the caller's jac buffer already hold their values
                                             (cplb_fill_jacobian_constants, or an earlier full evaluation into the same
                                             buffer): the library MAY skip transferring them.  It does for
                                             COMPONENT_MAJOR (whole rows of the buffer are skipped); for INSTANCE_MAJOR
                                             whole instance rows travel (measured faster than strided copies) */

/* cplb_eval_args.host_flags bit for cplb_eval_device: the caller vouches that x and the per-instance arrays are NOT
 * outputs of the kernel launched just before on the same stream (they were complete before it started -- e.g. a queue
 * of independent batches).  Evaluation kernels are launched with programmatic stream serialization; with this bit they
 * issue their loads before waiting for the preceding kernel, hiding a first-wave HBM latency behind its tail.  Outputs
 * are always written after the preceding kernel has completed.  Without the bit, plain stream order holds. */
#define CPLB_DEVICE_INPUTS_READY 2

/* cplb_eval_args.host_flags bit for every evaluation call, INSTANCE_MAJOR only: `jac` is a PACKED slice per instance that holds
 * only the x-dependent Jacobian slots, jac[i*nv + q] = value of slot packed_to_slot[q] of instance i (cplb_get_packed_jacobian_map;
 * nv = 102 of 174 for a 4-contact Ground problem, 150 of 174 for a Superquadric one, 6+24*nc of 6+27*nc without environment).
 * The x-independent slots -- CentroidalStatics' 1.0 identities (CentroidalStatics.cpp:93-95), EnvironmentNormal's
 * (EnvironmentNormal.cpp:66-68), everything a Ground contributes (Ground.cpp:33-34,49) -- are neither computed into the slice nor
 * transferred: cplb_get_jacobian_constants has their values, cplb_unpack_jacobian rebuilds full rows on the host, and the IFOPT
 * views (cplb/ifopt_views.hpp) read a packed batch through the slot map.  The kernel keeps a smaller output tile per instance
 * and a host call moves 35 % fewer device -> host bytes (4-contact Ground, g + Jacobian).  The packed values are bit-identical to
 * the same slots of a full evaluation.  Any other layout -> CPLB_INVALID_ARGUMENT. */
#define CPLB_JAC_PACKED 4

/* Same family, one step further (INSTANCE_MAJOR only, not together with CPLB_JAC_PACKED): `jac` is a COMPUTED slice per instance
 * that also leaves out the slots whose value is a plain copy of an entry of the instance's own x, +x[col] or -x[col] -- the p_k
 * entries of the moment rows (-skew(F_k), CentroidalStatics.cpp:108-113) and FrictionCone's first row (-n and -F,
 * FrictionCone.cpp:82-84, :93-95): 12 per contact.  The caller holds x already, so they need not come back over the link.  What
 * travels are the entries that take arithmetic: the 6 CoM sums, per contact the 6 moment-row entries +-(p - c), FrictionCone's
 * second row (6) and a Superquadric's 12 -- 54 of 174 doubles for a 4-contact Ground problem, 102 of 174 for a Superquadric one.
 * cplb_get_jacobian_slot_sources says for every structural slot where its value comes from; cplb_expand_jacobian rebuilds full
 * rows on the host (bit-identical to a full evaluation: a negation is exact); the IFOPT views read such a batch in place. */
#define CPLB_JAC_COMPUTED 8

typedef struct cplb_eval_args {
    int64_t num_instances;
    int32_t layout; /* cplb_layout */
    int32_t host_flags; /* 0, or CPLB_HOST_* (cplb_eval_host) / CPLB_DEVICE_* (cplb_eval_device) bits */
    int64_t ld;
    const double *x;
    double *g;
    double *jac;
    double *cost;
    double *grad;
    const cplb_instance_params *per_instance; /* NULL: every instance uses the problem's shared parameters */
} cplb_eval_args;

/* All pointers are DEVICE pointers on the problem's device; the kernel is enqueued on `cuda_stream`
 * (a cudaStream_t, NULL = default stream) and the call returns without synchronising. */
cplb_status cplb_eval_device(cplb_problem *p, const cplb_eval_args *args, void *cuda_stream);

/* cplb_eval_device for one shard of a sharded problem: all pointers are device pointers on THAT shard's device and hold the
 * shard's instances only (args->num_instances = their count), `cuda_stream` is a stream of that device. */
cplb_status cplb_eval_device_shard(cplb_problem *p, int32_t shard, const cplb_eval_args *args, void *cuda_stream);

/* All pointers are HOST pointers (pinned memory makes the copies asynchronous and faster, pageable
 * works).  Instances are cut into chunks; each chunk's host->device copy, kernel and device->host copy
 * run on one of several internal streams so that both copy directions overlap the kernels.  Returns
 * after every output has landed in the host buffers. */
cplb_status cplb_eval_host(cplb_problem *p, const cplb_eval_args *args);

/* The same call for a QUEUE of batches (several IPOPT callback rounds or planner requests in flight): _begin only
 * enqueues the chunked copies and kernels and hands back a ticket, _wait returns once that call's outputs have landed.
 * With two sets of host buffers (begin k+1, wait k) the device -> host link, which bounds the synchronous call, never
 * idles between batches.  Host buffers must be pinned (cplb_host_alloc; CPLB_INVALID_ARGUMENT otherwise) and stay
 * untouched until the wait; at most 4 calls may be outstanding (a ticket is reused after 4 more begins).
 * Replaces: N x the reference's Problem::Evaluate* calls per batch (ifopt, SURVEY Appendix B.5-6), as cplb_eval_host. */
cplb_status cplb_eval_host_begin(cplb_problem *p, const cplb_eval_args *args, int32_t *ticket);
cplb_status cplb_eval_host_wait(cplb_problem *p, int32_t ticket);

/* Structural Jacobian slots whose value does not depend on x: the 1.0 identities of CentroidalStatics
 * (CentroidalStatics.cpp:93-95) and EnvironmentNormal (EnvironmentNormal.cpp:66-68) and, for Ground, its explicit
 * zeros and the (0,0,1) gradient (Ground.cpp:33-34,49).  IPOPT keeps one values[] array per problem, so a consumer
 * can fill these once and let every later cplb_eval_host skip them (CPLB_HOST_JAC_CONSTANTS_PRESENT): for a 4-contact
 * Ground problem 72 of the 174 slots, i.e. 35 % of the device -> host bytes.
 * is_constant[nnz] (1/0) and value[nnz] (meaningful where is_constant) may each be NULL. */
cplb_status cplb_get_jacobian_constants(const cplb_problem *p, uint8_t *is_constant, double *value);
/* Writes the constant slots of a HOST jac buffer holding num_instances instances in the given layout. */
cplb_status cplb_fill_jacobian_constants(const cplb_problem *p, int64_t num_instances, int32_t layout, int64_t ld,
                                         double *jac_host);

/* The x-dependent slots in slot order: element q of a CPLB_JAC_PACKED slice is structural slot packed_to_slot[q] (0-based index
 * into the (iRow, jCol) list of cplb_get_jacobian_structure).  packed_to_slot[*num_packed] may be NULL to query the count only. */
cplb_status cplb_get_packed_jacobian_map(const cplb_problem *p, int32_t *num_packed, int32_t *packed_to_slot);
/* Host helper: expands num_instances packed slices (packed[i*nv + q]) into full instance-major rows full[i*nnz + s]: the
 * values[] array IpoptAdapter::eval_jac_g hands to IPOPT, constants included. */
cplb_status cplb_unpack_jacobian(const cplb_problem *p, int64_t num_instances, const double *packed, double *full);

/* Where each structural slot's value comes from, for consumers of CPLB_JAC_COMPUTED slices.  kind[nnz], source[nnz] (either may
 * be NULL): CPLB_SLOT_CONSTANT -> cplb_get_jacobian_constants' value (source -1); CPLB_SLOT_COPY -> x[source] of the same instance;
 * CPLB_SLOT_NEGATED_COPY -> -x[source]; CPLB_SLOT_COMPUTED -> element `source` of the instance's computed slice (the computed slots
 * appear in it in slot order).  *num_computed = doubles per instance of a computed slice. */
#define CPLB_SLOT_CONSTANT 0
#define CPLB_SLOT_COPY 1
#define CPLB_SLOT_NEGATED_COPY 2
#define CPLB_SLOT_COMPUTED 3
cplb_status cplb_get_jacobian_slot_sources(const cplb_problem *p, int32_t *num_computed, int32_t *kind, int32_t *source);
/* Host helper: expands num_instances computed slices (computed[i*nv + q]) and the x they were evaluated at (x[i*n + c]) into full
 * instance-major rows full[i*nnz + s], constants and copies included. */
cplb_status cplb_expand_jacobian(const cplb_problem *p, int64_t num_instances, const double *x, const double *computed, double *full);

/* ---- the caller of the path: lock-step solves --------------------------------------------------------------------------- */

/* Replaces, for N instances of the problem at once, cpl::CentroidalPlanner::Solve (src/CentroidalPlanner.cpp:22-34:
 * ifopt::IpoptSolver::Solve on one CplProblem, then CplProblem::GetSolution).  IPOPT is a host library that is not part of
 * this repository; the production integration keeps it (one IPOPT thread per instance over the IFOPT views in lock-step mode,
 * INTEGRATION.md).  cplb_solve_device is the same round with the solver written out and run on the GPU: the primal-dual
 * interior-point method IPOPT implements (slack reformulation, log barrier, fraction-to-the-boundary rule, monotone barrier update,
 * gradient-based scaling, bound push and relaxation, kappa_sigma safeguard, fixed variables removed, second-order correction; tol as
 * ifopt sets it), with a forward-difference Lagrangian Hessian (the reference runs IPOPT's limited-memory approximation), an l1
 * merit line search, Levenberg-Marquardt damping and a feasibility polish.  It is NOT IPOPT: iterates differ, solutions are local
 * minima of the same NLP to the same tolerances.  Every round is four batched evaluations of the hot path and four kernels that
 * keep one instance's KKT system in shared memory (csrc/cplb_solver.cu); x never leaves the device.
 * Options carry IPOPT's names where the meaning is IPOPT's. */
typedef struct cplb_solver_options {
    double tol;                      /* 1e-3: ifopt's IpoptSolver default */
    double mu_init;                  /* 0.1 */
    double bound_push, bound_frac;   /* 1e-2, 1e-2 */
    double nlp_scaling_max_gradient; /* 100 */
    double constr_viol_tol;          /* 1e-4 */
    double polish_viol_tol;          /* 1e-9: constraint violation after the feasibility polish */
    double bound_relax_factor;       /* 1e-8 */
    int32_t max_iter;                /* 500 */
    int32_t max_backtracks;          /* 30 */
    int32_t tail_instances;          /* -1.  Once no more than this many instances are still running, they leave the lock-step rounds
                                        and each finishes on its own inside one kernel (a straggler then costs only its own
                                        iterations).  -1: as many as the GPU holds at once; 0: lock-step rounds to the end. */
} cplb_solver_options;
void cplb_solver_default_options(cplb_solver_options *options);

#define CPLB_SOLVE_SUCCEEDED 0              /* Ipopt::Solve_Succeeded: at the final iterate the scaled error (dual_inf, the
                                               complementarity, the scaled primal residual) is <= tol and constr_viol <=
                                               polish_viol_tol.  (A feasibility polish with frozen multipliers follows IPOPT's
                                               test; an iterate it leaves with a scaled error above tol takes Newton steps again.) */
#define CPLB_SOLVE_MAX_ITERATIONS 1         /* Ipopt::Maximum_Iterations_Exceeded */
#define CPLB_SOLVE_INVALID_NUMBER 2         /* Ipopt::Invalid_Number_Detected */

/* Device arrays the solve fills (instance-major; lam and the three counters may be NULL). */
typedef struct cplb_solve_outputs {
    double *x;            /* [N n]  final iterates, clipped to the variable bounds (honor_original_bounds); CplProblem::GetSolution
                             reads one instance's slice (cplb::BatchedProblem::GetSolution) */
    int32_t *status;      /* [N]    CPLB_SOLVE_* */
    int32_t *iterations;  /* [N] */
    double *cost;         /* [N]    MinimizeCentroidalVariables::GetCost at the final iterate.  That is x, unless the clipping moved an
                             entry of x back onto its bound (by at most bound_relax_factor * max(|bound|, 1)): cost, constr_viol
                             and dual_inf are the values of the iterate before the clipping */
    double *constr_viol;  /* [N]    max over rows of the violation of the row's bounds at the final iterate: equality rows against
                             their value, inequality rows against their bounds relaxed by bound_relax_factor * max(|bound|, 1)
                             (the bounds the solver works with); NaN for a start rejected as CPLB_SOLVE_INVALID_NUMBER before its
                             first iteration (0 iterations) */
    double *dual_inf;     /* [N]    scaled dual infeasibility (IPOPT's, divided by s_d) at the final iterate; NaN for such a
                             rejected start */
    double *lam;          /* [N m]  constraint multipliers, unscaled, IPOPT's sign (L = f + lam^T g: >= 0 on an active upper
                             bound, <= 0 on an active lower one), or NULL */
    int32_t *rounds;              /* HOST: lock-step rounds executed, or NULL */
    int64_t *evaluations;         /* HOST: batched evaluations launched, or NULL */
    int64_t *instance_evaluations; /* HOST: instances evaluated in total, or NULL */
    int64_t *tail_instances;      /* HOST: instances that finished on their own after the lock-step rounds, or NULL */
} cplb_solve_outputs;

/* x0 [N n]: starting points (DEVICE pointer, like every array of `out`), variable and constraint bounds as set on the problem.
 * per_instance: NULL, or per-instance parameter arrays as for cplb_eval_device (DEVICE pointers, instance-major, row i = instance
 * i): every instance then solves ITS planning problem -- its own wrench, mass, friction coefficient, references ... -- which is what
 * a sweep over planning scenarios is; the bounds stay the problem's.
 * Synchronises `cuda_stream` (the host reads one counter per round).  Single-device problems only: one solve batch per GPU,
 * instances shard across GPUs by running one batch per device.
 * Shape limit: one instance's KKT system lives in one CTA's shared memory (227 KB on sm_100).  A problem whose block would not fit
 * -- above 10 contacts with an environment, 13 without one -- is refused with CPLB_INVALID_ARGUMENT and a message naming its
 * contact count and the largest count of its kind that fits. */
cplb_status cplb_solve_device(cplb_problem *p, int64_t num_instances, const double *x0, const cplb_instance_params *per_instance,
                              const cplb_solver_options *options, const cplb_solve_outputs *out, void *cuda_stream);

/* ---- first-order derivative test ----------------------------------------------------------------------------------------- */

/* Replaces, for N instances at once, the derivative check the reference turns on before every solve: cpl::CentroidalPlanner::Solve
 * sets IPOPT's `derivative_test first-order` (src/CentroidalPlanner.cpp:26), which compares the Jacobian and the cost gradient with
 * forward differences of the problem's own g and f at the starting point.  The rule, per instance with x its point:
 *   h_j  = perturbation * (|x_j| > 1 ? |x_j| : 1)                   (a NaN x_j takes h_j = perturbation)
 *   fd   = (g(x + h_j e_j) - g(x)) / h_j,  (f(x + h_j e_j) - f(x)) / h_j        (divided by h_j, as IPOPT does)
 *   rel  = |fd - exact| / (|exact| > 1 ? |exact| : 1)
 *   an entry is wrong iff !(rel <= tol): NaN and Inf count as wrong.
 * Every gradient entry and EVERY entry (r, c) of the dense m x n Jacobian is compared; outside the declared structure the exact
 * value is 0, so a derivative the structure misses is found too.  g, f, the Jacobian and the gradient are the batched evaluator's
 * own values, bit for bit what cplb_eval_device returns.  The worst entry is the first one with the largest rel (NaN counted as
 * +inf) in the order: gradient columns 0..n-1, then the Jacobian row by row, column ascending.  One CTA per instance evaluates
 * the n perturbed points in chunks inside shared memory (csrc/cplb_derivtest.cu); nothing is widened in global memory. */
typedef struct cplb_derivative_test_options {
    double perturbation; /* 1e-8: IPOPT's derivative_test_perturbation */
    double tol;          /* 1e-4: IPOPT's derivative_test_tol */
} cplb_derivative_test_options;
void cplb_derivative_test_default_options(cplb_derivative_test_options *options);

typedef struct cplb_derivative_test_outputs { /* DEVICE arrays, instance-major; every pointer may be NULL */
    int32_t *num_wrong;         /* [N]     wrong entries: gradient + every (row, col) of the dense Jacobian */
    int32_t *num_wrong_outside; /* [N]     of those, Jacobian entries outside the declared structure */
    double *max_rel_error;      /* [N]     rel of the worst entry, as computed (NaN stays NaN) */
    int32_t *worst_row;         /* [N]     -1 = cost gradient */
    int32_t *worst_col;         /* [N] */
    double *jac_fd;             /* [N nnz] forward differences at the structural slots, in slot order */
    double *grad_fd;            /* [N n] */
} cplb_derivative_test_outputs;

/* x [N n]: the points (DEVICE pointer; the caller's column order).  per_instance: NULL, or per-instance parameter arrays as for
 * cplb_solve_device (DEVICE pointers, instance-major).  options: NULL = defaults.  Asynchronous on `cuda_stream`, like
 * cplb_eval_device: it does not synchronise the stream (the first call on a problem uploads a table of the Jacobian structure
 * once, on a stream of its own).  Counts one launch in cplb_get_launch_count.  Argument errors are reported before any CUDA call:
 * NULL p or out, or NULL x with N > 0 -> CPLB_NULL_POINTER; N < 0, a perturbation that is not finite and positive, a tol that is
 * not positive -> CPLB_INVALID_ARGUMENT; N = 0 -> CPLB_OK, nothing launched.  Single-device problems only, like
 * cplb_solve_device.  Every shape up to CPLB_MAX_CONTACTS contacts is supported, in every environment. */
cplb_status cplb_derivative_test_device(cplb_problem *p, int64_t num_instances, const double *x, const cplb_instance_params *per_instance,
                                        const cplb_derivative_test_options *options, const cplb_derivative_test_outputs *out,
                                        void *cuda_stream);

/* ---- Jacobian products ------------------------------------------------------------------------------------------------------ */

/* What a first-order or penalty method, the Lagrangian gradient of an outside solver, or a reverse-mode autodiff caller needs
 * from the Jacobian, without materialising it: one kernel reads x (and lambda / v) and writes the products (csrc/cplb_products.cu).
 *   reverse  x_bar = obj_factor * grad f(x) + J(x)^T lambda        (IPOPT's sigma / lambda naming, as in eval_h)
 *   forward  g_dot = J(x) v,   f_dot = grad f(x) . v
 * Bit contract: the results are exactly those of a caller that materialises J and the gradient with cplb_eval_device (the
 * evaluator's bits, every structural slot present, Ground's explicit zeros included) and multiplies them in slot order, with one
 * IEEE multiply and one IEEE add per term and no FMA:
 *   x_bar[c] starts at obj_factor * grad[c] (at +0.0 when obj_factor is NULL); then + J[s] * lambda[iRow[s]] for every structural
 *            slot s with jCol[s] == c, slots ascending (= rows ascending);
 *   g_dot[r] starts at +0.0; then + J[s] * v[jCol[s]] for the slots of row r, slots ascending (= columns ascending);
 *   f_dot    starts at +0.0; then + grad[c] * v[c] for c = 0..n-1.
 * So 0 * Inf in a structural-zero slot gives NaN, as it would for the materialising caller.  (A multiply is dropped only where the
 * result has the same bits: by the 1.0 identity entries.) */
typedef struct cplb_jacobian_products_args {
    int64_t num_instances;
    const double *x;                          /* [N n] instance-major, DEVICE */
    const cplb_instance_params *per_instance; /* NULL, or device arrays as for cplb_solve_device (instance-major) */
    /* reverse mode */
    const double *lambda;                     /* [N m] or NULL (no J^T term) */
    const double *obj_factor;                 /* [N]   or NULL (no gradient term) */
    double *x_bar;                            /* [N n] or NULL (reverse product not computed) */
    /* forward mode */
    const double *v;                          /* [N n] */
    double *g_dot;                            /* [N m] or NULL */
    double *f_dot;                            /* [N]   or NULL */
} cplb_jacobian_products_args;

/* Every array is a DEVICE array on the problem's device, instance-major.  Asynchronous on `cuda_stream`; one launch, counted in
 * cplb_get_launch_count.  Argument errors are reported before any CUDA call: NULL p or args, or NULL x with N > 0 ->
 * CPLB_NULL_POINTER; g_dot or f_dot set with v NULL -> CPLB_NULL_POINTER; x_bar set with both lambda and obj_factor NULL, no output
 * requested, N < 0 or N >= 2^31 -> CPLB_INVALID_ARGUMENT.  N = 0 -> CPLB_OK, nothing launched.  Single-device problems only, like
 * cplb_solve_device.  Every shape up to CPLB_MAX_CONTACTS contacts is supported, in every environment.  No derivatives with
 * respect to the parameters, no second derivatives. */
cplb_status cplb_jacobian_products_device(cplb_problem *p, const cplb_jacobian_products_args *args, void *cuda_stream);

/* Pinned host memory for cplb_eval_host buffers (cudaHostAlloc / cudaFreeHost). */
cplb_status cplb_host_alloc(size_t bytes, void **out);
cplb_status cplb_host_free(void *ptr);

/* Which of the two COMPONENT_MAJOR kernels evaluates this problem.  AUTO (default) picks by shape and batch size: one thread
 * per (instance, contact) for small batches, one thread per instance once several waves of CTAs are in flight (4- and 8-contact
 * problems with shared parameters; measured crossovers in DESIGN.md 4.1b).  The two kernels run the same arithmetic in the
 * same order and must return the same bits: the parity tests force each of them on the same inputs, and dispatch
 * measurements time both.  PER_INSTANCE on a problem with another contact count -> CPLB_INVALID_ARGUMENT; evaluations with
 * per-instance parameter arrays always take the per-contact kernel.  No reference counterpart (the reference has one code path:
 * src/Constraints/CentroidalStatics.cpp:37-61,75-138 et al.). */
#define CPLB_KERNEL_AUTO 0
#define CPLB_KERNEL_PER_CONTACT 1
#define CPLB_KERNEL_PER_INSTANCE 2
cplb_status cplb_set_component_major_kernel(cplb_problem *p, int32_t kernel);
/* The same for the two INSTANCE_MAJOR kernels: a warp per tile of 32/LPI instances (lanes = an (instance, contact) grid) or a
 * CTA per tile (one warp per contact, lanes = consecutive instances).  Same arithmetic, same bits; AUTO picks by shape and, for
 * a few shapes, by the requested outputs and the batch size (measured crossovers: DESIGN.md 4.2b). */
#define CPLB_KERNEL_WARP_TILE 1
#define CPLB_KERNEL_CTA_TILE 2
cplb_status cplb_set_instance_major_kernel(cplb_problem *p, int32_t kernel);
/* CUDA ordinal this problem evaluates on; -1 while a problem created with device = -1 has not evaluated yet. */
cplb_status cplb_get_device(const cplb_problem *p, int32_t *device);

/* Number of kernels this problem has launched so far (bench.py's gpu_launches). */
cplb_status cplb_get_launch_count(const cplb_problem *p, int64_t *launches);
/* Average device time (ms, CUDA events on the launch stream) of the kernels launched by
 * cplb_eval_device between cplb_timing_begin and cplb_timing_end; used by bench.py for the roofline. */
cplb_status cplb_timing_begin(cplb_problem *p);
cplb_status cplb_timing_end(cplb_problem *p, double *avg_kernel_ms, int64_t *kernels);

#ifdef __cplusplus
}
#endif
#endif /* CPL_BATCHED_H */
