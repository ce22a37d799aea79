// cplb_kernels_im.cuh -- instance-major (per-instance slices) evaluation kernel and its launcher templates.  One translation
// unit per environment kind instantiates launch_im_env<ENV> (cplb_kernels_im_*.cu) so that the kinds compile in parallel.
#ifndef CPLB_KERNELS_IM_CUH
#define CPLB_KERNELS_IM_CUH

#include <mutex>
#include <vector>

#include "cplb_launch.cuh"

namespace cplb {

constexpr int kMaxDevices = 64;
// AUTO: the CTA-tile kernel where it measured faster (profiles/r02_instance_major.md): an even number of contacts from 4 on
// (n = 3 + 9 nc is then odd: its lane = instance shared-memory accesses are conflict-free), one contact, more than 8 contacts.
// With an odd contact count > 1 the row lengths n, m are even and lanes that step through instances collide on a few banks:
// those shapes and the two-contact one stay on the warp-tile kernel.
inline bool instance_major_auto_is_cta_tile(int nc) { return (nc % 2 == 0 && nc >= 4) || nc == 1 || nc > 8; }

// ================================================================================================
// instance-major (AoS): warp tile, LPI lanes per instance, bulk async copies in and out
// ================================================================================================

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// global -> shared bulk copy (TMA unit), completion signalled on the mbarrier
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global bulk copy
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

struct TileEmitter {
    double* gp;  // this instance's slices inside the warp's shared-memory tiles
    double* jp;
    double* gradp;
    __device__ __forceinline__ void g(int row, double v) const { gp[row] = v; }
    __device__ __forceinline__ void j(int slot, double v) const { jp[slot] = v; }
    __device__ __forceinline__ void grad(int col, double v) const { gradp[col] = v; }
};

// shared memory per warp (doubles): [x0: T*n][x1: T*n][g: T*m][jac: T*nnz][grad: T*n][cost: T]; then 2 mbarriers per warp
__host__ __device__ inline size_t tile_doubles(int T, int n, int m, int nnz, unsigned flags)
{
    size_t d = 2 * (size_t)T * n;
    if (flags & CPLB_WANT_G) d += (size_t)T * m;
    if (flags & CPLB_WANT_J) d += (size_t)T * nnz;
    if (flags & CPLB_WANT_GRAD) d += (size_t)T * n;
    if (flags & CPLB_WANT_COST) d += (size_t)T;
    return (d + 1) & ~(size_t)1;  // keep every warp's region 16-byte aligned
}

// warp-cooperative contiguous copy, used for ragged / misaligned tiles instead of the bulk engine
__device__ __forceinline__ void warp_copy(double* dst, const double* src, int count, int lane)
{
    for (int e = lane; e < count; e += 32) dst[e] = src[e];
}

// Persistent warps.  Warp w of the grid owns tiles w, w + W, w + 2W, ... (W = warps in the grid, the grid is
// sized to what is resident at once).  Per tile of T = 32/LPI consecutive instances:
//   - the x slice (T*n contiguous doubles) arrives by one bulk async copy into one of two buffers; the copy of
//     the NEXT tile is issued before the current one is consumed, so its HBM latency hides behind compute;
//   - LPI lanes per instance (one lane per contact; the six statics rows are dealt to the same lanes) scatter
//     results into shared-memory tiles laid out exactly like the output slices;
//   - the tiles leave with bulk async stores; the warp only waits for the engine to have READ the tiles
//     right before it overwrites them with the next tile's results.
// No block-wide barrier: every warp runs its own pipeline (mbarriers + __syncwarp only).
template <int ENV, int LPI, int WARPS, unsigned FLAGS, bool PERINST>
__global__ void __launch_bounds__(WARPS * 32) eval_instance_major(const __grid_constant__ CplbParams P, const CplbIo io,
                                                                   const unsigned flags_rt, const int aligned16,
                                                                   const __grid_constant__ CplbInstParams Q,
                                                                   const __grid_constant__ CplbParamTile PT)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    pdl_trigger();
    if (!(flags_rt & CPLB_INPUTS_READY)) pdl_wait();
    constexpr int T = 32 / LPI;  // instances per warp tile
    const unsigned flags = FLAGS ? FLAGS : (flags_rt & 15u);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nc = P.nc, n = P.n, m = P.m, nnz = P.nnz;
    const long long tiles = (io.N + T - 1) / T;
    const long long stride = (long long)gridDim.x * WARPS;
    long long tile = (long long)blockIdx.x * WARPS + warp;
    if (tile >= tiles) return;  // whole warp leaves together

    const int ptot = PERINST ? PT.total : 0;  // staged per-instance parameter slices, double-buffered like x
    const size_t per_warp = tile_doubles(T, n, m, nnz, flags) + 2 * (size_t)ptot;
    double* xbuf = reinterpret_cast<double*>(smem_raw) + (size_t)warp * per_warp;
    double* pbuf = xbuf + 2 * (size_t)T * n;
    double* cur = pbuf + 2 * (size_t)ptot;
    double* gs = nullptr;
    double* js = nullptr;
    double* grads = nullptr;
    double* costs = nullptr;
    if (flags & CPLB_WANT_G) { gs = cur; cur += (size_t)T * m; }
    if (flags & CPLB_WANT_J) { js = cur; cur += (size_t)T * nnz; }
    if (flags & CPLB_WANT_GRAD) { grads = cur; cur += (size_t)T * n; }
    if (flags & CPLB_WANT_COST) { costs = cur; }
    uint64_t* bar = reinterpret_cast<uint64_t*>(reinterpret_cast<double*>(smem_raw) + (size_t)WARPS * per_warp) + 2 * warp;

    const uint32_t xbytes = (uint32_t)(T * n * sizeof(double));
    // bulk copies need 16-byte aligned addresses and sizes: full tiles of 16B-aligned buffers only
    auto is_bulk = [&](long long t) { return aligned16 && (t + 1) * T <= io.N; };
    // a local copy: reading Q.arr in place changes the generated code of the per-instance variants
    const double* parr[CPLB_NUM_INST_ARRAYS];
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++) parr[a] = Q.arr[a];
    // one elected lane: x tile + every staged parameter slice of tile t into buffer `buf`, all on one mbarrier
    auto issue_loads = [&](long long t, int buf) {
        mbar_expect_tx(&bar[buf], xbytes + (uint32_t)(ptot * sizeof(double)));
        bulk_g2s(xbuf + (size_t)buf * T * n, io.x + t * T * n, xbytes, &bar[buf]);
        if (PERINST) {
#pragma unroll
            for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
                if (PT.off[a] >= 0)
                    bulk_g2s(pbuf + (size_t)buf * ptot + PT.off[a], parr[a] + t * T * PT.len[a],
                             (uint32_t)(T * PT.len[a] * sizeof(double)), &bar[buf]);
        }
    };

    if (lane == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        fence_proxy_async_smem();
        if (is_bulk(tile)) issue_loads(tile, 0);
    }
    __syncwarp();
    if (flags_rt & CPLB_INPUTS_READY) pdl_wait();  // the first tile's x is already on its way; nothing is stored before this

    const int inst = lane / LPI, s = lane % LPI;
    bool stores_in_flight = false;
    for (int it = 0; tile < tiles; tile += stride, it++) {
        const int b = it & 1;
        double* xs = xbuf + (size_t)b * T * n;
        const long long i0 = tile * T;
        const int cnt = (io.N - i0) < T ? (int)(io.N - i0) : T;
        const bool bulk = is_bulk(tile);

        // prefetch the next tile's x into the other buffer (its previous contents were consumed an iteration ago)
        const long long next = tile + stride;
        if (lane == 0 && next < tiles && is_bulk(next)) {
            fence_proxy_async_smem();
            issue_loads(next, b ^ 1);
        }
        const double* ptile = pbuf + (size_t)b * ptot;
        if (bulk) {
            mbar_wait(&bar[b], (uint32_t)((it >> 1) & 1));
        } else {
            warp_copy(xs, io.x + i0 * n, cnt * n, lane);
            if (PERINST) {
#pragma unroll
                for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
                    if (PT.off[a] >= 0)
                        warp_copy(pbuf + (size_t)b * ptot + PT.off[a], parr[a] + i0 * PT.len[a], cnt * PT.len[a], lane);
            }
        }
        // the output tiles are about to be overwritten: the engine must have finished reading the previous ones
        if (stores_in_flight) {
            if (lane == 0) bulk_wait_read_all();
            stores_in_flight = false;
        }
        __syncwarp();

        // ---- compute: lane (inst, s) handles contacts s, s+LPI, ... and statics rows s, s+LPI, ... ----
        // The body is instantiated per parameter source: shared block, staged per-instance tiles, or per-instance arrays read
        // with read-only global loads (kept free of any shared-memory alternative so that the compiler can hoist and batch them).
        const unsigned live = __ballot_sync(0xffffffffu, inst < cnt);  // lanes that hold an instance of this tile (shuffle mask)
        auto compute_instance = [&](const auto& ps) {
            const double* xi = xs + (size_t)inst * n;
            TileEmitter em{gs ? gs + (size_t)inst * m : nullptr, js ? js + (size_t)inst * nnz : nullptr,
                           grads ? grads + (size_t)inst * n : nullptr};
            const double c[3] = {xi[0], xi[1], xi[2]};
            for (int j = s; j < nc; j += LPI) {
                const int k = P.perm[j];
                const double* xk = xi + 3 + 9 * k;
                const double F[3] = {xk[0], xk[1], xk[2]};
                const double p[3] = {xk[3], xk[4], xk[5]};
                const double nn[3] = {xk[6], xk[7], xk[8]};
                contact_rows<ENV>(P, ps, em, nc, j, k, c, F, p, nn, flags);
            }
            // CentroidalStatics rows: row r's running sum visits the contacts in sorted-name order
            // (CentroidalStatics.cpp:44-54); the six rows are independent, so they are dealt to the lanes.
            // Lanes of a warp hold different r, so the row is selected by indices, not by a switch: row 3+q is
            //   v += d_{q+1} F_{q+2} - d_{q+2} F_{q+1}   [(p - CoM) x F]
            // and its CoM block is  a -= sa*F[ia],  b -= sb*F[ib]  (:128-133; multiplying by +-1 is exact).
            if (flags & (CPLB_WANT_G | CPLB_WANT_J)) {
                const int L = jac_moment_row_len(nc);
                for (int r = s; r < 6; r += LPI) {
                    const bool mom = r >= 3;
                    const int q = mom ? r - 3 : 0;
                    const int i1 = q == 2 ? 0 : q + 1, i2 = q == 0 ? 2 : q - 1;  // (q+1)%3, (q+2)%3
                    const int ia = q == 2 ? 1 : 2, ib = q == 0 ? 1 : 0;
                    const double sa = q == 1 ? -1.0 : 1.0, sb = q == 1 ? 1.0 : -1.0;
                    double v = 0.0, a = 0.0, bb = 0.0;
                    for (int j = 0; j < nc; j++) {
                        const double* xk = xi + 3 + 9 * P.perm[j];
                        if (mom) {
                            const double x1 = xk[3 + i1] - xi[i1], x2 = xk[3 + i2] - xi[i2];  // p - CoM
                            v += x1 * xk[i2] - x2 * xk[i1];
                            a -= sa * xk[ia];
                            bb -= sb * xk[ib];
                        } else {
                            v += xk[r];
                        }
                    }
                    if (flags & CPLB_WANT_G) em.g(r, mom ? v - ps.wrench(r) : (v - ps.wrench(r)) + ps.mg(r));
                    if ((flags & CPLB_WANT_J) && mom) {
                        em.j(3 * nc + q * L + 0, a);
                        em.j(3 * nc + q * L + 1, bb);
                    }
                }
            }
            if (flags & CPLB_WANT_COST) {  // MinimizeCentroidalVariables.cpp:126-147, sorted order
                // every lane evaluates the terms of its own contacts; lane 0 of the instance collects them with shuffles
                // in sorted order j = 0, 1, ... -- the same running sum as the reference's loop (0.0 + t0 is exact)
                double cost = 0.0;
                for (int r = 0; r * LPI < nc; r++) {
                    const int j = r * LPI + s;
                    double t = 0.0;
                    if (j < nc) {
                        const int k = P.perm[j];
                        const double* xk = xi + 3 + 9 * k;
                        const double F[3] = {xk[0], xk[1], xk[2]};
                        const double p[3] = {xk[3], xk[4], xk[5]};
                        t = contact_cost(ps, P.reduction_order, k, F, p);
                    }
#pragma unroll
                    for (int q = 0; q < LPI; q++) {
                        const double tq = __shfl_sync(live, t, inst * LPI + q);
                        if (r * LPI + q < nc) cost += tq;
                    }
                }
                if (s == 0) {
                    cost += com_cost(ps, P.reduction_order, c);
                    costs[inst] = cost;
                }
            }
            if (s == 0) {
                if (flags & CPLB_WANT_GRAD) {
#pragma unroll
                    for (int q = 0; q < 3; q++) em.grad(q, ps.W_com() * (c[q] - ps.com_ref(q)));
                }
            }
        };
        if (inst < cnt) {
            if constexpr (PERINST) {
                if (ptot)
                    compute_instance(TileInstanceParams{P, Q, PT, ptile, inst});
                else
                    compute_instance(InstanceParams<false>{P, Q, i0 + inst, 0});
            } else {
                compute_instance(SharedParams{P});
            }
        }

        // ---- ship the tiles ------------------------------------------------------------------------
        if (bulk) {
            fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the async (TMA) proxy
            __syncwarp();
            if (lane == 0) {
                if (gs) bulk_s2g(io.g + i0 * m, gs, (uint32_t)(T * m * sizeof(double)));
                if (js) bulk_s2g(io.jac + i0 * nnz, js, (uint32_t)(T * nnz * sizeof(double)));
                if (grads) bulk_s2g(io.grad + i0 * n, grads, (uint32_t)(T * n * sizeof(double)));
                bulk_commit();
            }
            stores_in_flight = true;
            if (costs && lane < T) io.cost[i0 + lane] = costs[lane];
        } else {
            __syncwarp();
            if (gs) warp_copy(io.g + i0 * m, gs, cnt * m, lane);
            if (js) warp_copy(io.jac + i0 * nnz, js, cnt * nnz, lane);
            if (grads) warp_copy(io.grad + i0 * n, grads, cnt * n, lane);
            if (costs && lane < cnt) io.cost[i0 + lane] = costs[lane];
        }
        __syncwarp();  // all lanes done with xs and the tiles before the next iteration touches them
    }
    if (stores_in_flight && lane == 0) bulk_wait_read_all();  // shared memory must outlive the engine's reads
    __syncwarp();
}

template <int ENV, int LPI, int WARPS, unsigned FLAGS, bool PERINST>
cudaError_t launch_im_kernel(const CplbParams& P, const CplbIo& io, unsigned flags, size_t smem, const CplbInstParams* Q,
                                    const CplbParamTile& PT, cudaStream_t st)
{
    constexpr int T = 32 / LPI;
    auto kern = eval_instance_major<ENV, LPI, WARPS, FLAGS, PERINST>;
    // Per kernel instantiation, process-wide: the opt-in dynamic shared memory limit of each device (only ever RAISED -- the
    // attribute belongs to the function on a device, not to a thread, so lowering it for a smaller request would make a
    // concurrent larger launch of another host thread fail) and the grid size that is resident at once per (device, smem).
    struct Cfg {
        std::mutex mu;
        size_t limit[kMaxDevices] = {};
        struct Entry { int device; size_t smem; int resident; };
        std::vector<Entry> seen;
    };
    static Cfg cfg;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
    int resident = 0;
    {
        std::lock_guard<std::mutex> lk(cfg.mu);
        if (smem > cfg.limit[dev]) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            cfg.limit[dev] = smem;
        }
        for (const auto& s : cfg.seen)
            if (s.device == dev && s.smem == smem) resident = s.resident;
        if (resident == 0) {
            int per_sm = 0, sms = 0;
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, WARPS * 32, smem);
            if (e != cudaSuccess) return e;
            e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            if (e != cudaSuccess) return e;
            resident = (per_sm > 0 ? per_sm : 1) * sms;
            cfg.seen.push_back({dev, smem, resident});
        }
    }
    const long long tiles = (io.N + T - 1) / T;
    const long long want = (tiles + WARPS - 1) / WARPS;
    const unsigned blocks = (unsigned)(want < resident ? want : resident);
    auto al16 = [](const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    int aligned16 = al16(io.x) && al16(io.g) && al16(io.jac) && al16(io.grad) && (T % 2 == 0);
    if (Q)
        for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++)
            if (PT.off[a] >= 0) aligned16 = aligned16 && al16(Q->arr[a]);
    return launch_pdl(kern, blocks, WARPS * 32, smem, st, P, io, flags, aligned16, Q ? *Q : kNoInstParams, PT);
}

// Which per-instance arrays the instance-major kernel stages for the requested outputs, and where (CplbParamTile).
inline CplbParamTile make_param_tile(const CplbParams& P, const CplbInstParams* Q, unsigned flags, int T)
{
    CplbParamTile PT = {};
    for (int a = 0; a < CPLB_NUM_INST_ARRAYS; a++) {
        PT.off[a] = -1;
        PT.len[a] = cplb_inst_len(a, P.nc);
    }
    if (!Q) return PT;
    // Staged for constraint-only evaluations: what the constraint rows read (9 + nc doubles per instance; measured 55 -> 61 %
    // of the roofline at 65,536 x 4 contacts, 69 -> 75 % at 1,048,576).  With the cost or the gradient requested nothing is
    // staged and every array is read with read-only global loads as before: that variant is bound by the cost lane's
    // critical path and by resident warps, and both staging everything (39 %) and staging only the constraint arrays (32 %)
    // measured below the plain loads (43 %).
    // Ground problems only: without an environment the extra 1.5 KB per warp costs a resident CTA (59 vs 53 KB: 70 -> 62 % at
    // 1,048,576 x 4 contacts) and the Superquadric rows are bound by their arithmetic (48 vs 45 %, 51 vs 52 %).
    if (flags & (CPLB_WANT_COST | CPLB_WANT_GRAD)) return PT;
    if (P.env != CPLB_ENV_GROUND_K || !(flags & (CPLB_WANT_G | CPLB_WANT_J))) return PT;
    for (int a = 0; a < CPLB_IA_COM_REF; a++)
        if (Q->arr[a]) {
            PT.off[a] = PT.total;
            PT.total += T * PT.len[a];
        }
    return PT;
}

template <int ENV, int LPI>
cudaError_t launch_im_cfg(const CplbParams& P, const CplbIo& io, unsigned flags, const CplbInstParams* Q, cudaStream_t st)
{
    constexpr int T = 32 / LPI;
    const CplbParamTile PT = make_param_tile(P, Q, flags & 15u, T);
    const size_t per_warp = (tile_doubles(T, P.n, P.m, P.nnz, flags & 15u) + 2 * (size_t)PT.total) * sizeof(double) + 2 * sizeof(uint64_t);
    const unsigned gj = CPLB_WANT_G | CPLB_WANT_J;
    if (4 * per_warp <= 72 * 1024) {  // the common shapes: 4 warps per CTA, 3 CTAs per SM
        if (Q) return launch_im_kernel<ENV, LPI, 4, 0u, true>(P, io, flags, 4 * per_warp, Q, PT, st);
        if ((flags & 15u) == gj) return launch_im_kernel<ENV, LPI, 4, gj, false>(P, io, flags, 4 * per_warp, Q, PT, st);
        return launch_im_kernel<ENV, LPI, 4, 0u, false>(P, io, flags, 4 * per_warp, Q, PT, st);
    }
    if (per_warp > 227 * 1024) return cudaErrorInvalidConfiguration;
    if (Q) return launch_im_kernel<ENV, LPI, 1, 0u, true>(P, io, flags, per_warp, Q, PT, st);
    return launch_im_kernel<ENV, LPI, 1, 0u, false>(P, io, flags, per_warp, Q, PT, st);  // many contacts: one warp per CTA
}

}  // namespace cplb

#include "cplb_kernels_imc.cuh"

namespace cplb {

// im_kernel: CPLB_IM_AUTO (pick by shape), CPLB_IM_WARP_TILE (eval_instance_major: a warp per tile), CPLB_IM_CTA_TILE
// (eval_instance_major_cta: a CTA per tile, one warp per contact) -- cplb_set_instance_major_kernel; the parity tests force
// each of them on the same inputs.
template <int ENV>
cudaError_t launch_im_env(const CplbParams& P, const CplbIo& io, unsigned flags, const CplbInstParams* Q, int im_kernel, cudaStream_t st)
{
    // (measured, profiles/r02_variants.md: a Superquadric evaluation with any other output set than g + Jacobian -- the variant with
    // run-time output flags -- runs at 64-76 % of the roofline on the warp-tile kernel and at 47-53 % on the CTA-tile one)
    const bool sq_other_outputs = ENV == CPLB_ENV_SUPERQUADRIC_K && (flags & 15u) != (CPLB_WANT_G | CPLB_WANT_J);
    // (same table: with more than 8 contacts the CTA-tile kernel wins at 65,536 instances, 81 -> 85 %, and loses in long launches,
    // 96 -> 89 % at 1,048,576; warp-tile ahead from 131,072 on: 89.7 vs 87.6 %)
    const bool many_contacts_long = P.nc > 8 && io.N >= (1LL << 17);
    const bool cta_tile = im_kernel == CPLB_IM_CTA_TILE ||
                          (im_kernel == CPLB_IM_AUTO && instance_major_auto_is_cta_tile(P.nc) && !sq_other_outputs && !many_contacts_long) ||
                          (flags & (CPLB_JAC_PACKED_K | CPLB_JAC_COMPUTED_K));  // packed Jacobian slices exist in the CTA-tile kernel only
    if (cta_tile) return launch_imc_env<ENV>(P, io, flags, Q, st);
    // lanes per instance: the smallest power of two >= nc (capped at 8; more contacts loop)
    if (P.nc <= 1) return launch_im_cfg<ENV, 1>(P, io, flags, Q, st);
    if (P.nc <= 2) return launch_im_cfg<ENV, 2>(P, io, flags, Q, st);
    if (P.nc <= 4) return launch_im_cfg<ENV, 4>(P, io, flags, Q, st);
    return launch_im_cfg<ENV, 8>(P, io, flags, Q, st);
}

}  // namespace cplb
#endif
