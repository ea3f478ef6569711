// batch.cu -- B independent registrations of small pairs in ONE launch per (minimiser, metric): thread block k owns pair pairs[k]
// and runs every iteration of its loop (selection, transform, exact 1-NN, weighting, rejection, the minimiser, pose update)
// without returning to the host.  No index build, no graph, no per-iteration launch: for a pair of a few thousand points the
// single-pair path's time is launch and dependency latency, not work (DESIGN.md section 4).  Every pair reads its own
// configuration (BatchCfg) and iteration schedule (icp_schedule).
//
//   staging   the pair's target points (float4, D1 layout) in dynamic shared memory, once; normals stay in global memory
//             and are read for the matched point only
//   selection the query set of iteration `it` exactly as make_plan (registration.cu) describes it: the level stride of the multi-resolution
//             schedule with its finite filter, the mt19937 mask drawn on the host, or the device selection stream keyed by the seed
//             and the iteration; masks and hash are indexed by the pair-local source index
//   search    one thread per query, every thread scans the staged target in index order: all lanes read the same entry
//             (a shared-memory broadcast).  D1 distances, strict '<' in index order = the lowest index of equal distances
//             (D2), valid iff d2 <= max_distance_sq (D3): the same correspondences as knn_brute_kernel and the oracle's scan
//   stages 3-4 query_active, xform_point / xform_normal, match_weight_and_reject: the device functions the other paths use
//   linear    (batch_icp_kernel) accumulate_match (solve.cuh, shared with reduce_kernel) into per-thread fp64 rows, warp
//             reduce-scatter, then a fixed-order sum over the warps (deterministic, no floating-point atomics); thread 0 solves
//             with the finishers of solve.cuh and updates the pose in fp32 (ICPOptimizer.h:614-620)
//   LM        (batch_lm_kernel) the matches go to the pair's scratch slice; then the trust-region loop of lm.cuh (shared with
//             lm_eval_kernel): the evaluation at x = 0 and up to lm_max_iterations candidate evaluations, each one block pass over
//             the matches summed in the same fixed order, thread 0 advancing the state machine between passes
// The symmetric metric needs the matched means before its rows: the first pass keeps every query's match in a per-pair
// slice of global scratch and the second pass reads it back instead of searching again.
// A pair stops on its own: early stop (increment_is_small), no surviving match (ICP_GPU_E_NO_MATCHES) or a singular
// system (ICP_GPU_E_NUMERIC); a failed pair keeps its last good pose.
#include "solve.cuh"
#include "lm.cuh"
#include "search.cuh"

static_assert(ICP_BATCH_THREADS % 32 == 0 && ICP_BATCH_THREADS <= 1024 && ICP_BATCH_LM_THREADS % 32 == 0, "whole warps");

__device__ __forceinline__ float4 load_packed3(const float* __restrict__ p, long long i, float w) {
    return make_float4(__ldg(&p[3 * i]), __ldg(&p[3 * i + 1]), __ldg(&p[3 * i + 2]), w);
}

// Index of the nearest staged target point to q, or -1.  `bound` is the smallest float above the threshold, so that strict '<'
// admits d2 == threshold and, scanning in index order, keeps the first (lowest) index of equal distances: the (d2, index)
// arg-min of knn_brute_kernel (whose start value is fminf(max_d2, FLT_BIG) with index INT_MAX).
__device__ __forceinline__ int nearest_staged(const float4* __restrict__ tgt, int n_t, float qx, float qy, float qz, float bound) {
    float bd = bound; int bj = -1;
#pragma unroll 4
    for (int j = 0; j < n_t; ++j) {
        const float d = dist3(qx, qy, qz, tgt[j]);
        if (d < bd) { bd = d; bj = j; }
    }
    return bj;
}

// Fixed-order block sum of one 32-double row per thread; the total ends in fin[0..31] for every thread.
template <int THREADS>
__device__ __forceinline__ void block_sum_row(double (&v)[32], double (*red)[32], double* fin) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    warp_reduce_scatter32(v, lane);
    red[wid][lane] = v[0];
    __syncthreads();
    if (threadIdx.x < 32) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < THREADS / 32; ++w) s += red[w][threadIdx.x];
        fin[threadIdx.x] = s;
    }
    __syncthreads();
}

// Staging common to both kernels: the pair's configuration, pose, its inverse-transpose and target, in shared memory.
struct BatchPair {
    int b, n_s, n_t;
    long long s0, t0;
    const float* src_xyz; const float* src_nrm; const float* tgt_nrm;
    const unsigned int* mask;    // mt19937 masks of the pair, or null
    int mask_words;
};

__device__ __forceinline__ BatchPair batch_stage(const BatchArgs& a, BatchCfg& c, float4* tgt_sm, float* P, float* Nm) {
    BatchPair q;
    q.b = a.pairs[blockIdx.x];
    q.s0 = a.src_off[q.b]; q.t0 = a.tgt_off[q.b];
    q.n_s = (int)(a.src_off[q.b + 1] - q.s0); q.n_t = (int)(a.tgt_off[q.b + 1] - q.t0);
    q.tgt_nrm = a.tgt_nrm ? a.tgt_nrm + 3 * q.t0 : nullptr;
    q.src_nrm = a.src_nrm ? a.src_nrm + 3 * q.s0 : nullptr;
    q.src_xyz = a.src_xyz + 3 * q.s0;
    q.mask_words = ((q.n_s > 0 ? q.n_s : 1) + 31) / 32;
    for (int j = threadIdx.x; j < q.n_t; j += blockDim.x) tgt_sm[j] = load_packed3(a.tgt_xyz + 3 * q.t0, j, 0.f);
    if (threadIdx.x < 16) P[threadIdx.x] = a.poses_in[16 * (size_t)q.b + threadIdx.x];
    if (threadIdx.x == 0) c = a.cfgs[a.cfg_index[q.b]];
    __syncthreads();
    q.mask = c.mt_mask ? a.mask + a.mask_off[q.b] : nullptr;
    if (threadIdx.x == 0) inv_transpose3_pinned(P, Nm);
    return q;
}

// The query set of iteration `it` (make_plan, registration.cu): the level stride and finite filter of the multi-resolution schedule, the
// mt19937 mask or the device selection stream (keyed by the seed and the iteration)
__device__ __forceinline__ IterDesc batch_iter_desc(const BatchCfg& c, const IcpSchedule& sch, int it, int mask_words) {
    IterDesc d;
    d.stride = icp_schedule_stride(sch, it); d.filter_finite = c.multires; d.mask_word_offset = c.mt_mask ? it * mask_words : -1;
    d.proba = c.proba; d.rng_key = c.seed * 2654435761u + (unsigned int)(it + 1) * 0x9E3779B9u;
    d.pad0 = d.pad1 = d.pad2 = 0;
    return d;
}

// Matching of source point i at pose P (stages 2-4): the staged target index or -1, the match weight in w, the transformed point
// in (sx, sy, sz), the target point and normal in tp / tn.
__device__ __forceinline__ int batch_match(const BatchCfg& c, const BatchPair& q, const IterDesc& d, const float4* tgt_sm, const float* P,
                                           const float* Nm, float bound, int i, float& sx, float& sy, float& sz, float4& tp, float4& tn, float& w) {
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 sp = load_packed3(q.src_xyz, i, __int_as_float(i));
    const float4 sn = q.src_nrm ? load_packed3(q.src_nrm, i, 0.f) : zero4;
    int j = -1;
    if (query_active(d, q.mask, sp, sn)) {
        xform_point(P, sp.x, sp.y, sp.z, sx, sy, sz);
        if (finite3(sx, sy, sz)) j = nearest_staged(tgt_sm, q.n_t, sx, sy, sz, bound);
        if (j >= 0) {
            tp = tgt_sm[j];
            if (q.tgt_nrm) tn = load_packed3(q.tgt_nrm, j, 0.f);
            float nx, ny, nz;
            xform_normal(Nm, sn.x, sn.y, sn.z, nx, ny, nz);
            w = 1.0f;
            if (!match_weight_and_reject(c.weighting, c.rejection, c.weight_max_d2, sx, sy, sz, nx, ny, nz, 0u, tp, tn, w)) j = -1;
            else if (!finite3(tp.x, tp.y, tp.z)) j = -1;                       // ICPOptimizer.h:590-592
        }
    }
    return j;
}

// METRIC 0 point-to-point, 1 point-to-plane, 2 symmetric
template <int METRIC>
__global__ void __launch_bounds__(ICP_BATCH_THREADS, 1) batch_icp_kernel(const BatchArgs a) {
    extern __shared__ float4 tgt_sm[];
    __shared__ float P[16], Nm[9], mS[3], mD[3];
    __shared__ double red[ICP_BATCH_THREADS / 32][32];
    __shared__ double fin[32];
    __shared__ int s_done;
    __shared__ BatchCfg c;
    if (threadIdx.x < 3) { mS[threadIdx.x] = 0.f; mD[threadIdx.x] = 0.f; }
    if (threadIdx.x == 0) s_done = 0;
    const BatchPair q = batch_stage(a, c, tgt_sm, P, Nm);
    const int b = q.b, n_s = q.n_s;
    const long long s0 = q.s0;
    __syncthreads();
    const IcpSchedule sch = icp_schedule(c.n_iterations, c.multires, n_s);
    const float bound = nextafterf(fminf(c.max_d2, FLT_BIG), INFINITY);
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    int status = 0, iters_done = 0;                       // meaningful in thread 0
    for (int it = 0; it < sch.n_iters; ++it) {
        const IterDesc d = batch_iter_desc(c, sch, it, q.mask_words);
        double v[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = 0.0;
        for (int i = threadIdx.x; i < n_s; i += blockDim.x) {
            float w = 0.0f, sx = 0.f, sy = 0.f, sz = 0.f;
            float4 tp = zero4, tn = zero4;
            const int j = batch_match(c, q, d, tgt_sm, P, Nm, bound, i, sx, sy, sz, tp, tn, w);
            if (METRIC == 2) a.scratch[s0 + i] = make_int2(j, __float_as_int(w));
            if (j < 0) continue;
            const float4 sn = q.src_nrm ? load_packed3(q.src_nrm, i, 0.f) : zero4;
            accumulate_match<METRIC == 2 ? 3 : METRIC>(v, sx, sy, sz, tp, tn, sn, Nm, mS, mD, (double)w);
        }
        block_sum_row<ICP_BATCH_THREADS>(v, red, fin);
        if (METRIC == 2) {
            if (threadIdx.x == 0) {                        // unweighted means of the kept matches, rounded to fp32 (finish_sums, solve.cu)
                const double M = fin[0];
                for (int k = 0; k < 3; ++k) { mS[k] = M > 0.0 ? (float)(fin[1 + k] / M) : 0.f; mD[k] = M > 0.0 ? (float)(fin[4 + k] / M) : 0.f; }
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 32; ++k) v[k] = 0.0;
            for (int i = threadIdx.x; i < n_s; i += blockDim.x) {
                const int2 m = a.scratch[s0 + i];          // written by this thread in the first pass
                if (m.x < 0) continue;
                const float4 sp = load_packed3(q.src_xyz, i, 0.f);
                const float4 sn = q.src_nrm ? load_packed3(q.src_nrm, i, 0.f) : zero4;
                const float4 tn = q.tgt_nrm ? load_packed3(q.tgt_nrm, m.x, 0.f) : zero4;
                float sx, sy, sz;
                xform_point(P, sp.x, sp.y, sp.z, sx, sy, sz);
                accumulate_match<2>(v, sx, sy, sz, tgt_sm[m.x], tn, sn, Nm, mS, mD, (double)__int_as_float(m.y));
            }
            block_sum_row<ICP_BATCH_THREADS>(v, red, fin);
        }
        if (threadIdx.x == 0) {
            float inc[16]; int rc;
            if (METRIC == 0) rc = finish_p2p(fin, inc);
            else if (METRIC == 1) rc = finish_p2plane(fin, inc);
            else rc = finish_symmetric(fin, mS, mD, inc);
            if (rc != 0) { status = rc; s_done = 1; }
            else {
                float np[16];
                mat4_mul_pinned(inc, P, np);               // ICPOptimizer.h:614-620
                for (int k = 0; k < 16; ++k) P[k] = np[k];
                inv_transpose3_pinned(np, Nm);
                if (a.history) for (int k = 0; k < 16; ++k) a.history[((size_t)b * a.history_rows + iters_done) * 16 + k] = np[k];
                ++iters_done;
                if (increment_is_small(inc, c.stop_rot, c.stop_trans)) s_done = 1;
            }
        }
        __syncthreads();
        if (s_done) break;
    }
    if (threadIdx.x < 16) a.poses_out[16 * (size_t)b + threadIdx.x] = P[threadIdx.x];
    if (threadIdx.x == 0) { a.n_iter_out[b] = iters_done; a.status_out[b] = status; }
}

// The Ceres path (CeresICPOptimizer, lm.cu) for one pair per block: the matches of an outer iteration go to the pair's scratch
// slice, then every evaluation of the trust-region loop is one block pass over them.
template <int METRIC>
__global__ void __launch_bounds__(ICP_BATCH_LM_THREADS, 1) batch_lm_kernel(const BatchArgs a) {
    extern __shared__ float4 tgt_sm[];
    __shared__ float P[16], Nm[9];
    __shared__ double red[ICP_BATCH_LM_THREADS / 32][32];
    __shared__ double fin[32];
    __shared__ double xs[6];
    __shared__ LmState lm;
    __shared__ int s_done, s_rc;
    __shared__ BatchCfg c;
    if (threadIdx.x == 0) s_done = 0;
    const BatchPair q = batch_stage(a, c, tgt_sm, P, Nm);
    const int b = q.b, n_s = q.n_s;
    const long long s0 = q.s0;
    __syncthreads();
    const IcpSchedule sch = icp_schedule(c.n_iterations, c.multires, n_s);
    const float bound = nextafterf(fminf(c.max_d2, FLT_BIG), INFINITY);
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    int status = 0, iters_done = 0;                       // meaningful in thread 0
    for (int it = 0; it < sch.n_iters; ++it) {
        const IterDesc d = batch_iter_desc(c, sch, it, q.mask_words);
        for (int i = threadIdx.x; i < n_s; i += blockDim.x) {
            float w = 0.0f, sx, sy, sz;
            float4 tp = zero4, tn = zero4;
            const int j = batch_match(c, q, d, tgt_sm, P, Nm, bound, i, sx, sy, sz, tp, tn, w);
            a.scratch[s0 + i] = make_int2(j, __float_as_int(w));     // kept matches: both points finite (ICPOptimizer.h:378)
        }
        for (int step = 0; step <= c.lm_max_iterations; ++step) {
            if (threadIdx.x < 6) xs[threadIdx.x] = step == 0 ? 0.0 : lm.cand[threadIdx.x];
            __syncthreads();
            double v[32];
#pragma unroll
            for (int k = 0; k < 32; ++k) v[k] = 0.0;
            LmJets J;
            lm_jets_init<METRIC>(J, xs);
            for (int i = threadIdx.x; i < n_s; i += blockDim.x) {
                const int2 m = a.scratch[s0 + i];          // written by this thread above
                if (m.x < 0) continue;
                const float4 sp = load_packed3(q.src_xyz, i, 0.f);
                float sx, sy, sz;
                xform_point(P, sp.x, sp.y, sp.z, sx, sy, sz);
                lm_accumulate_match<METRIC>(v, J, sx, sy, sz, tgt_sm[m.x], (double)__int_as_float(m.y), Nm,
                                            [&] { return q.tgt_nrm ? load_packed3(q.tgt_nrm, m.x, 0.f) : zero4; },
                                            [&] { return q.src_nrm ? load_packed3(q.src_nrm, i, 0.f) : zero4; });
            }
            block_sum_row<ICP_BATCH_LM_THREADS>(v, red, fin);
            if (threadIdx.x == 0) s_rc = lm_advance(&lm, fin, step, c.lm_max_iterations);
            __syncthreads();
            if (s_rc != LM_NEXT_EVAL) break;
        }
        if (threadIdx.x == 0) {                            // lm_finalize / apply_increment (lm.cu, icp_internal.cuh)
            float inc[16];
            increment_matrix(lm.x, inc);
            if (s_rc != 0) { status = s_rc; s_done = 1; }
            else {
                float np[16];
                mat4_mul_pinned(inc, P, np);               // ICPOptimizer.h:614-620
                for (int k = 0; k < 16; ++k) P[k] = np[k];
                inv_transpose3_pinned(np, Nm);
                if (a.history) for (int k = 0; k < 16; ++k) a.history[((size_t)b * a.history_rows + iters_done) * 16 + k] = np[k];
                ++iters_done;
                if (increment_is_small(inc, c.stop_rot, c.stop_trans)) s_done = 1;
            }
        }
        __syncthreads();
        if (s_done) break;
    }
    if (threadIdx.x < 16) a.poses_out[16 * (size_t)b + threadIdx.x] = P[threadIdx.x];
    if (threadIdx.x == 0) { a.n_iter_out[b] = iters_done; a.status_out[b] = status; }
}

cudaError_t icp_launch_batch(const BatchArgs& a, int metric, int lm, int n_pairs, int max_tgt, cudaStream_t s) {
    if (n_pairs <= 0) return cudaSuccess;
    void (*k)(const BatchArgs);
    if (lm) k = metric == ICP_GPU_METRIC_P2P ? batch_lm_kernel<0> : metric == ICP_GPU_METRIC_P2PLANE ? batch_lm_kernel<1> : batch_lm_kernel<2>;
    else k = metric == ICP_GPU_METRIC_P2P ? batch_icp_kernel<0> : metric == ICP_GPU_METRIC_P2PLANE ? batch_icp_kernel<1> : batch_icp_kernel<2>;
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ICP_BATCH_MAX_TARGET * sizeof(float4)));
    if (e != cudaSuccess) return e;
    const size_t smem = (size_t)(max_tgt > 0 ? max_tgt : 1) * sizeof(float4);
    k<<<n_pairs, lm ? ICP_BATCH_LM_THREADS : ICP_BATCH_THREADS, smem, s>>>(a);
    return cudaGetLastError();
}
