// solve.cu -- stages 5-6 of one ICP iteration: residual / Jacobian assembly reduced straight to the
// normal equations (never materialising the reference's 4M x 6 matrix A), the 6x6 solve (or the 3x3
// Procrustes SVD), and the pose update, in ONE launch per iteration:
//   every block: per-thread fp64 accumulators -> recursive-halving warp reduce-scatter (62 shuffles
//   for 32 values) -> fixed-order block sum -> partial row in global memory;
//   last block (atomic ticket): fixed-order sum of all partial rows -> solve -> pose <- inc * pose.
// Deterministic: no floating-point atomics anywhere.
//
// Reference: gather (ICPOptimizer.h:583-610), estimatePosePointToPoint -> ProcrustesAligner
// (ICPOptimizer.h:666-674, ProcrustesAligner.h:6-70), estimatePosePointToPlane (:676-782),
// estimatePoseSymmetricICP (:784-898), pose accumulation (:614-620).
#include "icp_internal.cuh"
#include "solve.cuh"

struct PoseSmR { float P[16]; };

__device__ void finish_row(DevState* st, const double* row, int mode, float* history) {
    float inc[16]; int rc;
    if (mode == 0) rc = finish_p2p(row, inc);
    else if (mode == 1) rc = finish_p2plane(row, inc);
    else rc = finish_symmetric(row, st->mean_s, st->mean_d, inc);
    apply_increment(st, inc, rc, history);
}

// The same for the last block of reduce_kernel: the current pose and the means come from the block's shared-memory copies and
// the three loop counters from registers (loaded at kernel start), so the serial tail makes no dependent global-memory round
// trip; everything is written once at the end.
struct LoopRegs { int status, iters_done, iter; };

__device__ __forceinline__ void finish_row_local(DevState* st, const double* row, int mode, float* history, const float* P, const float* mS,
                                                 const float* mD, const LoopRegs lr) {
    float inc[16]; int rc;
    if (mode == 0) rc = finish_p2p(row, inc);
    else if (mode == 1) rc = finish_p2plane(row, inc);
    else rc = finish_symmetric(row, mS, mD, inc);
    if (lr.status == 0) {
        if (rc != 0) st->status = rc;
        else {
            float np[16], nm[9];
            mat4_mul_pinned(inc, P, np);                       // ICPOptimizer.h:614-620
            inv_transpose3_pinned(np, nm);
#pragma unroll
            for (int i = 0; i < 16; ++i) st->pose[i] = np[i];
#pragma unroll
            for (int i = 0; i < 9; ++i) st->nrm[i] = nm[i];
            if (history) {
#pragma unroll
                for (int i = 0; i < 16; ++i) history[16 * lr.iters_done + i] = np[i];
            }
            st->iters_done = lr.iters_done + 1;
            if (increment_is_small(inc, st->stop_rot, st->stop_trans)) st->converged = 1;
        }
    }
    st->iter = lr.iter + 1;
}

__device__ void finish_sums(DevState* st, const double* row) {
    // unweighted means of the kept matches, rounded to fp32 (ICPOptimizer.h:797-798)
    const double M = row[0];
    for (int k = 0; k < 3; ++k) {
        st->mean_s[k] = M > 0.0 ? (float)(row[1 + k] / M) : 0.f;
        st->mean_d[k] = M > 0.0 ? (float)(row[4 + k] / M) : 0.f;
    }
}

#ifdef ICP_TIMELINE   // diagnostic build (profiles/): see knn.cu; per block of iteration 12 {start, loop end}, [511] = {pose written, 0}
__device__ unsigned long long g_timeline_r[512][2];
__device__ __forceinline__ unsigned long long tlr_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
extern "C" int icp_gpu_debug_timeline_reduce(unsigned long long* out, int reset) {
    if (reset) { void* p = nullptr; cudaGetSymbolAddress(&p, g_timeline_r); return (int)cudaMemset(p, 0, sizeof(g_timeline_r)); }
    return (int)cudaMemcpyFromSymbol(out, g_timeline_r, sizeof(g_timeline_r));
}
#endif

// ---------------------------------------------------------------------------- the reduction kernel
// MODE 0 p2p moments, 1 point-to-plane, 2 symmetric (needs means in state), 3 sums only
template <int MODE, bool FUSED>
__global__ void __launch_bounds__(ICP_REDUCE_THREADS) reduce_kernel(const ReduceArgs a) {
    __shared__ float P[16];
    __shared__ float mS[3], mD[3], Nm[9];
    __shared__ double red[ICP_REDUCE_THREADS / 32][32];
    __shared__ double fin[ICP_REDUCE_THREADS / 32][32];
    __shared__ bool is_last;
    unsigned long long t_start = 0, t_loop = 0;
    if (a.state->converged) return;                          // early stop reached (uniform across the grid)
    if (a.profile && threadIdx.x == 0) { t_start = global_timer_ns(); if (blockIdx.x == 0) a.state->prof[0] = t_start; }
    // the first point's independent loads are requested before the pose / descriptor loads and the barrier
    const int stride = gridDim.x * blockDim.x;
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int pos_n = -1; float wf_n = 0.f;
    float4 sp_n = make_float4(0.f, 0.f, 0.f, 0.f), sn_n = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i < a.n_src) {
        pos_n = FUSED ? a.nn_pos[i] : a.match_pos[i];
        sp_n = __ldg(&a.src_pts[i]);
        if (FUSED || MODE == 2) sn_n = __ldg(&a.src_nrm[i]);
        if (!FUSED) wf_n = a.match_w[i];
    }
    const int state_iter = a.state->iter;
#ifdef ICP_TIMELINE
    const bool tl_on = state_iter == 12 && threadIdx.x == 0 && blockIdx.x < 511;
    if (tl_on) g_timeline_r[blockIdx.x][0] = tlr_now();
#endif
    LoopRegs lr; lr.status = 0; lr.iters_done = 0; lr.iter = state_iter;
    if (threadIdx.x == 0) { lr.status = a.state->status; lr.iters_done = a.state->iters_done; }
    if (threadIdx.x < 16) P[threadIdx.x] = a.state->pose[threadIdx.x];
    if (threadIdx.x >= 32 && threadIdx.x < 35) { mS[threadIdx.x - 32] = a.state->mean_s[threadIdx.x - 32]; mD[threadIdx.x - 32] = a.state->mean_d[threadIdx.x - 32]; }
    if (threadIdx.x >= 64 && threadIdx.x < 73) Nm[threadIdx.x - 64] = a.state->nrm[threadIdx.x - 64];
    __syncthreads();
    double v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = 0.0;
    // queries are addressed by their position in the Morton-sorted source
    IterDesc d; d.stride = 1; d.filter_finite = 0; d.mask_word_offset = -1; d.rng_key = 0u; d.proba = -1.0f;
    if (FUSED) d = a.desc[a.desc_index >= 0 ? a.desc_index : state_iter];
    // Software pipeline over the thread's points: the loads that depend on nothing (search result / match record,
    // source point and normal) are issued one point ahead, so the only latency a point exposes is its gather of the
    // matched target point -- the kernel is latency-bound (4 warps per scheduler at 128 registers), not HBM-bound.
    for (; i < a.n_src; i += stride) {
        const int pos = pos_n; float wf = wf_n; const float4 sp = sp_n, sn4 = sn_n;
        // a query without a (surviving) match has pos -1
        const bool gather = pos >= 0 && (!FUSED || pos < a.n_tgt);
        float4 tp = make_float4(0.f, 0.f, 0.f, 0.f), tn = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gather) {
            tp = __ldg(&a.tgt_pts[pos]);
            if (FUSED || MODE == 1 || MODE == 2) tn = __ldg(&a.tgt_nrm[pos]);
        }
        {
            const int i2 = i + stride;
            if (i2 < a.n_src) {
                pos_n = FUSED ? a.nn_pos[i2] : a.match_pos[i2];
                sp_n = __ldg(&a.src_pts[i2]);
                if (FUSED || MODE == 2) sn_n = __ldg(&a.src_nrm[i2]);
                if (!FUSED) wf_n = a.match_w[i2];
            }
        }
        if (!gather) continue;
        float sxf, syf, szf;
        if (FUSED) {
            // stages 3-4 evaluated here from the search result (same code path as match_finish_kernel)
            if (!query_active(d, a.mask, sp, sn4)) continue;
            xform_point(P, sp.x, sp.y, sp.z, sxf, syf, szf);
            if (!finite3(sxf, syf, szf)) continue;
            float nx, ny, nz;
            xform_normal(Nm, sn4.x, sn4.y, sn4.z, nx, ny, nz);
            wf = 1.0f;
            if (!match_weight_and_reject(a.weighting, a.rejection, a.weight_max_d2, sxf, syf, szf, nx, ny, nz, __float_as_uint(sn4.w), tp, tn, wf)) continue;
        } else {
            xform_point(P, sp.x, sp.y, sp.z, sxf, syf, szf);
        }
        if (!finite3(sxf, syf, szf) || !finite3(tp.x, tp.y, tp.z)) continue;        // ICPOptimizer.h:590-592
        accumulate_match<MODE>(v, sxf, syf, szf, tp, tn, sn4, Nm, mS, mD, (double)wf);
    }
    if (a.profile && threadIdx.x == 0) t_loop = global_timer_ns();
#ifdef ICP_TIMELINE
    if (tl_on) g_timeline_r[blockIdx.x][1] = tlr_now();
#endif
    if (!grid_reduce_row<ICP_REDUCE_THREADS>(v, a.partials, &a.state->ticket, red, fin, &is_last, a.solve ? &a.peer : nullptr, a.state)) return;
    if (threadIdx.x == 0) {
        if (a.profile) { a.state->prof[1] = t_start; a.state->prof[2] = t_loop; a.state->prof[3] = global_timer_ns(); }
        if (!a.solve) { for (int k = 0; k < ICP_NRED; ++k) a.state->shard_partials[k] = fin[0][k]; }
        else if (MODE == 3) finish_sums(a.state, fin[0]);
        else finish_row_local(a.state, fin[0], MODE, a.pose_history, P, mS, mD, lr);
        if (a.profile) { __threadfence(); a.state->prof[4] = global_timer_ns(); }
#ifdef ICP_TIMELINE
        if (state_iter == 12) g_timeline_r[511][0] = tlr_now();
#endif
    }
}

// Blocks of reduce_kernel per SM: 1 / 4 measured 6.46 / 6.36 ms per registration, both slower than 2 (round 1, profiles/README.md);
// 3 do not fit the registers (DESIGN §4).
#define REDUCE_BLOCKS_PER_SM 2

int icp_reduce_blocks(int n_src, int n_sms) {
    int nb = (n_src + ICP_REDUCE_THREADS - 1) / ICP_REDUCE_THREADS;
    if (nb > REDUCE_BLOCKS_PER_SM * n_sms) nb = REDUCE_BLOCKS_PER_SM * n_sms;
    if (nb < 1) nb = 1;
    return nb;
}

template <int MODE>
static void launch_reduce_mode(const ReduceArgs& a, int n_blocks, cudaStream_t s) {
    if (a.fused) reduce_kernel<MODE, true><<<n_blocks, ICP_REDUCE_THREADS, 0, s>>>(a);
    else reduce_kernel<MODE, false><<<n_blocks, ICP_REDUCE_THREADS, 0, s>>>(a);
}

cudaError_t icp_launch_reduce(const ReduceArgs& a, int n_blocks, cudaStream_t s, int* n_launches) {
    int launches = 0;
    if (a.metric == ICP_GPU_METRIC_P2P) { launch_reduce_mode<0>(a, n_blocks, s); ++launches; }
    else if (a.metric == ICP_GPU_METRIC_P2PLANE) { launch_reduce_mode<1>(a, n_blocks, s); ++launches; }
    else {
        launch_reduce_mode<3>(a, n_blocks, s); ++launches;
        launch_reduce_mode<2>(a, n_blocks, s); ++launches;
    }
    if (n_launches) *n_launches += launches;
    return cudaGetLastError();
}

cudaError_t icp_launch_reduce_phase(const ReduceArgs& a, int n_blocks, int phase, cudaStream_t s, int* n_launches) {
    if (a.metric == ICP_GPU_METRIC_P2P) launch_reduce_mode<0>(a, n_blocks, s);
    else if (a.metric == ICP_GPU_METRIC_P2PLANE) launch_reduce_mode<1>(a, n_blocks, s);
    else if (phase == 0) launch_reduce_mode<3>(a, n_blocks, s);
    else launch_reduce_mode<2>(a, n_blocks, s);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- pose upload / shard apply
__global__ void pose_init_kernel(DevState* st, const float* pose16, float stop_rot, float stop_trans) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    for (int i = 0; i < 16; ++i) st->pose[i] = pose16[i];
    inv_transpose3_pinned(st->pose, st->nrm);
    st->iter = 0; st->iters_done = 0; st->status = 0; st->ticket = 0; st->ticket2 = 0;
    st->n_queries = 0; st->n_matched = 0; st->n_evals = 0; st->n_nodes = 0;
    for (int k = 0; k < 3; ++k) { st->mean_s[k] = 0.f; st->mean_d[k] = 0.f; }
    st->lm.done = 0; st->lm.iter = 0;
    st->stop_rot = stop_rot; st->stop_trans = stop_trans; st->converged = 0;
}

cudaError_t icp_launch_pose_init(DevState* st, const float* pose_dev16, cudaStream_t s, float stop_rot, float stop_trans) {
    pose_init_kernel<<<1, 32, 0, s>>>(st, pose_dev16, stop_rot, stop_trans);
    return cudaGetLastError();
}

__global__ void shard_apply_kernel(DevState* st, int mode, float* history) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    if (mode == 3) finish_sums(st, st->shard_partials);
    else finish_row(st, st->shard_partials, mode, history);
}

cudaError_t icp_launch_shard_apply(DevState* st, int mode, float* history, cudaStream_t s) {
    shard_apply_kernel<<<1, 32, 0, s>>>(st, mode, history);
    return cudaGetLastError();
}
