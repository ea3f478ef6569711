// lm.cu -- the Levenberg-Marquardt minimiser of CeresICPOptimizer on the device (the algebra and the trust-region loop: lm.cuh).
//
// One launch = one evaluation of all residual blocks at a parameter vector x: cost, J^T J and J^T r
// (29 doubles) are reduced across the grid and the block that finishes last advances the
// trust-region state machine in DevState (accept / reject, radius update, next candidate, or
// convergence -> pose update).  An outer ICP iteration is 1 + max_num_iterations such launches,
// enqueued back to back; launches that arrive after convergence return immediately.
#include "lm.cuh"

namespace {

__device__ void lm_finalize(DevState* st, int rc, float* history) {
    float inc[16];
    increment_matrix(st->lm.x, inc);
    apply_increment(st, inc, rc, history);
}

template <int METRIC>
__global__ void __launch_bounds__(ICP_REDUCE_THREADS) lm_eval_kernel(const ReduceArgs a, int step_index, int max_iterations) {
    __shared__ float P[16];
    __shared__ float Nm[9];
    __shared__ double xs[6];
    __shared__ double red[ICP_REDUCE_THREADS / 32][32];
    __shared__ double fin[ICP_REDUCE_THREADS / 32][32];
    __shared__ bool is_last;
    if (a.state->converged) return;                          // early stop reached in an earlier outer iteration
    if (step_index > 0 && a.state->lm.done) return;          // converged earlier in this outer iteration (uniform across the grid)
    if (threadIdx.x < 16) P[threadIdx.x] = a.state->pose[threadIdx.x];
    if (threadIdx.x >= 32 && threadIdx.x < 41) Nm[threadIdx.x - 32] = a.state->nrm[threadIdx.x - 32];
    if (threadIdx.x >= 64 && threadIdx.x < 70) xs[threadIdx.x - 64] = step_index == 0 ? 0.0 : a.state->lm.cand[threadIdx.x - 64];
    __syncthreads();
    double v[32];
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = 0.0;
    LmJets J;
    lm_jets_init<METRIC>(J, xs);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.n_src; i += gridDim.x * blockDim.x) {
        const int pos = a.match_pos[i];
        if (pos < 0) continue;
        const float4 sp = __ldg(&a.src_pts[i]);
        float sxf, syf, szf;
        xform_point(P, sp.x, sp.y, sp.z, sxf, syf, szf);
        const float4 tp = __ldg(&a.tgt_pts[pos]);
        if (!finite3(sxf, syf, szf) || !finite3(tp.x, tp.y, tp.z)) continue;        // ICPOptimizer.h:378
        lm_accumulate_match<METRIC>(v, J, sxf, syf, szf, tp, (double)a.match_w[i], Nm,
                                    [&] { return __ldg(&a.tgt_nrm[pos]); }, [&] { return __ldg(&a.src_nrm[i]); });
    }
    if (!grid_reduce_row<ICP_REDUCE_THREADS>(v, a.partials, &a.state->ticket, red, fin, &is_last, &a.peer, a.state)) return;
    if (threadIdx.x == 0) {
        const int rc = lm_advance(&a.state->lm, fin[0], step_index, max_iterations);
        if (rc != LM_NEXT_EVAL) lm_finalize(a.state, rc, a.pose_history);
    }
}

}  // namespace

cudaError_t icp_launch_lm(const ReduceArgs& a, int n_blocks, int lm_max_iterations, cudaStream_t s, int* n_launches) {
    for (int step = 0; step <= lm_max_iterations; ++step) {
        if (a.metric == ICP_GPU_METRIC_P2P) lm_eval_kernel<0><<<n_blocks, ICP_REDUCE_THREADS, 0, s>>>(a, step, lm_max_iterations);
        else if (a.metric == ICP_GPU_METRIC_P2PLANE) lm_eval_kernel<1><<<n_blocks, ICP_REDUCE_THREADS, 0, s>>>(a, step, lm_max_iterations);
        else lm_eval_kernel<2><<<n_blocks, ICP_REDUCE_THREADS, 0, s>>>(a, step, lm_max_iterations);
        if (n_launches) *n_launches += 1;
    }
    return cudaGetLastError();
}
