// standalone.cu -- the value-level operations of the reference's API that its drivers and tests call OUTSIDE estimatePose, on the
// device behind their own C-ABI entry points (the loop itself runs them fused, match.cu / knn.cu / solve.cu -- same device functions):
//   transformPoints / transformNormals           utils.h:106-133      icp_gpu_transform_points / _normals
//   WeightingMethod::applyWeights                weighting.h:39-99    icp_gpu_apply_weights
//   ProcrustesAligner::estimatePose and the two linear-system solvers of LinearICPOptimizer
//                                                ProcrustesAligner.h:6-29, ICPOptimizer.h:676-898    icp_gpu_solve_linear
#include "icp_internal.cuh"

struct Pose16 { float m[16]; };

__global__ void __launch_bounds__(256) transform_points_kernel(const float* __restrict__ in, long long n, const Pose16 P, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float x, y, z;
    xform_point(P.m, in[3 * i], in[3 * i + 1], in[3 * i + 2], x, y, z);
    out[3 * i] = x; out[3 * i + 1] = y; out[3 * i + 2] = z;
}

__global__ void __launch_bounds__(256) transform_normals_kernel(const float* __restrict__ in, long long n, const Pose16 P, float* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float N[9];
    inv_transpose3_pinned(P.m, N);                       // rotation.inverse().transpose(), utils.h:129
    float x, y, z;
    xform_normal(N, in[3 * i], in[3 * i + 1], in[3 * i + 2], x, y, z);
    out[3 * i] = x; out[3 * i + 1] = y; out[3 * i + 2] = z;
}

cudaError_t icp_launch_transform(const float* in, long long n, const float pose16[16], int normals, float* out, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    Pose16 P; for (int k = 0; k < 16; ++k) P.m[k] = pose16[k];
    const unsigned int nb = (unsigned int)((n + 255) / 256);
    if (normals) transform_normals_kernel<<<nb, 256, 0, s>>>(in, n, P, out);
    else transform_points_kernel<<<nb, 256, 0, s>>>(in, n, P, out);
    return cudaGetLastError();
}

// applyWeights: one thread per source point; matches[i].idx < 0 is left alone (weighting.h:52-53), CONSTANT_WEIGHTING returns at once (:44)
__global__ void __launch_bounds__(256) apply_weights_kernel(int method, float max_d2, const float* __restrict__ sp, const float* __restrict__ sn,
                                                            const unsigned int* __restrict__ sc, const float* __restrict__ tp,
                                                            const float* __restrict__ tn, const unsigned int* __restrict__ tc, long long n_tgt,
                                                            const int* __restrict__ idx, float* __restrict__ w, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const long long j = idx[i];
    if (j < 0 || j >= n_tgt) return;
    const float4 tp4 = make_float4(tp[3 * j], tp[3 * j + 1], tp[3 * j + 2], 0.f);
    const float4 tn4 = make_float4(tn ? tn[3 * j] : 0.f, tn ? tn[3 * j + 1] : 0.f, tn ? tn[3 * j + 2] : 0.f, __uint_as_float(tc ? tc[j] : 0u));
    float wi = w[i];
    match_weight_and_reject(method, 0, max_d2, sp[3 * i], sp[3 * i + 1], sp[3 * i + 2], sn ? sn[3 * i] : 0.f, sn ? sn[3 * i + 1] : 0.f,
                            sn ? sn[3 * i + 2] : 0.f, sc ? sc[i] : 0u, tp4, tn4, wi);
    w[i] = wi;
}

cudaError_t icp_launch_apply_weights(int method, float max_d2, const float* sp, const float* sn, const unsigned int* sc, const float* tp, const float* tn,
                                     const unsigned int* tc, long long n_tgt, const int* idx, float* w, long long n, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    apply_weights_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, s>>>(method, max_d2, sp, sn, sc, tp, tn, tc, n_tgt, idx, w, n);
    return cudaGetLastError();
}

// n matched pairs as the record arrays the reduction reads: pair i = (source i, target i), match_pos[i] = i
__global__ void __launch_bounds__(256) pack_pairs_kernel(const float* __restrict__ s, const float* __restrict__ sn, const float* __restrict__ t,
                                                         const float* __restrict__ tn, const float* __restrict__ w, int n, float4* __restrict__ sp4,
                                                         float4* __restrict__ sn4, float4* __restrict__ tp4, float4* __restrict__ tn4,
                                                         int* __restrict__ pos, float* __restrict__ wo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    sp4[i] = make_float4(s[3 * i], s[3 * i + 1], s[3 * i + 2], __int_as_float(i));
    sn4[i] = sn ? make_float4(sn[3 * i], sn[3 * i + 1], sn[3 * i + 2], 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    tp4[i] = make_float4(t[3 * i], t[3 * i + 1], t[3 * i + 2], __int_as_float(i));
    tn4[i] = tn ? make_float4(tn[3 * i], tn[3 * i + 1], tn[3 * i + 2], 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    pos[i] = i;
    wo[i] = w ? w[i] : 1.0f;
}

cudaError_t icp_launch_pack_pairs(const float* s, const float* sn, const float* t, const float* tn, const float* w, int n, float4* sp4, float4* sn4,
                                  float4* tp4, float4* tn4, int* pos, float* wo, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    pack_pairs_kernel<<<(n + 255) / 256, 256, 0, st>>>(s, sn, t, tn, w, n, sp4, sn4, tp4, tn4, pos, wo);
    return cudaGetLastError();
}
