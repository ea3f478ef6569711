// prep.cu -- the steps either side of the registration loop (SURVEY.md section 8f, ranks 1 and 2):
//   depth map -> camera-space points + central-difference normals + validity filter
//                                             PointCloud(float* depthMap, BYTE* colorFrame, ...)  PointCloud.h:78-165
//   per-iteration convergence metrics over known correspondences, evaluated on the device from the pose history
//                                             ConvergenceMeasure::rmseAlignmentError   ConvergenceMeasure.h:50-66
//                                             ConvergenceMeasure::benchmarkError       ConvergenceMeasure.h:104-151
// Both are HBM-bound streaming kernels: 4 B (depth) + 4 neighbour reads (cached) in, 28 B out per pixel; 24 B per
// correspondence and iteration.
#include "icp_internal.cuh"

#define PREP_THREADS 256

// ---------------------------------------------------------------------------- depth -> cloud
// One thread per candidate pixel i = k * downsample.  Writes the point, the normal and the colour of the candidate to
// slot k of the staging arrays and its keep flag; the kept candidates are then compacted in order (scan + scatter).
__global__ void __launch_bounds__(PREP_THREADS) depth_cloud_kernel(const float* __restrict__ depth, const unsigned char* __restrict__ color, DepthArgs a,
                                                                   float* __restrict__ pts, float* __restrict__ nrm, unsigned char* __restrict__ rgba,
                                                                   unsigned int* __restrict__ flag) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= a.n_candidates) return;
    const long long i = k * (long long)a.downsample;
    const int u = (int)(i % a.width), v = (int)(i / a.width);
    const float d = __ldg(&depth[i]);
    float px = MINF_F, py = MINF_F, pz = MINF_F;
    if (d != MINF_F) {
        // Back-projection (PointCloud.h:101-108): rotationInv * ((u - cX) / fovX * depth, (v - cY) / fovY * depth, depth) + translationInv
        const float cx = pmul(pdiv(psub((float)u, a.cX), a.fovX), d), cy = pmul(pdiv(psub((float)v, a.cY), a.fovY), d);
        xform_point(a.Einv, cx, cy, d, px, py, pz);
    }
    float nx = MINF_F, ny = MINF_F, nz = MINF_F;
    if (u >= 1 && v >= 1 && u < (int)a.width - 1 && v < (int)a.height - 1) {
        // PointCloud.h:116-131: central differences of the DEPTH map, normal (-du, -dv, 1) normalised
        const float du = pmul(0.5f, psub(__ldg(&depth[i + 1]), __ldg(&depth[i - 1])));
        const float dv = pmul(0.5f, psub(__ldg(&depth[i + a.width]), __ldg(&depth[i - a.width])));
        if (isfinite(du) && isfinite(dv) && !(fabsf(du) > a.half_max_distance) && !(fabsf(dv) > a.half_max_distance)) {
            const float ax = -du, ay = -dv;
            const float nn = __fsqrt_rn(padd(padd(pmul(ax, ax), pmul(ay, ay)), 1.0f));
            nx = pdiv(ax, nn); ny = pdiv(ay, nn); nz = pdiv(1.0f, nn);
        }
    }
    pts[3 * k] = px; pts[3 * k + 1] = py; pts[3 * k + 2] = pz;
    nrm[3 * k] = nx; nrm[3 * k + 1] = ny; nrm[3 * k + 2] = nz;
    // PointCloud.h:151-152 reads bytes colorFrame[i .. i+3] with the PIXEL index i (not 4*i): replicated
    unsigned int c = 0;
    if (color) c = (unsigned int)__ldg(&color[i]) | ((unsigned int)__ldg(&color[i + 1]) << 8) | ((unsigned int)__ldg(&color[i + 2]) << 16) | ((unsigned int)__ldg(&color[i + 3]) << 24);
    reinterpret_cast<unsigned int*>(rgba)[k] = c;
    flag[k] = (a.keep_original_size || (finite3(px, py, pz) && finite3(nx, ny, nz))) ? 1u : 0u;
}

// Order-preserving compaction of 0/1 flags: per-block counts, one-block scan of the counts, scatter.
__global__ void __launch_bounds__(PREP_THREADS) flag_count_kernel(const unsigned int* __restrict__ flag, long long n, unsigned int* __restrict__ block_count) {
    __shared__ unsigned int s_w[PREP_THREADS / 32];
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned int f = (k < n) ? flag[k] : 0u;
    const unsigned int b = __popc(__ballot_sync(0xFFFFFFFFu, f != 0u));
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = b;
    __syncthreads();
    if (threadIdx.x == 0) { unsigned int t = 0; for (int w = 0; w < PREP_THREADS / 32; ++w) t += s_w[w]; block_count[blockIdx.x] = t; }
}

__global__ void __launch_bounds__(1024) block_scan_kernel(unsigned int* __restrict__ block_count, int n_blocks, unsigned int* __restrict__ total) {
    // exclusive scan of n_blocks counts by one block, 1024 at a time (n_blocks is a few thousand at most)
    __shared__ unsigned int s[1024];
    __shared__ unsigned int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n_blocks; base += 1024) {
        const int j = base + (int)threadIdx.x;
        const unsigned int v = j < n_blocks ? block_count[j] : 0u;
        s[threadIdx.x] = v;
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            const unsigned int t = threadIdx.x >= (unsigned)off ? s[threadIdx.x - off] : 0u;
            __syncthreads();
            s[threadIdx.x] += t;
            __syncthreads();
        }
        if (j < n_blocks) block_count[j] = carry + s[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += s[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(PREP_THREADS) flag_scatter_kernel(const unsigned int* __restrict__ flag, long long n, const unsigned int* __restrict__ block_offset,
                                                                    const float* __restrict__ pts, const float* __restrict__ nrm, const unsigned char* __restrict__ rgba,
                                                                    float* __restrict__ pts_out, float* __restrict__ nrm_out, unsigned char* __restrict__ rgba_out) {
    __shared__ unsigned int s_w[PREP_THREADS / 32];
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool f = (k < n) && flag[k] != 0u;
    const unsigned int m = __ballot_sync(0xFFFFFFFFu, f);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) s_w[w] = __popc(m);
    __syncthreads();
    unsigned int before = block_offset[blockIdx.x];
    for (int j = 0; j < w; ++j) before += s_w[j];
    if (f) {
        const size_t o = before + __popc(m & ((1u << lane) - 1u));
        pts_out[3 * o] = pts[3 * k]; pts_out[3 * o + 1] = pts[3 * k + 1]; pts_out[3 * o + 2] = pts[3 * k + 2];
        nrm_out[3 * o] = nrm[3 * k]; nrm_out[3 * o + 1] = nrm[3 * k + 1]; nrm_out[3 * o + 2] = nrm[3 * k + 2];
        reinterpret_cast<unsigned int*>(rgba_out)[o] = reinterpret_cast<const unsigned int*>(rgba)[k];
    }
}

cudaError_t icp_launch_depth_cloud(const float* depth, const unsigned char* color, const DepthArgs& a, float* pts_tmp, float* nrm_tmp,
                                   unsigned char* rgba_tmp, unsigned int* flag, unsigned int* block_count, unsigned int* total,
                                   float* pts_out, float* nrm_out, unsigned char* rgba_out, cudaStream_t s, int* n_launches) {
    if (a.n_candidates <= 0) return cudaMemsetAsync(total, 0, 4, s);
    const int nb = (int)((a.n_candidates + PREP_THREADS - 1) / PREP_THREADS);
    depth_cloud_kernel<<<nb, PREP_THREADS, 0, s>>>(depth, color, a, pts_tmp, nrm_tmp, rgba_tmp, flag);
    flag_count_kernel<<<nb, PREP_THREADS, 0, s>>>(flag, a.n_candidates, block_count);
    block_scan_kernel<<<1, 1024, 0, s>>>(block_count, nb, total);
    flag_scatter_kernel<<<nb, PREP_THREADS, 0, s>>>(flag, a.n_candidates, block_count, pts_tmp, nrm_tmp, rgba_tmp, pts_out, nrm_out, rgba_out);
    if (n_launches) *n_launches += 4;
    return cudaGetLastError();
}

static_assert(PREP_THREADS == ICP_FLAG_SCAN_BLOCK, "the compaction's blocks are PREP_THREADS flags");
cudaError_t icp_launch_flag_scan(const unsigned int* flag, long long n, unsigned int* block_offset, unsigned int* total, cudaStream_t s, int* n_launches) {
    if (n <= 0) return cudaMemsetAsync(total, 0, 4, s);
    const int nb = (int)((n + PREP_THREADS - 1) / PREP_THREADS);
    flag_count_kernel<<<nb, PREP_THREADS, 0, s>>>(flag, n, block_offset);
    block_scan_kernel<<<1, 1024, 0, s>>>(block_offset, nb, total);
    if (n_launches) *n_launches += 2;
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- convergence metrics
// The correspondences reconstructRoom uses (main.cpp:300-307): every source point against itself under a ground-truth
// pose, gtTargetPoints = transformPoints(source.getPoints(), currentToZeroCoordinates), built from the resident source.
__global__ void __launch_bounds__(256) gt_from_source_kernel(const float4* __restrict__ src_raw, long long n, const float* __restrict__ pose16,
                                                             float* __restrict__ gt_src, float* __restrict__ gt_ref) {
    __shared__ float P[16];
    if (threadIdx.x < 16) P[threadIdx.x] = pose16[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = __ldg(&src_raw[i]);
    float x, y, z;
    xform_point(P, p.x, p.y, p.z, x, y, z);
    gt_src[3 * i] = p.x; gt_src[3 * i + 1] = p.y; gt_src[3 * i + 2] = p.z;
    gt_ref[3 * i] = x; gt_ref[3 * i + 1] = y; gt_ref[3 * i + 2] = z;
}
cudaError_t icp_launch_gt_from_source(const float4* src_raw, long long n, const float* pose16_dev, float* gt_src, float* gt_ref, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    gt_from_source_kernel<<<(unsigned int)((n + 255) / 256), 256, 0, s>>>(src_raw, n, pose16_dev, gt_src, gt_ref);
    return cudaGetLastError();
}

// grid (blocks, iterations).  partial[(it * blocks + b) * 6 + ..] = {sum |T s - u|^2, pairs, sum x, sum y, sum z, finite T s}
#define MET_THREADS 256
__device__ __forceinline__ double block_sum(double v, double* sm) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xFFFFFFFFu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0) for (int w = 0; w < MET_THREADS / 32; ++w) t += sm[w];
    return t;   // valid in thread 0
}

__global__ void __launch_bounds__(MET_THREADS) metrics_pass1_kernel(const float* __restrict__ src, const float* __restrict__ ref, long long m,
                                                                    const float* __restrict__ history, double* __restrict__ partial) {
    __shared__ float P[16];
    __shared__ double sm[MET_THREADS / 32];
    const int it = blockIdx.y;
    if (threadIdx.x < 16) P[threadIdx.x] = history[16 * it + threadIdx.x];
    __syncthreads();
    double sq = 0.0, cnt = 0.0, cx = 0.0, cy = 0.0, cz = 0.0, cn = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        float x, y, z;
        xform_point(P, src[3 * i], src[3 * i + 1], src[3 * i + 2], x, y, z);
        const float ux = ref[3 * i], uy = ref[3 * i + 1], uz = ref[3 * i + 2];
        if (finite3(x, y, z)) {
            cx += x; cy += y; cz += z; cn += 1.0;
            if (finite3(ux, uy, uz)) {
                const float dx = psub(x, ux), dy = psub(y, uy), dz = psub(z, uz);
                sq += (double)padd(padd(pmul(dx, dx), pmul(dy, dy)), pmul(dz, dz));
                cnt += 1.0;
            }
        }
    }
    double* out = partial + ((size_t)it * gridDim.x + blockIdx.x) * 6;
    double r;
    r = block_sum(sq, sm);  if (threadIdx.x == 0) out[0] = r;
    r = block_sum(cnt, sm); if (threadIdx.x == 0) out[1] = r;
    r = block_sum(cx, sm);  if (threadIdx.x == 0) out[2] = r;
    r = block_sum(cy, sm);  if (threadIdx.x == 0) out[3] = r;
    r = block_sum(cz, sm);  if (threadIdx.x == 0) out[4] = r;
    r = block_sum(cn, sm);  if (threadIdx.x == 0) out[5] = r;
}

// one thread per iteration: fixed-order sum of the block partials -> {rmse, centroid (fp32, as pcl::PointXYZ)}
__global__ void metrics_final1_kernel(const double* __restrict__ partial, int n_blocks, int n_iters, float* __restrict__ rmse, float* __restrict__ centroid) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= n_iters) return;
    double s[6] = {0, 0, 0, 0, 0, 0};
    for (int b = 0; b < n_blocks; ++b) for (int k = 0; k < 6; ++k) s[k] += partial[((size_t)it * n_blocks + b) * 6 + k];
    rmse[it] = sqrtf((float)(s[0] / s[1]));            // rmse /= counter; sqrt(rmse)  (ConvergenceMeasure.h:63-65)
    for (int k = 0; k < 3; ++k) centroid[3 * it + k] = s[5] > 0.0 ? (float)(s[2 + k] / s[5]) : 0.0f;
}

__global__ void __launch_bounds__(MET_THREADS) metrics_pass2_kernel(const float* __restrict__ src, const float* __restrict__ ref, long long m,
                                                                    const float* __restrict__ history, const float* __restrict__ centroid,
                                                                    double* __restrict__ partial) {
    __shared__ float P[16];
    __shared__ double sm[MET_THREADS / 32];
    const int it = blockIdx.y;
    if (threadIdx.x < 16) P[threadIdx.x] = history[16 * it + threadIdx.x];
    __syncthreads();
    const float c0 = centroid[3 * it], c1 = centroid[3 * it + 1], c2 = centroid[3 * it + 2];
    double err = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x) {
        float x, y, z;
        xform_point(P, src[3 * i], src[3 * i + 1], src[3 * i + 2], x, y, z);
        const float ex = psub(x, c0), ey = psub(y, c1), ez = psub(z, c2);
        const float dx = psub(x, ref[3 * i]), dy = psub(y, ref[3 * i + 1]), dz = psub(z, ref[3 * i + 2]);
        // pcl::euclideanDistance in fp32, the quotient and the sum in double (ConvergenceMeasure.h:143-145)
        const double cd = (double)__fsqrt_rn(padd(padd(pmul(ex, ex), pmul(ey, ey)), pmul(ez, ez)));
        err += (double)__fsqrt_rn(padd(padd(pmul(dx, dx), pmul(dy, dy)), pmul(dz, dz))) / cd;
    }
    const double r = block_sum(err, sm);
    if (threadIdx.x == 0) partial[(size_t)it * gridDim.x + blockIdx.x] = r;
}

__global__ void metrics_final2_kernel(const double* __restrict__ partial, int n_blocks, int n_iters, long long m, double* __restrict__ bench) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= n_iters) return;
    double s = 0.0;
    for (int b = 0; b < n_blocks; ++b) s += partial[(size_t)it * n_blocks + b];
    bench[it] = m > 0 ? s / (double)m : 0.0;
}

int icp_metrics_blocks(long long m, int n_sms) {
    long long nb = (m + MET_THREADS - 1) / MET_THREADS;
    if (nb > 2LL * n_sms) nb = 2LL * n_sms;
    return nb < 1 ? 1 : (int)nb;
}

cudaError_t icp_launch_metrics(const float* src, const float* ref, long long m, const float* history, int n_iters, int n_blocks, double* partial,
                               float* rmse, float* centroid, double* bench /* nullable */, cudaStream_t s, int* n_launches) {
    if (n_iters <= 0) return cudaSuccess;
    metrics_pass1_kernel<<<dim3(n_blocks, n_iters), MET_THREADS, 0, s>>>(src, ref, m, history, partial);
    metrics_final1_kernel<<<(n_iters + 63) / 64, 64, 0, s>>>(partial, n_blocks, n_iters, rmse, centroid);
    if (n_launches) *n_launches += 2;
    if (bench) {
        metrics_pass2_kernel<<<dim3(n_blocks, n_iters), MET_THREADS, 0, s>>>(src, ref, m, history, centroid, partial);
        metrics_final2_kernel<<<(n_iters + 63) / 64, 64, 0, s>>>(partial, n_blocks, n_iters, m, bench);
        if (n_launches) *n_launches += 2;
    }
    return cudaGetLastError();
}
