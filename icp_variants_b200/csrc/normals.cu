// normals.cu -- k-NN PCA normals of the indexed (target) cloud: PointCloud(pcl::PointCloud<pcl::PointXYZ>::Ptr)
// (PointCloud.h:41-76), i.e. pcl::NormalEstimation with setKSearch(5) and the viewpoint at the origin.  PCL is an
// un-vendored dependency of the reference; the algorithm is restated from PCL's published one (features/normal_3d.h)
// exactly as oracle/icp_oracle.c:orc_pca_normals states it: the k nearest neighbours of every point (itself included;
// exact, (d2, original index) order under contract D1), the covariance of the neighbourhood about its mean in double,
// the eigenvector of the smallest eigenvalue (cyclic Jacobi), flipped towards the viewpoint.
//
// One thread per point of the cell-sorted cloud (the 32 points of a warp are spatial neighbours).  The k-best list lives
// in registers.  The point's own leaf is scanned first; if the ball of the k-th distance lies inside the leaf's inflated
// box, only the leaves of its adjacency list (grid.cu) can hold closer points; otherwise the thread walks the BVH with a
// private stack.  This file is compiled with -fmad=false: the double arithmetic below is the oracle's, operation for
// operation, so the normals agree bit for bit.
#include "icp_internal.cuh"
#include <limits.h>

#define NRM_KMAX 8
#define NRM_STACK (32 * ICP_BVH_MAX_LEVELS)
#define FLT_BIG 3.4028234e38f

struct KBest { float d[NRM_KMAX]; int idx[NRM_KMAX]; int pos[NRM_KMAX]; int m; };

__device__ __forceinline__ float nrm_box_dist2(float qx, float qy, float qz, const float4 lo, const float4 hi) {
    const float gx = fmaxf(fmaxf(psub(lo.x, qx), psub(qx, hi.x)), 0.0f);
    const float gy = fmaxf(fmaxf(psub(lo.y, qy), psub(qy, hi.y)), 0.0f);
    const float gz = fmaxf(fmaxf(psub(lo.z, qz), psub(qz, hi.z)), 0.0f);
    return padd(padd(pmul(gx, gx), pmul(gy, gy)), pmul(gz, gz));
}

// the distance a candidate has to beat: the k-th best so far, or "anything" while the list is not full
__device__ __forceinline__ float kth(const KBest& b, int k) { return b.m < k ? FLT_BIG : b.d[k - 1]; }

__device__ __forceinline__ void kbest_insert(KBest& b, int k, float d, int idx, int pos) {
    // ascending (d, idx); a candidate enters if the list is not full or it precedes the last entry
    if (b.m == k && !(d < b.d[k - 1] || (d == b.d[k - 1] && idx < b.idx[k - 1]))) return;
    int at = b.m < k ? b.m : k - 1;
#pragma unroll
    for (int s = NRM_KMAX - 1; s > 0; --s) {
        if (s <= at && (d < b.d[s - 1] || (d == b.d[s - 1] && idx < b.idx[s - 1]))) { b.d[s] = b.d[s - 1]; b.idx[s] = b.idx[s - 1]; b.pos[s] = b.pos[s - 1]; at = s - 1; }
    }
#pragma unroll
    for (int s = 0; s < NRM_KMAX; ++s) if (s == at) { b.d[s] = d; b.idx[s] = idx; b.pos[s] = pos; }
    if (b.m < k) ++b.m;
}

__device__ __forceinline__ void nrm_scan_leaf(const float4* __restrict__ pts, const unsigned int* __restrict__ leaf_start, unsigned int leaf,
                                              float qx, float qy, float qz, KBest& b, int k) {
    const unsigned int ls = __ldg(&leaf_start[leaf]), le = __ldg(&leaf_start[leaf + 1]);
    for (unsigned int i = ls; i < le; ++i) {
        const float4 p = __ldg(&pts[i]);
        const float dx = psub(qx, p.x), dy = psub(qy, p.y), dz = psub(qz, p.z);
        const float d = padd(padd(pmul(dx, dx), pmul(dy, dy)), pmul(dz, dz));      // D1
        if (!isfinite(d)) continue;
        kbest_insert(b, k, d, __float_as_int(p.w), (int)i);
    }
}

// cyclic Jacobi, identical to oracle/icp_oracle.c:orc_eig3
__device__ void nrm_eig3(double* A, double* V, double* evals) {
#pragma unroll
    for (int i = 0; i < 9; ++i) V[i] = (i % 4 == 0) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 64; ++sweep) {
        const double off = (fabs(A[1]) + fabs(A[2])) + fabs(A[5]);
        if (off < 1e-300) break;
        for (int p = 0; p < 2; ++p) for (int q = p + 1; q < 3; ++q) {
            const double apq = A[p * 3 + q];
            if (apq == 0.0) continue;
            const double theta = (A[q * 3 + q] - A[p * 3 + p]) / (2.0 * apq);
            const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
            for (int k = 0; k < 3; ++k) { const double akp = A[k * 3 + p], akq = A[k * 3 + q]; A[k * 3 + p] = c * akp - s * akq; A[k * 3 + q] = s * akp + c * akq; }
            for (int k = 0; k < 3; ++k) { const double apk = A[p * 3 + k], aqk = A[q * 3 + k]; A[p * 3 + k] = c * apk - s * aqk; A[q * 3 + k] = s * apk + c * aqk; }
            for (int k = 0; k < 3; ++k) { const double vkp = V[k * 3 + p], vkq = V[k * 3 + q]; V[k * 3 + p] = c * vkp - s * vkq; V[k * 3 + q] = s * vkp + c * vkq; }
        }
    }
    int ord[3] = {0, 1, 2};
    for (int i = 0; i < 2; ++i) for (int j = 0; j < 2 - i; ++j) if (A[ord[j + 1] * 4] < A[ord[j] * 4]) { const int t = ord[j]; ord[j] = ord[j + 1]; ord[j + 1] = t; }
    double Vs[9];
    for (int k = 0; k < 3; ++k) { evals[k] = A[ord[k] * 4]; for (int i = 0; i < 3; ++i) Vs[i * 3 + k] = V[i * 3 + ord[k]]; }
    for (int i = 0; i < 9; ++i) V[i] = Vs[i];
}

__global__ void __launch_bounds__(128) pca_normals_kernel(const NormalArgs a) {
    __shared__ BvhDesc s_bvh;
    if (threadIdx.x < sizeof(BvhDesc) / 4) reinterpret_cast<int*>(&s_bvh)[threadIdx.x] = reinterpret_cast<const int*>(a.bvh)[threadIdx.x];
    __syncthreads();
    const BvhDesc& bvh = s_bvh;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.n) return;
    const float4 q4 = __ldg(&a.pts[p]);
    const int orig = __float_as_int(q4.w);
    const float nanv = __int_as_float(0x7fc00000);
    float nx = nanv, ny = nanv, nz = nanv, curv = nanv;
    const float qx = q4.x, qy = q4.y, qz = q4.z;
    const int k = a.k;
    if (finite3(qx, qy, qz) && bvh.n_leaves > 0) {
        KBest b; b.m = 0;
#pragma unroll
        for (int s = 0; s < NRM_KMAX; ++s) { b.d[s] = FLT_BIG; b.idx[s] = INT_MAX; b.pos[s] = -1; }
        const int leaf = (int)(__ldg(&a.leaf_rank[p + 1]) - 1u);
        nrm_scan_leaf(a.pts, a.leaf_start, (unsigned int)leaf, qx, qy, qz, b, k);
        bool done = false;
        if (b.m == k && leaf < a.adj_capacity) {
            const float r = __fmul_ru(__fsqrt_ru(b.d[k - 1]), 1.00001f);
            const float4 ilo = __ldg(&a.adj_box[2 * (size_t)leaf]), ihi = __ldg(&a.adj_box[2 * (size_t)leaf + 1]);
            if (ball_inside(qx, qy, qz, r, ilo, ihi)) {          // never true for the inverted "no list" box
                const int na = __float_as_int(ilo.w);
                for (int j = 0; j < na; ++j) {
                    const unsigned int l2 = __ldg(&a.adj[(size_t)leaf * 32 + j]);
                    const float clb = nrm_box_dist2(qx, qy, qz, __ldg(&a.bvh_box[2 * (size_t)l2]), __ldg(&a.bvh_box[2 * (size_t)l2 + 1]));
                    if (!(clb > kth(b, k))) nrm_scan_leaf(a.pts, a.leaf_start, l2, qx, qy, qz, b, k);
                }
                done = true;
            }
        }
        if (!done) {
            // exact fallback: depth-first walk with a private stack (the own leaf is met again; duplicates are rejected below)
            unsigned int st[NRM_STACK]; int top = 0;
            const int top_level = bvh.n_levels - 1;
            // restart the list: the walk meets every leaf within range, the own one included
            b.m = 0;
#pragma unroll
            for (int s = 0; s < NRM_KMAX; ++s) { b.d[s] = FLT_BIG; b.idx[s] = INT_MAX; b.pos[s] = -1; }
            nrm_scan_leaf(a.pts, a.leaf_start, (unsigned int)leaf, qx, qy, qz, b, k);
            for (int c0 = 0; c0 < bvh.count[top_level]; ++c0) {      // one top-level subtree at a time: the stack holds <= 31 * levels + 1 entries
                st[0] = ((unsigned int)top_level << 27) | (unsigned int)c0; top = 1;
                while (top > 0) {
                    const unsigned int e = st[--top];
                    const int lvl = (int)(e >> 27); const unsigned int j = e & 0x7FFFFFFu;
                    const float clb = nrm_box_dist2(qx, qy, qz, __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[lvl] + j)]), __ldg(&a.bvh_box[2 * (size_t)(bvh.offset[lvl] + j) + 1]));
                    if (clb > kth(b, k)) continue;
                    if (lvl == 0) { if ((int)j != leaf) nrm_scan_leaf(a.pts, a.leaf_start, j, qx, qy, qz, b, k); continue; }
                    const unsigned int first = __ldg(&a.child_start[bvh.coffset[lvl] + j]), last = __ldg(&a.child_start[bvh.coffset[lvl] + j + 1]);
                    for (unsigned int c = first; c < last && top < NRM_STACK; ++c) st[top++] = ((unsigned int)(lvl - 1) << 27) | c;
                }
            }
        }
        if (b.m >= 3) {
            // mean and covariance of the neighbourhood, in double, in list order (oracle: orc_pca_normals)
            double nbr[NRM_KMAX][3];
            double mean[3] = {0.0, 0.0, 0.0};
#pragma unroll
            for (int s = 0; s < NRM_KMAX; ++s) if (s < b.m) {
                const float4 t = __ldg(&a.pts[b.pos[s]]);
                nbr[s][0] = t.x; nbr[s][1] = t.y; nbr[s][2] = t.z;
                mean[0] += nbr[s][0]; mean[1] += nbr[s][1]; mean[2] += nbr[s][2];
            }
            const double dm = (double)b.m;
            mean[0] /= dm; mean[1] /= dm; mean[2] /= dm;
            double C[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int s = 0; s < NRM_KMAX; ++s) if (s < b.m) {
                const double d[3] = {nbr[s][0] - mean[0], nbr[s][1] - mean[1], nbr[s][2] - mean[2]};
#pragma unroll
                for (int r = 0; r < 3; ++r)
#pragma unroll
                    for (int c = 0; c < 3; ++c) C[r * 3 + c] += d[r] * d[c];
            }
#pragma unroll
            for (int i = 0; i < 9; ++i) C[i] /= dm;
            double V[9], ev[3];
            nrm_eig3(C, V, ev);
            double ex = V[0], ey = V[3], ez = V[6];
            const double sum = (ev[0] + ev[1]) + ev[2];
            const double vx = (double)a.vp[0] - (double)qx, vy = (double)a.vp[1] - (double)qy, vz = (double)a.vp[2] - (double)qz;
            if ((vx * ex + vy * ey) + vz * ez < 0) { ex = -ex; ey = -ey; ez = -ez; }       // flipNormalTowardsViewpoint
            nx = (float)ex; ny = (float)ey; nz = (float)ez;
            curv = sum != 0 ? (float)fabs(ev[0] / sum) : 0.f;
        }
    }
    // results: compact output in ORIGINAL order, and the cloud's own normal arrays (sorted + original), colours kept
    a.out_nrm[3 * (size_t)orig] = nx; a.out_nrm[3 * (size_t)orig + 1] = ny; a.out_nrm[3 * (size_t)orig + 2] = nz;
    a.out_curv[orig] = curv;
    float4 ns = a.nrm_sorted[p]; ns.x = nx; ns.y = ny; ns.z = nz; a.nrm_sorted[p] = ns;
    float4 no = a.nrm_orig[orig]; no.x = nx; no.y = ny; no.z = nz; a.nrm_orig[orig] = no;
}

cudaError_t icp_launch_pca_normals(const NormalArgs& a, cudaStream_t s) {
    if (a.n <= 0) return cudaSuccess;
    pca_normals_kernel<<<(a.n + 127) / 128, 128, 0, s>>>(a);
    return cudaGetLastError();
}
