// voxel.cu -- voxel-grid downsampling on the device (pcl::VoxelGrid, Open3D's voxel_down_sample): one centroid per occupied voxel,
// many clouds in one pass.  DESIGN.md section 4 rows V1-V5 fix the arithmetic; tests/voxel_reference.c restates it.
//
// Launches of one call, whatever the number of clouds:
//   voxel_coords_kernel       each point's voxel (V1) and each cloud's integer bounds (min / max atomics: deterministic)
//   (host)                    the bounds read back: the refusals, and the widths of the key's fields from the actual extents
//   per 32-bit key word, least significant first: voxel_key_kernel (the word + pass 0's histogram, as keys_kernel counts it), then
//                             the passes of grid.cu's stable radix sort -- one word for keys of up to 31 bits, LSD over the words
//                             beyond (stable, hence lexicographic)
//   voxel_head_kernel         1 where a sorted position starts a new voxel
//   flag count + block scan   prep.cu's compaction: every voxel's rank
//   voxel_run_kernel          the first sorted position of every voxel (and the end of the last)
//   voxel_centroid_kernel     one thread per voxel: V3-V5 over its run in ascending original index, off_out
#include "icp_internal.cuh"
#include <limits.h>

#define VOX_THREADS 256
#define VOX_CHUNK 8
static_assert(VOX_THREADS == ICP_FLAG_SCAN_BLOCK, "voxel_run_kernel reads the compaction's block offsets");

// The cloud of input point i: the last c with off[c] <= i (empty clouds own no point).
__device__ __forceinline__ int cloud_of(const long long* __restrict__ off, int n_clouds, long long i) {
    int lo = 0, hi = n_clouds;          // off[lo] <= i < off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(&off[mid]) <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// V1: voxel (floorf(x * inv), ...) of the points with three finite coordinates.  The bounds are reduced per warp over the lanes of one
// cloud, and per block when the block's points all belong to one cloud (the common case: one block, six global atomics).
__global__ void __launch_bounds__(VOX_THREADS) voxel_coords_kernel(const float* __restrict__ xyz, int n, const long long* __restrict__ off, int n_clouds,
                                                                   float inv, int4* __restrict__ vox, int* __restrict__ bounds, unsigned int* __restrict__ bad) {
    __shared__ int s_c[2], s_b[6];
    const int i0 = blockIdx.x * VOX_THREADS, i = i0 + threadIdx.x;
    if (threadIdx.x < 2) s_c[threadIdx.x] = cloud_of(off, n_clouds, threadIdx.x == 0 ? i0 : min(n, i0 + VOX_THREADS) - 1);
    if (threadIdx.x < 6) s_b[threadIdx.x] = threadIdx.x < 3 ? INT_MAX : INT_MIN;
    __syncthreads();
    const bool one = s_c[0] == s_c[1];
    int c = -1, v[3] = {0, 0, 0};
    if (i < n) {
        const int ci = one ? s_c[0] : cloud_of(off, n_clouds, i);
        const float p[3] = {xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2]};
        if (finite3(p[0], p[1], p[2])) {
            bool fits = true;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float f = floorf(__fmul_rn(p[a], inv));
                if (f >= -2147483648.0f && f < 2147483648.0f) v[a] = (int)f; else fits = false;
            }
            if (fits) c = ci; else bad[ci] = 1u;
        }
        vox[i] = make_int4(v[0], v[1], v[2], c);
    }
    const unsigned int peers = __match_any_sync(0xFFFFFFFFu, c);
    int mn[3], mx[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) { mn[a] = __reduce_min_sync(peers, v[a]); mx[a] = __reduce_max_sync(peers, v[a]); }
    if (c >= 0 && (peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0u) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (one) { atomicMin(&s_b[a], mn[a]); atomicMax(&s_b[3 + a], mx[a]); }
            else { atomicMin(&bounds[6 * c + a], mn[a]); atomicMax(&bounds[6 * c + 3 + a], mx[a]); }
        }
    }
    __syncthreads();
    if (one && threadIdx.x < 6) {
        if (threadIdx.x < 3) atomicMin(&bounds[6 * s_c[0] + threadIdx.x], s_b[threadIdx.x]);
        else atomicMax(&bounds[6 * s_c[0] + threadIdx.x], s_b[threadIdx.x]);
    }
}

// Word `word` of the key of item i (the point idx_in[i], or i), and its count in pass 0's histogram (cleared by the caller).  A
// non-finite point's top word is 1 << top_bits: after every voxel of every cloud.
__global__ void __launch_bounds__(VOX_THREADS) voxel_key_kernel(const int4* __restrict__ vox, const unsigned int* __restrict__ idx_in, int n,
                                                                const int* __restrict__ bounds, VoxKeyLayout L, int word, unsigned int* __restrict__ keys,
                                                                int tile_items, int tiles_pad, int shift, int bits, unsigned int* __restrict__ hist0) {
    const int i = blockIdx.x * VOX_THREADS + threadIdx.x;
    if (i >= n) return;
    const int4 v = vox[idx_in ? idx_in[i] : (unsigned int)i];
    unsigned int key;
    if (v.w < 0) {
        key = word == L.n_words - 1 ? (1u << L.top_bits) : 0u;
    } else {
        const int* b = bounds + 6 * v.w;
        unsigned __int128 k = (unsigned int)v.w;
        k = (k << L.bz) | (unsigned int)(v.z - __ldg(&b[2]));
        k = (k << L.by) | (unsigned int)(v.y - __ldg(&b[1]));
        k = (k << L.bx) | (unsigned int)(v.x - __ldg(&b[0]));
        key = (unsigned int)(k >> (32 * word));
    }
    keys[i] = key;
    atomicAdd(&hist0[(size_t)((key >> shift) & ((1u << bits) - 1u)) * tiles_pad + (unsigned int)i / (unsigned int)tile_items], 1u);
}

__device__ __forceinline__ bool same_voxel(int4 a, int4 b) { return a.x == b.x && a.y == b.y && a.z == b.z && a.w == b.w; }

// flag[p] = 1 where sorted position p holds a finite point whose voxel differs from position p - 1's.
__global__ void __launch_bounds__(VOX_THREADS) voxel_head_kernel(const unsigned int* __restrict__ idx, int n, const int4* __restrict__ vox,
                                                                 unsigned int* __restrict__ flag) {
    const int p = blockIdx.x * VOX_THREADS + threadIdx.x;
    if (p >= n) return;
    const int4 v = vox[idx[p]];
    flag[p] = (v.w >= 0 && (p == 0 || !same_voxel(v, vox[idx[p - 1]]))) ? 1u : 0u;
}

// run_start[rank of the voxel] = its first sorted position; the last finite position also writes run_start[n_vox] (its end).
__global__ void __launch_bounds__(VOX_THREADS) voxel_run_kernel(const unsigned int* __restrict__ flag, int n, const unsigned int* __restrict__ block_offset,
                                                                const unsigned int* __restrict__ n_vox, const unsigned int* __restrict__ idx,
                                                                const int4* __restrict__ vox, unsigned int* __restrict__ run_start) {
    __shared__ unsigned int s_w[VOX_THREADS / 32];
    const int p = blockIdx.x * VOX_THREADS + threadIdx.x;
    const bool f = p < n && flag[p] != 0u;
    const unsigned int m = __ballot_sync(0xFFFFFFFFu, f);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) s_w[w] = __popc(m);
    __syncthreads();
    unsigned int before = block_offset[blockIdx.x];
    for (int j = 0; j < w; ++j) before += s_w[j];
    if (f) run_start[before + __popc(m & ((1u << lane) - 1u))] = (unsigned int)p;
    if (p < n && vox[idx[p]].w >= 0 && (p == n - 1 || vox[idx[p + 1]].w < 0)) run_start[*n_vox] = (unsigned int)p + 1u;
}

// One thread per voxel: V3 (fp64 sequential sums in ascending original index -- the stable sort's order within a run -- over the
// count), V4 (the same sum of the finite normals over its fp64 norm; MINF when there is none or the norm is 0), V5 ((2 sum + k) / 2k
// per channel).  No contraction: every operation is an explicitly rounded intrinsic, as the -ffp-contract=off C of tests/voxel_reference.c.  The voxel
// whose cloud differs from the previous voxel's writes the offsets of the clouds in between (empty clouds included); the last voxel
// those after it.
__global__ void __launch_bounds__(VOX_THREADS) voxel_centroid_kernel(const unsigned int* __restrict__ run_start, const unsigned int* __restrict__ n_vox,
                                                                     const unsigned int* __restrict__ idx, const int4* __restrict__ vox,
                                                                     const float* __restrict__ xyz, const float* __restrict__ nrm,
                                                                     const uint8_t* __restrict__ rgba, int n_clouds, float* __restrict__ xyz_out,
                                                                     float* __restrict__ nrm_out, uint8_t* __restrict__ rgba_out,
                                                                     long long* __restrict__ off_out) {
    const unsigned int v = blockIdx.x * VOX_THREADS + threadIdx.x, nv = *n_vox;
    if (v >= nv) return;
    const unsigned int s = run_start[v], e = run_start[v + 1];
    double px = 0.0, py = 0.0, pz = 0.0, nx = 0.0, ny = 0.0, nz = 0.0;
    unsigned long long col[4] = {0ull, 0ull, 0ull, 0ull};
    bool any_normal = false;
    // Chunks of VOX_CHUNK points: the chunk's index loads, then its gathered loads, are all in flight at once (a voxel near a lidar holds
    // thousands of points, and one at a time its thread waits on two dependent loads per point); the sums still run point by point.
    for (unsigned int q0 = s; q0 < e; q0 += VOX_CHUNK) {
        const unsigned int m = min(e - q0, (unsigned int)VOX_CHUNK);
        unsigned int j[VOX_CHUNK];
        float p[VOX_CHUNK][3];
#pragma unroll
        for (int t = 0; t < VOX_CHUNK; ++t) j[t] = (unsigned int)t < m ? __ldg(&idx[q0 + t]) : 0u;
#pragma unroll
        for (int t = 0; t < VOX_CHUNK; ++t)
            if ((unsigned int)t < m) for (int a = 0; a < 3; ++a) p[t][a] = __ldg(&xyz[3 * (size_t)j[t] + a]);
#pragma unroll
        for (int t = 0; t < VOX_CHUNK; ++t)
            if ((unsigned int)t < m) { px = __dadd_rn(px, (double)p[t][0]); py = __dadd_rn(py, (double)p[t][1]); pz = __dadd_rn(pz, (double)p[t][2]); }
        if (nrm) {
#pragma unroll
            for (int t = 0; t < VOX_CHUNK; ++t)
                if ((unsigned int)t < m) for (int a = 0; a < 3; ++a) p[t][a] = __ldg(&nrm[3 * (size_t)j[t] + a]);
#pragma unroll
            for (int t = 0; t < VOX_CHUNK; ++t)
                if ((unsigned int)t < m && finite3(p[t][0], p[t][1], p[t][2])) {
                    nx = __dadd_rn(nx, (double)p[t][0]); ny = __dadd_rn(ny, (double)p[t][1]); nz = __dadd_rn(nz, (double)p[t][2]); any_normal = true;
                }
        }
        if (rgba) {
#pragma unroll
            for (int t = 0; t < VOX_CHUNK; ++t)
                if ((unsigned int)t < m) {
                    const unsigned int c = __ldg(reinterpret_cast<const unsigned int*>(rgba) + j[t]);
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) col[ch] += (c >> (8 * ch)) & 0xFFu;
                }
        }
    }
    const unsigned int k = e - s;
    const double dk = (double)k;
    xyz_out[3 * (size_t)v] = (float)__ddiv_rn(px, dk); xyz_out[3 * (size_t)v + 1] = (float)__ddiv_rn(py, dk); xyz_out[3 * (size_t)v + 2] = (float)__ddiv_rn(pz, dk);
    if (nrm_out) {
        const double len = __dsqrt_rn(__dadd_rn(__dadd_rn(__dmul_rn(nx, nx), __dmul_rn(ny, ny)), __dmul_rn(nz, nz)));
        float o[3] = {MINF_F, MINF_F, MINF_F};
        if (any_normal && len != 0.0) { o[0] = (float)__ddiv_rn(nx, len); o[1] = (float)__ddiv_rn(ny, len); o[2] = (float)__ddiv_rn(nz, len); }
        nrm_out[3 * (size_t)v] = o[0]; nrm_out[3 * (size_t)v + 1] = o[1]; nrm_out[3 * (size_t)v + 2] = o[2];
    }
    if (rgba_out) {
        unsigned int c = 0;
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) c |= (unsigned int)((2ull * col[ch] + k) / (2ull * k)) << (8 * ch);
        reinterpret_cast<unsigned int*>(rgba_out)[v] = c;
    }
    const int cl = vox[idx[s]].w, prev = v == 0 ? -1 : vox[idx[run_start[v - 1]]].w;
    for (int b = prev + 1; b <= cl; ++b) off_out[b] = v;
    if (v == nv - 1) for (int b = cl + 1; b <= n_clouds; ++b) off_out[b] = nv;
}

cudaError_t icp_launch_voxel_coords(const float* xyz, int n, const long long* off, int n_clouds, float inv, int4* vox, int* bounds, unsigned int* bad,
                                    cudaStream_t s, int* n_launches) {
    if (n <= 0) return cudaSuccess;
    voxel_coords_kernel<<<(n + VOX_THREADS - 1) / VOX_THREADS, VOX_THREADS, 0, s>>>(xyz, n, off, n_clouds, inv, vox, bounds, bad);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

cudaError_t icp_launch_voxel_sort(const int4* vox, int n, const int* bounds, const VoxKeyLayout& L, unsigned int* keys_a, unsigned int* keys_b,
                                  unsigned int* idx_a, unsigned int* idx_b, unsigned int* hist, cudaStream_t s, unsigned int** idx_sorted, int* n_launches) {
    unsigned int* idx = nullptr;
    int launches = 0;
    for (int w = 0; w < L.n_words && n > 0; ++w) {
        // the lower words are whole 32-bit words (T = 31: 32 key bits); the top word holds the rest and the non-finite bit above it
        const int T = w == L.n_words - 1 ? L.top_bits : 31;
        IcpRadixPlan p; icp_radix_plan(n, T, &p);
        cudaError_t e = cudaMemsetAsync(hist, 0, icp_radix_hist_words(n, T) * 4, s);
        if (e != cudaSuccess) return e;
        voxel_key_kernel<<<(n + VOX_THREADS - 1) / VOX_THREADS, VOX_THREADS, 0, s>>>(vox, idx, n, bounds, L, w, keys_a, p.tile_items, p.tiles_pad, p.shift[0],
                                                                                    p.bits[0], hist);
        ++launches;
        unsigned int* ks;
        // the previous word's order (idx) is the items' index of this word's pass 0; the passes then start writing the other buffer
        unsigned int* ia = idx == idx_a ? idx_b : idx_a;
        icp_radix_passes(p, n, keys_a, keys_b, idx, ia, ia == idx_a ? idx_b : idx_a, hist, nullptr, s, &ks, &idx, &launches);
    }
    *idx_sorted = idx;
    if (n_launches) *n_launches += launches;
    return cudaGetLastError();
}

cudaError_t icp_launch_voxel_centroids(const unsigned int* idx_sorted, const int4* vox, int n, const float* xyz, const float* nrm, const uint8_t* rgba,
                                       int n_clouds, unsigned int* flag, unsigned int* block_offset, unsigned int* n_vox, unsigned int* run_start,
                                       float* xyz_out, float* nrm_out, uint8_t* rgba_out, long long* off_out, cudaStream_t s, int* n_launches) {
    if (n <= 0) return cudaSuccess;
    const int nb = (n + VOX_THREADS - 1) / VOX_THREADS;
    voxel_head_kernel<<<nb, VOX_THREADS, 0, s>>>(idx_sorted, n, vox, flag);
    cudaError_t e = icp_launch_flag_scan(flag, n, block_offset, n_vox, s, n_launches);
    if (e != cudaSuccess) return e;
    voxel_run_kernel<<<nb, VOX_THREADS, 0, s>>>(flag, n, block_offset, n_vox, idx_sorted, vox, run_start);
    // at most n voxels: the threads past the count return at once
    voxel_centroid_kernel<<<nb, VOX_THREADS, 0, s>>>(run_start, n_vox, idx_sorted, vox, xyz, nrm, rgba, n_clouds, xyz_out, nrm_out, rgba_out, off_out);
    if (n_launches) *n_launches += 3;
    return cudaGetLastError();
}
