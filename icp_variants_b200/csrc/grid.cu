// grid.cu -- buildIndex: the on-device search structure that replaces FLANN's kd-tree
// (reference: NearestNeighborSearchFlann::buildIndex, NearestNeighbor.h:122-141 / :209-232).
//
// Structure: a uniform grid of 2^T cells (T = 30 for a target: 10 bits per axis) whose cell codes are Morton-style
// bit interleavings of the per-axis cell indices (the axis taken at each bit is the currently longest one, so cells end up
// near-cubic).  The cloud is sorted by (cell code, original index) with a stable LSD RADIX SORT -- 4 passes of 7-8 bits,
// every pass = per-tile digit histograms, their scan, and a ranking scatter (warp-level multi-split with match.any, no atomics in the
// ranking: the order inside a cell is the original index order, so two uploads of the same cloud give the same structure
// bit for bit).  There is no dense cell table: the implicit binary tree over the cells is read off the SORTED KEYS -- the
// node of depth d around point i is the maximal run of points around i whose neighbouring keys share >= d leading bits
// (delta(i) = common-prefix length of key[i-1] and key[i]).  Leaves = the shallowest such nodes with <= 32 points, level-l
// nodes = the shallowest with <= 32 nodes of level l-1; both are found per element from a +-32 window of delta values.
//
// Launches of one target build (no host synchronisation): pack+bbox+grid parameters, keys+hist, (scan, scatter) x passes, gather,
// leaf flags, leaf ranks, leaf boxes, level-1 flags / ranks / boxes, one single-block kernel for all levels above,
// two adjacency kernels.
#include "search.cuh"
#include <string.h>

// ---------------------------------------------------------------------------- pack AoS3 -> float4, bounding box
__device__ __forceinline__ unsigned int enc_f(float f) { unsigned int b = __float_as_uint(f); return (b & 0x80000000u) ? ~b : (b | 0x80000000u); }
__device__ __forceinline__ float dec_f(unsigned int e) { return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e); }

// Layout in HBM: points {x,y,z,original index bits}, normals {nx,ny,nz,rgba bits}.
// scratch words: [0..2] encoded min, [3..5] encoded max of the finite points (initialised to 0xFFFFFFFF / 0), [6] block ticket,
// [7] number of points with a non-finite coordinate.  The kernel also clears the radix sort's histograms (zero / zero_words)
// and its last block derives the grid parameters from the finished bounding box -- no launch of their own.
__device__ void grid_params_from_bbox(const unsigned int* bbox, int T, GridParams& P);

__global__ void __launch_bounds__(256) pack_bbox_kernel(const float* __restrict__ xyz, const float* __restrict__ nrm, const uint8_t* __restrict__ rgba,
                                                        int n, float4* __restrict__ pts, float4* __restrict__ nrmo, unsigned int* bbox, int T,
                                                        GridParams* __restrict__ gp_out, unsigned int* __restrict__ zero, long long zero_words,
                                                        int with_normals) {
    for (long long z = (long long)blockIdx.x * blockDim.x + threadIdx.x; z < zero_words; z += (long long)gridDim.x * blockDim.x) zero[z] = 0u;
    unsigned int mn[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, mx[3] = {0u, 0u, 0u};
    unsigned int bad = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 p; p.x = xyz[3 * (size_t)i]; p.y = xyz[3 * (size_t)i + 1]; p.z = xyz[3 * (size_t)i + 2]; p.w = __int_as_float(i);
        pts[i] = p;
        if (with_normals) {
            unsigned int c = 0;
            if (rgba) c = reinterpret_cast<const unsigned int*>(rgba)[i];
            float4 m = make_float4(0.f, 0.f, 0.f, __uint_as_float(c));
            if (nrm) { m.x = nrm[3 * (size_t)i]; m.y = nrm[3 * (size_t)i + 1]; m.z = nrm[3 * (size_t)i + 2]; }
            nrmo[i] = m;
        }
        if (finite3(p.x, p.y, p.z)) {
            const unsigned int e[3] = {enc_f(p.x), enc_f(p.y), enc_f(p.z)};
#pragma unroll
            for (int a = 0; a < 3; ++a) { mn[a] = min(mn[a], e[a]); mx[a] = max(mx[a], e[a]); }
        } else ++bad;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        mn[a] = __reduce_min_sync(0xFFFFFFFFu, mn[a]);
        mx[a] = __reduce_max_sync(0xFFFFFFFFu, mx[a]);
    }
    bad = __reduce_add_sync(0xFFFFFFFFu, bad);
    // one atomic per block and value (thousands of same-address atomics from every warp cost tens of microseconds)
    __shared__ unsigned int s_mn[3][8], s_mx[3][8], s_bad[8];
    __shared__ bool s_last;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) {
#pragma unroll
        for (int a = 0; a < 3; ++a) { s_mn[a][wid] = mn[a]; s_mx[a][wid] = mx[a]; }
        s_bad[wid] = bad;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        const int a = threadIdx.x % 3; const bool is_max = threadIdx.x >= 3;
        unsigned int v = is_max ? 0u : 0xFFFFFFFFu;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v = is_max ? max(v, s_mx[a][w]) : min(v, s_mn[a][w]);
        if (is_max) atomicMax(&bbox[3 + a], v); else atomicMin(&bbox[a], v);
    } else if (threadIdx.x == 6) {
        unsigned int v = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += s_bad[w];
        if (v) atomicAdd(&bbox[7], v);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&bbox[6], 1u) == gridDim.x - 1;
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        __threadfence();
        unsigned int bb[6];
        for (int k = 0; k < 6; ++k) bb[k] = *reinterpret_cast<volatile unsigned int*>(&bbox[k]);
        GridParams P;
        grid_params_from_bbox(bb, T, P);
        *gp_out = P;
    }
}

// The normal / colour records alone: host uploads deliver them after the points, and only the last pass of the sort reads them.
__global__ void __launch_bounds__(256) pack_normals_kernel(const float* __restrict__ nrm, const uint8_t* __restrict__ rgba, int n, float4* __restrict__ nrmo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned int c = 0;
    if (rgba) c = reinterpret_cast<const unsigned int*>(rgba)[i];
    float4 m = make_float4(0.f, 0.f, 0.f, __uint_as_float(c));
    if (nrm) { m.x = nrm[3 * (size_t)i]; m.y = nrm[3 * (size_t)i + 1]; m.z = nrm[3 * (size_t)i + 2]; }
    nrmo[i] = m;
}

// with_normals = 0: only the point records (the normal records follow through IcpLatePack / icp_launch_cloud_sort)
cudaError_t icp_launch_pack_cloud(const float* xyz, const float* nrm, const uint8_t* rgba, int n, float4* pts, float4* nrmo,
                                  unsigned int* bbox, int T, GridParams* grid, unsigned int* zero, long long zero_words, int with_normals,
                                  cudaStream_t s) {
    cudaError_t e;
    if ((e = cudaMemsetAsync(bbox, 0xFF, 3 * sizeof(unsigned int), s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(bbox + 3, 0x00, 5 * sizeof(unsigned int), s)) != cudaSuccess) return e;   // max[3], ticket, non-finite counter
    int nb = min((n + 255) / 256, 148 * 4); if (nb < 1) nb = 1;           // n == 0: one block still writes the (empty-cloud) grid parameters
    pack_bbox_kernel<<<nb, 256, 0, s>>>(xyz, nrm, rgba, n, pts, nrmo, bbox, T, grid, zero, zero_words, with_normals);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- grid parameters and cell codes
// A pure function of the bounding box: every block that needs the parameters derives them itself (no launch of its own);
// the oracle restates this arithmetic (oracle/icp_oracle.c: voxel levels), hence no FMA.
__device__ void grid_params_from_bbox(const unsigned int* bbox, int T, GridParams& P) {
    float e[3], maxabs[3];
    const bool empty = bbox[0] == 0xFFFFFFFFu && bbox[3] == 0u;
    for (int a = 0; a < 3; ++a) {
        const float lo = empty ? 0.f : dec_f(bbox[a]), hi = empty ? 0.f : dec_f(bbox[3 + a]);
        P.o[a] = lo;
        maxabs[a] = fmaxf(fabsf(lo), fabsf(hi));
        e[a] = fmaxf(psub(hi, lo), padd(1e-20f, pmul(1e-6f, maxabs[a])));   // zero-extent axes stay well defined
        P.bits[a] = 0;
    }
    // Level k of the implicit tree halves the axis whose cells are currently the longest.
    float cur[3] = {e[0], e[1], e[2]};
    unsigned long long seq = 0ull;
    for (int k = 0; k < T; ++k) {
        int a = -1; float best = -1.f;
        for (int c = 0; c < 3; ++c) if (P.bits[c] < ICP_MAX_BITS_PER_AXIS && cur[c] > best) { best = cur[c]; a = c; }
        if (a < 0) a = 0;   // unreachable for T <= 3*ICP_MAX_BITS_PER_AXIS
        seq |= (unsigned long long)a << (2 * k);
        P.bits[a] += 1; cur[a] = pmul(cur[a], 0.5f);
    }
    for (int a = 0; a < 3; ++a) {
        P.h[a] = pdiv(pmul(e[a], 1.00001f), (float)(1 << P.bits[a]));
        P.inv_h[a] = pdiv(1.0f, P.h[a]);
        P.delta[a] = 1e-3f * P.h[a] + 1e-6f * maxabs[a];
    }
    P.T = T; P.axis_seq = seq; P.n_finite = 0; P.pad = 0;
    // where the bits of an axis' cell index go in the code: level k (root split = most significant code bit) takes the
    // highest not yet used bit of its axis
    int r[3] = {P.bits[0], P.bits[1], P.bits[2]};
    for (int a = 0; a < 3; ++a) for (int j = 0; j < ICP_MAX_BITS_PER_AXIS; ++j) P.bitpos[a][j] = 0;
    for (int k = 0; k < T; ++k) { const int a = (int)((seq >> (2 * k)) & 3ull); --r[a]; P.bitpos[a][r[a]] = (unsigned char)(T - 1 - k); }
}


// ---------------------------------------------------------------------------- stable LSD radix sort of (key, index)
// key = cell code (T bits); a point with a non-finite coordinate gets 1 << T: it sorts after every cell (sources keep such
// points at the end -- every point needs a slot; targets simply never look past n_finite).  T + 1 bits are sorted in
// passes of <= 8 bits over tiles of 512 threads x ipt contiguous items (one tile per SM for clouds up to ~600k points).
// Per pass:
//   digit histograms per tile, digit-major (hist[d * tiles_pad + tile]): pass 0's by the key kernel; pass p+1's by the
//     scatter kernel of pass p (an item's next tile is known once its slot is: one L2 atomic per item);
//   radix_scan_kernel: one warp per digit turns the digit's row into exclusive prefixes over the tiles (+ the digit's total);
//   radix_scatter_kernel: a tile's first slot per digit = digits before it (block scan of the totals) + the same digit in
//     earlier tiles; the tile's items are ranked per warp (contiguous chunk per warp, rounds of 32 in order; match.any groups
//     equal digits, the group's lowest lane advances the warp's running slot) and written to their slots: stable,
//     deterministic -- no atomics decide any position.
// A final gather moves the point and normal records into the sorted order (coalesced writes).
#define KEY_THREADS 256
#define RS_THREADS 512
#define RS_WARPS (RS_THREADS / 32)
#define RS_MAX_BITS 8
#define RS_MAX_BINS (1 << RS_MAX_BITS)
#define RS_REG_IPT 8

// Thread per point: key + the point's count in pass 0's histogram (cleared by the pack kernel).
__global__ void __launch_bounds__(KEY_THREADS) keys_kernel(const float4* __restrict__ pts, int n, const GridParams* __restrict__ gp,
                                                           unsigned int* __restrict__ keys, int tile_items, int tiles_pad, int shift, int bits,
                                                           unsigned int* __restrict__ hist0) {
    __shared__ GridParams g;
    if (threadIdx.x < sizeof(GridParams) / 4) reinterpret_cast<unsigned int*>(&g)[threadIdx.x] = reinterpret_cast<const unsigned int*>(gp)[threadIdx.x];
    __syncthreads();
    const int i = blockIdx.x * KEY_THREADS + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i];
    const unsigned int key = finite3(p.x, p.y, p.z) ? cell_code(g, p.x, p.y, p.z) : (1u << g.T);   // non-finite: can never win the strict '>' scan of NearestNeighbor.h:87
    keys[i] = key;
    atomicAdd(&hist0[(size_t)((key >> shift) & ((1u << bits) - 1u)) * tiles_pad + (unsigned int)i / (unsigned int)tile_items], 1u);
}

// One warp per digit: the digit's per-tile counts -> exclusive prefixes over the tiles; totals[d] = the digit's count.
__global__ void __launch_bounds__(256) radix_scan_kernel(unsigned int* __restrict__ hist, int bins, int n_tiles, int tiles_pad, unsigned int* __restrict__ totals) {
    const int d = (blockIdx.x * 256 + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (d >= bins) return;
    unsigned int* row = hist + (size_t)d * tiles_pad;
    unsigned int carry = 0;
    for (int c = 0; c < tiles_pad; c += 32) {
        const unsigned int v = c + lane < n_tiles ? row[c + lane] : 0u;      // the pad columns are never written
        unsigned int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
        row[c + lane] = carry + inc - v;
        carry += __shfl_sync(0xFFFFFFFFu, inc, 31);
    }
    if (lane == 0) totals[d] = carry;
}

__device__ __forceinline__ unsigned int block_exclusive_scan(unsigned int v, unsigned int* total) {
    __shared__ unsigned int warp_sums[32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    unsigned int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { unsigned int t = __shfl_up_sync(0xFFFFFFFFu, inc, o); if (lane >= o) inc += t; }
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    if (w == 0) {
        unsigned int s = lane < (int)(blockDim.x >> 5) ? warp_sums[lane] : 0u, si = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { unsigned int t = __shfl_up_sync(0xFFFFFFFFu, si, o); if (lane >= o) si += t; }
        warp_sums[lane] = si - s;
        if (lane == 31 && total) *total = si;
    }
    __syncthreads();
    const unsigned int r = inc - v + warp_sums[w];
    __syncthreads();
    return r;
}

// idx_in == nullptr: the identity (pass 0).  hist: this pass's scanned histogram; hist_next (nullable): the next pass's, counted
// here.  msd_start (nullable, last pass): first output slot of every digit of the pass, bins + 1 entries.  ipt <= RS_REG_IPT: a
// thread's keys, indices and slots stay in registers between the phases (all loads of a phase in flight at once: with one
// block per SM the kernel is bound by the length of its chains of dependent instructions, not by bandwidth).
// One count for the next pass's histogram, aggregated over the lanes of the warp that hit the same counter: sorted keys
// put neighbours into the same (digit, tile) cell -- 32 same-address L2 atomics per warp otherwise, and the high digits of a
// room scan take only a few dozen values.
__device__ __forceinline__ void count_next(unsigned int* __restrict__ hist_next, unsigned int cell) {
    const unsigned int peers = __match_any_sync(__activemask(), cell);
    if ((peers & ((1u << (threadIdx.x & 31)) - 1u)) == 0u) atomicAdd(&hist_next[cell], (unsigned int)__popc(peers));
}

template <bool REG>
__global__ void __launch_bounds__(RS_THREADS) radix_scatter_kernel(const unsigned int* __restrict__ keys_in, const unsigned int* __restrict__ idx_in,
                                                                   unsigned int* __restrict__ keys_out, unsigned int* __restrict__ idx_out, int n,
                                                                   int ipt, int tiles_pad, int shift, int bits,
                                                                   const unsigned int* __restrict__ hist, const unsigned int* __restrict__ totals,
                                                                   unsigned int* __restrict__ hist_next, int shift_next, int bits_next,
                                                                   unsigned int* __restrict__ msd_start) {
    __shared__ unsigned short wcnt[RS_WARPS][RS_MAX_BINS];     // per warp and digit: count, then tile-relative first slot, then running slot
    __shared__ unsigned int base[RS_MAX_BINS];                 // per digit: first output slot of this tile
    const unsigned int FULL = 0xFFFFFFFFu;
    const int bins = 1 << bits;
    const unsigned int mask = (unsigned int)bins - 1u;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned int lt = (1u << lane) - 1u;
    const int tile_items = ipt * RS_THREADS;
    const int chunk = ipt * 32;                                // the warp's contiguous share of the tile
    const long long w0 = (long long)blockIdx.x * tile_items + (long long)w * chunk;
    unsigned int kreg[RS_REG_IPT], ireg[RS_REG_IPT];
    if (REG) {
#pragma unroll
        for (int r = 0; r < RS_REG_IPT; ++r) {
            const long long i = w0 + r * 32 + lane;
            const bool valid = r < ipt && i < n;
            kreg[r] = valid ? keys_in[i] : 0u;
            ireg[r] = valid ? (idx_in ? idx_in[i] : (unsigned int)i) : 0u;
        }
    }
    {
        unsigned int* z = reinterpret_cast<unsigned int*>(&wcnt[0][0]);
        for (int d = threadIdx.x; d < RS_WARPS * RS_MAX_BINS / 2; d += RS_THREADS) z[d] = 0u;
    }
    // the loads of the offsets below depend on nothing: issue them before the counting phase (thread d < bins owns digit d)
    const int d_own = threadIdx.x;
    unsigned int before = 0u, tot = 0u;
    if (d_own < bins) { before = __ldg(&hist[(size_t)d_own * tiles_pad + blockIdx.x]); tot = __ldg(&totals[d_own]); }
    __syncthreads();
    // phase A: digit counts of the warp's chunk, rounds of 32 items
    if (REG) {
#pragma unroll
        for (int r = 0; r < RS_REG_IPT; ++r) {
            if (r < ipt) {
                const bool valid = w0 + r * 32 + lane < n;
                const unsigned int vm = __ballot_sync(FULL, valid);
                if (valid) {
                    const unsigned int dg = (kreg[r] >> shift) & mask;
                    const unsigned int peers = __match_any_sync(vm, dg);
                    if ((peers & lt) == 0u) wcnt[w][dg] = (unsigned short)(wcnt[w][dg] + __popc(peers));
                }
                __syncwarp();
            }
        }
    } else {
        for (int r = 0; r < chunk; r += 32) {
            const long long i = w0 + r + lane;
            const bool valid = i < n;
            const unsigned int vm = __ballot_sync(FULL, valid);
            if (valid) {
                const unsigned int dg = (keys_in[i] >> shift) & mask;
                const unsigned int peers = __match_any_sync(vm, dg);
                if ((peers & lt) == 0u) wcnt[w][dg] = (unsigned short)(wcnt[w][dg] + __popc(peers));
            }
            __syncwarp();
            if (vm != FULL) break;
        }
    }
    __syncthreads();
    // per digit: warp counts -> exclusive prefix over the warps (tile-relative first slot of the warp's items with the digit)
    if (d_own < bins) {
        unsigned int acc = 0;
#pragma unroll
        for (int ww = 0; ww < RS_WARPS; ++ww) { const unsigned int c = wcnt[ww][d_own]; wcnt[ww][d_own] = (unsigned short)acc; acc += c; }
    }
    // exclusive scan of the digits' totals: the first slot of every digit in the output
    const unsigned int digit_base = block_exclusive_scan(d_own < bins ? tot : 0u, nullptr);
    if (d_own < bins) {
        base[d_own] = digit_base + before;
        if (msd_start && blockIdx.x == 0) { msd_start[d_own] = digit_base; if (d_own == bins - 1) msd_start[bins] = (unsigned int)n; }
    }
    __syncthreads();
    // phase B: the same rounds again; the group's lowest lane advances the warp's running slot of the digit
    const unsigned int mask_next = (1u << bits_next) - 1u;
    if (REG) {
        unsigned int pos[RS_REG_IPT];
#pragma unroll
        for (int r = 0; r < RS_REG_IPT; ++r) {
            pos[r] = 0xFFFFFFFFu;
            if (r < ipt) {
                const bool valid = w0 + r * 32 + lane < n;
                const unsigned int vm = __ballot_sync(FULL, valid);
                if (valid) {
                    const unsigned int dg = (kreg[r] >> shift) & mask;
                    const unsigned int peers = __match_any_sync(vm, dg);
                    const int leader = __ffs((int)peers) - 1;
                    unsigned int old = 0;
                    if (lane == leader) { old = wcnt[w][dg]; wcnt[w][dg] = (unsigned short)(old + __popc(peers)); }
                    old = __shfl_sync(peers, old, leader);
                    pos[r] = base[dg] + old + (unsigned int)__popc(peers & lt);
                }
                __syncwarp();
            }
        }
        // every slot is known: the moves are independent of each other
#pragma unroll
        for (int r = 0; r < RS_REG_IPT; ++r) {
            if (pos[r] != 0xFFFFFFFFu) {
                keys_out[pos[r]] = kreg[r];
                idx_out[pos[r]] = ireg[r];
                if (hist_next) count_next(hist_next, ((kreg[r] >> shift_next) & mask_next) * (unsigned int)tiles_pad + pos[r] / (unsigned int)tile_items);
            }
        }
    } else {
        for (int r = 0; r < chunk; r += 32) {
            const long long i = w0 + r + lane;
            const bool valid = i < n;
            const unsigned int vm = __ballot_sync(FULL, valid);
            if (valid) {
                const unsigned int key = keys_in[i];
                const unsigned int src = idx_in ? idx_in[i] : (unsigned int)i;
                const unsigned int dg = (key >> shift) & mask;
                const unsigned int peers = __match_any_sync(vm, dg);
                const int leader = __ffs((int)peers) - 1;
                unsigned int old = 0;
                if (lane == leader) { old = wcnt[w][dg]; wcnt[w][dg] = (unsigned short)(old + __popc(peers)); }
                old = __shfl_sync(peers, old, leader);
                const unsigned int p = base[dg] + old + (unsigned int)__popc(peers & lt);
                keys_out[p] = key;
                idx_out[p] = src;
                if (hist_next) count_next(hist_next, ((key >> shift_next) & mask_next) * (unsigned int)tiles_pad + p / (unsigned int)tile_items);
            }
            __syncwarp();
            if (vm != FULL) break;
        }
    }
}

// The records in sorted order: thread per output slot (coalesced writes, gathered reads).
__global__ void __launch_bounds__(256) gather_records_kernel(const unsigned int* __restrict__ idx, int n, const float4* __restrict__ pts_in,
                                                             const float4* __restrict__ nrm_in, float4* __restrict__ pts_out, float4* __restrict__ nrm_out) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const unsigned int s = idx[i];
    pts_out[i] = __ldg(&pts_in[s]);
    nrm_out[i] = __ldg(&nrm_in[s]);
}

void icp_radix_plan(int n, int T, IcpRadixPlan* p) {
    const int total = T + 1;
    p->n_pass = (total + RS_MAX_BITS - 1) / RS_MAX_BITS;
    const int lo = total / p->n_pass, extra = total % p->n_pass;
    int shift = 0;
    for (int k = 0; k < p->n_pass; ++k) { p->bits[k] = lo + (k < extra ? 1 : 0); p->shift[k] = shift; shift += p->bits[k]; }
    // One tile per SM while that keeps a thread's items in registers (2 .. 8 items per thread), more tiles beyond; only clouds
    // of more than 16 M points get larger tiles (the histograms have one column per tile).
    long long ipt = ((long long)n + RS_THREADS * 148 - 1) / (RS_THREADS * 148);
    if (ipt < 2) ipt = 2;
    if (ipt > RS_REG_IPT) ipt = RS_REG_IPT;
    while ((long long)n > ipt * RS_THREADS * 4096 && ipt < 120) ipt += 8;
    p->ipt = (int)ipt;
    p->tile_items = (int)(ipt * RS_THREADS);
    p->n_tiles = n > 0 ? (int)(((long long)n + p->tile_items - 1) / p->tile_items) : 0;
    p->tiles_pad = ((p->n_tiles > 0 ? p->n_tiles : 1) + 31) / 32 * 32;
}

// words of histogram scratch: one digit-major matrix per pass, then the per-digit totals
size_t icp_radix_hist_words(int n, int T) {
    IcpRadixPlan p; icp_radix_plan(n, T, &p);
    return (size_t)p.n_pass * RS_MAX_BINS * p.tiles_pad + RS_MAX_BINS;
}

void icp_radix_passes(const IcpRadixPlan& p, int n, unsigned int* kin, unsigned int* kout, unsigned int* iin, unsigned int* idx_a, unsigned int* idx_b,
                      unsigned int* hist, unsigned int* msd_start, cudaStream_t s, unsigned int** keys_sorted_out, unsigned int** idx_sorted_out,
                      int* launches) {
    unsigned int* iout = idx_a;
    const size_t mat = (size_t)RS_MAX_BINS * p.tiles_pad;
    unsigned int* totals = hist + (size_t)p.n_pass * mat;
    for (int k = 0; k < p.n_pass && n > 0; ++k) {
        const bool last = k == p.n_pass - 1;
        const int bins = 1 << p.bits[k];
        radix_scan_kernel<<<(bins * 32 + 255) / 256, 256, 0, s>>>(hist + k * mat, bins, p.n_tiles, p.tiles_pad, totals); ++*launches;
        unsigned int* hn = last ? nullptr : hist + (k + 1) * mat;
        const int sn = last ? 0 : p.shift[k + 1], bn = last ? 1 : p.bits[k + 1];
        if (p.ipt <= RS_REG_IPT)
            radix_scatter_kernel<true><<<p.n_tiles, RS_THREADS, 0, s>>>(kin, iin, kout, iout, n, p.ipt, p.tiles_pad, p.shift[k], p.bits[k], hist + k * mat, totals, hn, sn, bn,
                                                                       last ? msd_start : nullptr);
        else
            radix_scatter_kernel<false><<<p.n_tiles, RS_THREADS, 0, s>>>(kin, iin, kout, iout, n, p.ipt, p.tiles_pad, p.shift[k], p.bits[k], hist + k * mat, totals, hn, sn, bn,
                                                                        last ? msd_start : nullptr);
        ++*launches;
        unsigned int* t = kin; kin = kout; kout = t;
        iin = iout; iout = (iout == idx_a) ? idx_b : idx_a;
    }
    *keys_sorted_out = kin; *idx_sorted_out = iin;
}

// Sorts a packed cloud into (cell code, original index) order.  grid / hist: written / cleared by icp_launch_pack_cloud on the
// same stream before.  keys_a / keys_b: n entries each (the sorted keys end up in *keys_sorted_out, one of the two);
// idx_a / idx_b: n entries each; hist: icp_radix_hist_words(); msd_start: ICP_MSD_WORDS entries (nullable).
cudaError_t icp_launch_cloud_sort(const float4* pts_in, const float4* nrm_in, int n, int T, const GridParams* grid,
                                  unsigned int* keys_a, unsigned int* keys_b, unsigned int* idx_a, unsigned int* idx_b,
                                  unsigned int* hist, float4* pts_sorted, float4* nrm_sorted, unsigned int* msd_start,
                                  unsigned int** keys_sorted_out, int* msd_shift_out, const IcpLatePack* late, cudaStream_t s, int* n_launches) {
    IcpRadixPlan p; icp_radix_plan(n, T, &p);
    int launches = 0;
    if (msd_shift_out) *msd_shift_out = p.shift[p.n_pass - 1];
    if (n > 0) { keys_kernel<<<(n + KEY_THREADS - 1) / KEY_THREADS, KEY_THREADS, 0, s>>>(pts_in, n, grid, keys_a, p.tile_items, p.tiles_pad, p.shift[0], p.bits[0], hist); ++launches; }
    unsigned int *kin, *iin;
    icp_radix_passes(p, n, keys_a, keys_b, nullptr, idx_a, idx_b, hist, msd_start, s, &kin, &iin, &launches);
    if (n > 0) {
        if (late) {
            // the normal records (nrm_in) are packed only now: their upload had the whole sort to finish
            cudaError_t e = cudaStreamWaitEvent(s, late->ready, 0);
            if (e != cudaSuccess) return e;
            pack_normals_kernel<<<(n + 255) / 256, 256, 0, s>>>(late->nrm, late->rgba, n, late->nrmo); ++launches;
        }
        gather_records_kernel<<<(n + 255) / 256, 256, 0, s>>>(iin, n, pts_in, nrm_in, pts_sorted, nrm_sorted); ++launches;
    }
    if (keys_sorted_out) *keys_sorted_out = kin;
    if (n_launches) *n_launches += launches;
    return cudaGetLastError();
}

__global__ void extract_order_kernel(const float4* __restrict__ pts_sorted, int n, int* __restrict__ order) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) order[i] = __float_as_int(pts_sorted[i].w);
}
cudaError_t icp_launch_extract_order(const float4* pts_sorted, int n, int* order, cudaStream_t s) {
    if (n > 0) extract_order_kernel<<<(n + 255) / 256, 256, 0, s>>>(pts_sorted, n, order);
    return cudaGetLastError();
}

__global__ void fill_int_kernel(int* __restrict__ p, int n, int v) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}
cudaError_t icp_launch_fill_int(int* p, int n, int v, cudaStream_t s) {
    if (n > 0) fill_int_kernel<<<(n + 255) / 256, 256, 0, s>>>(p, n, v);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- first-iteration seeds from the sorted keys
// A query that remembers no neighbour (nn_pos < 0, or `reset`: a new cloud made every remembered neighbour stale) gets the
// point key_seed (search.cuh) reads off the sorted keys at its transformed position.  The search uses a seed only as its
// starting bound and first leaf, so any target point is a valid seed -- a near one lets the first iteration run like the later
// ones (fast path for most queries).
__global__ void seed_from_keys_kernel(const float4* __restrict__ src_pts, int n_src, const DevState* __restrict__ st,
                                      const GridParams* __restrict__ gp, const unsigned int* __restrict__ keys, int n_tgt,
                                      const unsigned int* __restrict__ nonfinite, const unsigned int* __restrict__ msd_start, int msd_shift,
                                      const unsigned int* __restrict__ leaf_rank, int* __restrict__ nn_pos, int* __restrict__ nn_leaf, int reset) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_src) return;
    if (!reset && nn_pos[p] >= 0) return;
    int out_leaf = -1;
    const float4 s = src_pts[p];
    float P[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) P[k] = st->pose[k];
    float x, y, z;
    xform_point(P, s.x, s.y, s.z, x, y, z);
    const int out_pos = key_seed(gp, keys, n_tgt - (int)*nonfinite, msd_start, msd_shift, x, y, z);
    if (out_pos >= 0) out_leaf = (int)(leaf_rank[out_pos + 1] - 1u);
    if (reset || out_pos >= 0) { nn_pos[p] = out_pos; nn_leaf[p] = out_leaf; }
}

cudaError_t icp_launch_seed_from_keys(const float4* src_pts, int n_src, const DevState* st, const GridParams* grid, const unsigned int* keys, int n_tgt,
                                      const unsigned int* nonfinite, const unsigned int* msd_start, int msd_shift, const unsigned int* leaf_rank,
                                      int* nn_pos, int* nn_leaf, int reset, cudaStream_t s) {
    if (n_src <= 0) return cudaSuccess;
    seed_from_keys_kernel<<<(n_src + 255) / 256, 256, 0, s>>>(src_pts, n_src, st, grid, keys, n_tgt, nonfinite, msd_start, msd_shift, leaf_rank,
                                                             nn_pos, nn_leaf, reset);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- BVH over the sorted cloud
// Level 0 (leaves): elements = sorted points, delta(i) = number of leading bits (of T) key[i-1] and key[i] share
// (T when equal; -1 before the first and after the last finite point).  Level l >= 1: elements = nodes of level l-1,
// delta(k) = delta of the first element of node k one level down (the boundary between node k-1 and node k).  The cell-tree
// node of depth d around element i is the maximal run around i whose inner boundaries all have delta >= d; an element starts
// a node of the level iff it is the first element of the SHALLOWEST such run with <= 32 elements.  A finest cell (run of
// equal keys) with more than 32 elements is cut at the positions divisible by 32.  Cell-aligned nodes are pairwise disjoint
// in space -- a search ball meets only the few leaves around it, unlike fixed runs of the Z-curve, whose boxes straddle the
// curve's jumps.
#define LV_THREADS 1024     // one element per thread: the per-element work is a chain of dependent shared-memory loads -- many warps hide it
#define LV_ITEMS 1
#define LV_TILE (LV_THREADS * LV_ITEMS)
#define LV_HALO 32

__device__ __forceinline__ int key_delta(unsigned int a, unsigned int b, int T) {
    const unsigned int x = a ^ b;
    return x ? __clz((int)x) - (32 - T) : T;
}

// flags[i] = 1 iff element i starts a node; tile_count[tile] = flags set in the tile.  count = *count_ptr - *minus_ptr.
template <bool FROM_KEYS>
__global__ void __launch_bounds__(LV_THREADS) level_flags_kernel(const unsigned int* __restrict__ keys, const int* __restrict__ delta_in,
                                                                 const int* count_ptr, int count_host, const unsigned int* __restrict__ minus_ptr,
                                                                 int min_count, int T, unsigned char* __restrict__ flags,
                                                                 unsigned int* __restrict__ tile_count) {
    __shared__ int sd[LV_TILE + 2 * LV_HALO + 1];
    __shared__ unsigned int wsum[LV_THREADS / 32];
    const int count = (count_ptr ? *count_ptr : count_host) - (minus_ptr ? (int)*minus_ptr : 0);
    if (count <= min_count) return;                            // the level below already is the top
    const int n_tiles = (count + LV_TILE - 1) / LV_TILE;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = (long long)tile * LV_TILE;
        __syncthreads();
        // sd[j] = delta(base - LV_HALO + j), j = 0 .. LV_TILE + 2 * LV_HALO
        for (int j = threadIdx.x; j < LV_TILE + 2 * LV_HALO + 1; j += LV_THREADS) {
            const long long i = base - LV_HALO + j;
            int d = -1;
            if (i > 0 && i < count) d = FROM_KEYS ? key_delta(keys[i - 1], keys[i], T) : delta_in[i];
            sd[j] = d;
        }
        __syncthreads();
        unsigned int mine = 0;
#pragma unroll
        for (int k = 0; k < LV_ITEMS; ++k) {
            const int t = k * LV_THREADS + threadIdx.x;
            const long long i = base + t;
            if (i >= count) continue;
            const int* dl = sd + LV_HALO + t;                  // dl[o] = delta(i + o)
            // Element i starts a node iff joining it with its left neighbour -- at the depth d = delta(i) where the two
            // first share a cell -- would make a run of more than 32 elements (the shallowest run with <= 32 elements
            // around i then starts at i).  The run of depth d around i: to the left while delta >= d, to the right alike.
            const int di = dl[0];
            bool f = true;
            if (di >= 0) {
                int size = 2, j = -1;
                while (size <= 32 && dl[j] >= di) { ++size; --j; }
                j = 1;
                while (size <= 32 && dl[j] >= di) { ++size; ++j; }
                f = size > 32 && (di < T || (i & 31) == 0);    // a finest cell with more than 32 elements is cut at multiples of 32
            }
            flags[i] = f ? 1 : 0;
            mine += f ? 1u : 0u;
        }
        mine = __reduce_add_sync(0xFFFFFFFFu, mine);
        if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = mine;
        __syncthreads();
        if (threadIdx.x == 0) { unsigned int s = 0; for (int w = 0; w < LV_THREADS / 32; ++w) s += wsum[w]; tile_count[tile] = s; }
    }
}

// Exclusive scan of the flags: rank[i] = nodes starting before element i (count + 1 entries), start[rank] = i for every flagged element (and start[total] = count), delta_out[rank] = delta of the
// flagged element; the descriptor gains the level.  level 0: rank = leaf_rank, start = leaf_start.
template <bool FROM_KEYS>
__global__ void __launch_bounds__(LV_THREADS) level_rank_kernel(const unsigned int* __restrict__ keys, const int* __restrict__ delta_in,
                                                                const int* count_ptr, int count_host, const unsigned int* __restrict__ minus_ptr,
                                                                int min_count, int T, const unsigned char* __restrict__ flags,
                                                                const unsigned int* __restrict__ tile_count, unsigned int* __restrict__ rank_base,
                                                                unsigned int* __restrict__ start_base, int* __restrict__ delta_out,
                                                                BvhDesc* bvh, int level, int n_alloc) {
    __shared__ unsigned int s_red[LV_THREADS / 32];
    __shared__ unsigned int s_before, s_total;
    const int count = (count_ptr ? *count_ptr : count_host) - (minus_ptr ? (int)*minus_ptr : 0);
    if (level == 0) {
        if (count <= 0) {                                      // empty cloud: a descriptor with no leaves
            if (blockIdx.x == 0 && threadIdx.x == 0) {
                BvhDesc b; b.n_leaves = 0; b.n_levels = 1;
                for (int k = 0; k < ICP_BVH_MAX_LEVELS; ++k) { b.count[k] = 0; b.offset[k] = 0; b.coffset[k] = 0; }
                *bvh = b; start_base[0] = 0u;
            }
            for (int i = blockIdx.x * LV_THREADS + threadIdx.x; i < n_alloc + 2; i += gridDim.x * LV_THREADS) rank_base[i] = 0u;
            return;
        }
    } else if (count <= min_count) return;
    // level >= 1: the level's rank / child arrays start at coffset[level] (set when the level below was finished)
    const int coff = level == 0 ? 0 : bvh->coffset[level];
    unsigned int* rank = rank_base + coff;
    unsigned int* start = start_base + coff;
    const int n_tiles = (count + LV_TILE - 1) / LV_TILE;
    {   // nodes of the whole level
        unsigned int a = 0;
        for (int t = threadIdx.x; t < n_tiles; t += LV_THREADS) a += tile_count[t];
        a = __reduce_add_sync(0xFFFFFFFFu, a);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = a;
        __syncthreads();
        if (threadIdx.x == 0) { unsigned int s = 0; for (int w = 0; w < LV_THREADS / 32; ++w) s += s_red[w]; s_total = s; }
        __syncthreads();
    }
    const unsigned int total = s_total;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const long long base = (long long)tile * LV_TILE;
        __syncthreads();
        unsigned int b = 0;                                    // nodes before this tile
        for (int t = threadIdx.x; t < tile; t += LV_THREADS) b += tile_count[t];
        b = __reduce_add_sync(0xFFFFFFFFu, b);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = b;
        __syncthreads();
        if (threadIdx.x == 0) { unsigned int s = 0; for (int w = 0; w < LV_THREADS / 32; ++w) s += s_red[w]; s_before = s; }
        __syncthreads();
        const unsigned int before = s_before;
        // every thread owns LV_ITEMS consecutive elements
        const long long i0 = base + (long long)threadIdx.x * LV_ITEMS;
        unsigned int f[LV_ITEMS]; unsigned int s = 0;
#pragma unroll
        for (int k = 0; k < LV_ITEMS; ++k) { f[k] = (i0 + k < count) ? flags[i0 + k] : 0u; s += f[k]; }
        unsigned int ex = block_exclusive_scan(s, nullptr) + before;
#pragma unroll
        for (int k = 0; k < LV_ITEMS; ++k) {
            const long long i = i0 + k;
            if (i < count) {
                rank[i] = ex;
                if (f[k]) {
                    start[ex] = (unsigned int)i;
                    if (delta_out) delta_out[ex] = i == 0 ? -1 : (FROM_KEYS ? key_delta(keys[i - 1], keys[i], T) : delta_in[i]);
                }
            }
            ex += f[k];
        }
    }
    // rank[count] = the number of nodes; level 0 keeps leaf_rank defined for every sorted position up to n_alloc + 1
    // (the non-finite points at the end included)
    const long long tail_end = level == 0 ? (long long)n_alloc + 2 : (long long)count + 1;
    for (long long i = (long long)count + blockIdx.x * LV_THREADS + threadIdx.x; i < tail_end; i += (long long)gridDim.x * LV_THREADS) rank[i] = total;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        start[total] = (unsigned int)count;
        if (level == 0) {
            BvhDesc d;
            d.n_leaves = (int)total; d.n_levels = 1;
            for (int k = 0; k < ICP_BVH_MAX_LEVELS; ++k) { d.count[k] = 0; d.offset[k] = 0; d.coffset[k] = 0; }
            d.count[0] = (int)total;
            *bvh = d;
        } else {
            const int n_prev = count;
            bvh->count[level] = (int)total;
            bvh->offset[level] = bvh->offset[level - 1] + n_prev;
            if (level + 1 < ICP_BVH_MAX_LEVELS) bvh->coffset[level + 1] = coff + n_prev + 1;
            bvh->n_levels = level + 1;
        }
    }
}

// All levels above level 1 in ONE single-block launch (a 370k-point cloud has ~1.5k level-1 nodes, then ~90, then ~6):
// per level the flags (same window rule, delta values read from global memory), the scan, the children ranges, the next
// level's delta values and the boxes.  delta_a holds the deltas of level `first_level - 1`'s nodes; the levels ping-pong
// between delta_a and delta_b.
#define UP_THREADS 1024
#define UP_STAGE 4096
__global__ void __launch_bounds__(UP_THREADS) upper_levels_kernel(int* delta_a, int* delta_b, unsigned int* node_rank,
                                                                  unsigned int* child_start, BvhDesc* bvh,
                                                                  float4* box, int T, int first_level) {
    __shared__ unsigned int s_carry, s_total;
    __shared__ BvhDesc sb;
    __shared__ int s_delta[UP_STAGE];                        // the level's deltas when they fit (dependent loads: shared memory is 10x nearer than L2)
    const int lane = threadIdx.x & 31;
    int* din = delta_a; int* dout = delta_b;
    for (int lvl = first_level; lvl < ICP_BVH_MAX_LEVELS; ++lvl) {
        __syncthreads();
        if (threadIdx.x < sizeof(BvhDesc) / 4) reinterpret_cast<int*>(&sb)[threadIdx.x] = reinterpret_cast<volatile int*>(bvh)[threadIdx.x];
        if (threadIdx.x == 0) s_carry = 0u;
        __syncthreads();
        if (sb.n_levels != lvl) return;                        // the level below was not created
        const int n_prev = sb.count[lvl - 1];
        if (n_prev <= 32) return;                              // the level below already is the top
        const int coff = sb.coffset[lvl];
        unsigned int* rank = node_rank + coff;
        unsigned int* start = child_start + coff;
        const bool staged = n_prev <= UP_STAGE;
        if (staged) for (int j = threadIdx.x; j < n_prev; j += UP_THREADS) s_delta[j] = din[j];
        __syncthreads();
        for (int base = 0; base < n_prev; base += UP_THREADS) {
            const int i = base + threadIdx.x;
            unsigned int f = 0u;
            if (i < n_prev) {
                // the rule of level_flags_kernel; delta(j) of this level's elements, -1 outside (1 .. n_prev - 1)
                auto dl = [&](int o) -> int { const int j = i + o; return (j > 0 && j < n_prev) ? (staged ? s_delta[j] : din[j]) : -1; };
                const int di = dl(0);
                f = 1u;
                if (di >= 0) {
                    int size = 2, j = -1;
                    while (size <= 32 && dl(j) >= di) { ++size; --j; }
                    j = 1;
                    while (size <= 32 && dl(j) >= di) { ++size; ++j; }
                    f = (size > 32 && (di < T || (i & 31) == 0)) ? 1u : 0u;
                }
            }
            const unsigned int ex = block_exclusive_scan(f, &s_total) + s_carry;
            if (i < n_prev) {
                rank[i] = ex;
                if (f) { start[ex] = (unsigned int)i; dout[ex] = i == 0 ? -1 : (staged ? s_delta[i] : din[i]); }
            }
            __syncthreads();
            if (threadIdx.x == 0) s_carry += s_total;
            __syncthreads();
        }
        const int total = (int)s_carry;
        if (threadIdx.x == 0) {
            rank[n_prev] = (unsigned int)total;
            start[total] = (unsigned int)n_prev;
            bvh->count[lvl] = total;
            bvh->offset[lvl] = sb.offset[lvl - 1] + n_prev;
            if (lvl + 1 < ICP_BVH_MAX_LEVELS) bvh->coffset[lvl + 1] = coff + n_prev + 1;
            bvh->n_levels = lvl + 1;
            __threadfence();
        }
        __syncthreads();
        // boxes of the new level: one warp per node over its (<= 32) child boxes
        const int off_prev = sb.offset[lvl - 1], off = sb.offset[lvl - 1] + n_prev;
        for (int node = threadIdx.x >> 5; node < total; node += UP_THREADS / 32) {
            float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
            unsigned int clo[3] = {255u, 255u, 255u}, chi[3] = {0u, 0u, 0u};
            const unsigned int c = start[node] + lane;
            if (c < start[node + 1]) {
                const float4 u = box[2 * (size_t)(off_prev + c)], v = box[2 * (size_t)(off_prev + c) + 1];
                lo[0] = u.x; lo[1] = u.y; lo[2] = u.z; hi[0] = v.x; hi[1] = v.y; hi[2] = v.z;
                const unsigned int cu = __float_as_uint(u.w), cv = __float_as_uint(v.w);
#pragma unroll
                for (int k = 0; k < 3; ++k) { clo[k] = (cu >> (8 * k)) & 0xFFu; chi[k] = (cv >> (8 * k)) & 0xFFu; }
            }
#pragma unroll
            for (int k = 0; k < 3; ++k) { clo[k] = __reduce_min_sync(0xFFFFFFFFu, clo[k]); chi[k] = __reduce_max_sync(0xFFFFFFFFu, chi[k]); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], __shfl_xor_sync(0xFFFFFFFFu, lo[k], o)); hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xFFFFFFFFu, hi[k], o)); }
            if (lane == 0) {
                box[2 * (size_t)(off + node)] = make_float4(lo[0], lo[1], lo[2], __uint_as_float(clo[0] | (clo[1] << 8) | (clo[2] << 16)));
                box[2 * (size_t)(off + node) + 1] = make_float4(hi[0], hi[1], hi[2], __uint_as_float(chi[0] | (chi[1] << 8) | (chi[2] << 16)));
            }
        }
        int* t = din; din = dout; dout = t;
    }
}

// one warp per node (grid-stride): level 0 reads the leaf's points, level l > 0 reads its (<= 32) child boxes
// The w components of the two box entries carry the node's COLOUR range (min / max of r, g, b as packed bytes), which the
// 6-D colour search adds to its lower bounds (search.cuh: box_dist2c).
// Level 0 also re-orders every leaf's records by ORIGINAL index (they arrive in (cell code, original index) order): a scan of
// the leaf in storage order with a strict '<' on the distance then returns the lowest original index among equal distances --
// contract D2 inside a leaf without comparing indices per candidate (knn.cu: thread_scan_leaf).
__global__ void bvh_level_kernel(float4* __restrict__ pts, float4* __restrict__ nrm, const unsigned int* __restrict__ leaf_start,
                                 const unsigned int* __restrict__ child_start, const BvhDesc* __restrict__ bvh, float4* __restrict__ box,
                                 int level) {
    const BvhDesc b = *bvh;
    if (level >= b.n_levels) return;
    const int lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
    const int count = b.count[level], offset = b.offset[level];
    for (int node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; node < count; node += warps) {
        float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
        unsigned int clo[3] = {255u, 255u, 255u}, chi[3] = {0u, 0u, 0u};
        if (level == 0) {
            const unsigned int ls = leaf_start[node], i = ls + lane;
            const bool in = i < leaf_start[node + 1];
            float4 p = make_float4(0.f, 0.f, 0.f, 0.f), m = p;
            if (in) {
                p = pts[i]; m = nrm[i]; lo[0] = hi[0] = p.x; lo[1] = hi[1] = p.y; lo[2] = hi[2] = p.z;
                const unsigned int c = __float_as_uint(m.w);
#pragma unroll
                for (int k = 0; k < 3; ++k) clo[k] = chi[k] = (c >> (8 * k)) & 0xFFu;
            }
            // rank of this lane's record among the leaf's by original index (unique), then the in-place permutation
            const unsigned int mine = in ? __float_as_uint(p.w) : 0xFFFFFFFFu;
            unsigned int rank = 0;
#pragma unroll
            for (int l = 0; l < 32; ++l) rank += __shfl_sync(0xFFFFFFFFu, mine, l) < mine ? 1u : 0u;
            __syncwarp();                                    // every record of the leaf is in registers before any is overwritten
            if (in) { pts[ls + rank] = p; nrm[ls + rank] = m; }
        } else {
            const unsigned int c = child_start[b.coffset[level] + node] + lane;
            if (c < child_start[b.coffset[level] + node + 1]) {
                const float4 u = box[2 * (size_t)(b.offset[level - 1] + c)], v = box[2 * (size_t)(b.offset[level - 1] + c) + 1];
                lo[0] = u.x; lo[1] = u.y; lo[2] = u.z; hi[0] = v.x; hi[1] = v.y; hi[2] = v.z;
                const unsigned int cu = __float_as_uint(u.w), cv = __float_as_uint(v.w);
#pragma unroll
                for (int k = 0; k < 3; ++k) { clo[k] = (cu >> (8 * k)) & 0xFFu; chi[k] = (cv >> (8 * k)) & 0xFFu; }
            }
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) { clo[k] = __reduce_min_sync(0xFFFFFFFFu, clo[k]); chi[k] = __reduce_max_sync(0xFFFFFFFFu, chi[k]); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int k = 0; k < 3; ++k) { lo[k] = fminf(lo[k], __shfl_xor_sync(0xFFFFFFFFu, lo[k], o)); hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xFFFFFFFFu, hi[k], o)); }
        if (lane == 0) {
            box[2 * (size_t)(offset + node)] = make_float4(lo[0], lo[1], lo[2], __uint_as_float(clo[0] | (clo[1] << 8) | (clo[2] << 16)));
            box[2 * (size_t)(offset + node) + 1] = make_float4(hi[0], hi[1], hi[2], __uint_as_float(chi[0] | (chi[1] << 8) | (chi[2] << 16)));
        }
    }
}

// ---------------------------------------------------------------------------- voxel pyramid levels
// ICP_GPU_PYRAMID_VOXEL: a pyramid level keeps ONE point per occupied cell of the source grid at depth D -- the valid
// (finite point and normal) point with the lowest original index -- instead of every f-th point of the scan order
// (PointCloud.h:325-343).  The level is delivered as a selection mask (bit per original index).
__global__ void voxel_min_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm, int n, const GridParams* __restrict__ gp,
                                 int T, int D, unsigned int* __restrict__ table) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i], m = nrm[i];
    if (!finite3(p.x, p.y, p.z) || !finite3(m.x, m.y, m.z)) return;
    const GridParams g = *gp;
    atomicMin(&table[cell_code(g, p.x, p.y, p.z) >> (T - D)], (unsigned int)__float_as_int(p.w));
}
__global__ void voxel_mask_kernel(const float4* __restrict__ pts, const float4* __restrict__ nrm, int n, const GridParams* __restrict__ gp,
                                  int T, int D, const unsigned int* __restrict__ table, unsigned int* __restrict__ mask) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 p = pts[i], m = nrm[i];
    if (!finite3(p.x, p.y, p.z) || !finite3(m.x, m.y, m.z)) return;
    const GridParams g = *gp;
    const unsigned int o = (unsigned int)__float_as_int(p.w);
    if (table[cell_code(g, p.x, p.y, p.z) >> (T - D)] == o) atomicOr(&mask[o >> 5], 1u << (o & 31u));
}

cudaError_t icp_launch_voxel_level(const float4* pts_sorted, const float4* nrm_sorted, int n, const GridParams* grid, int T, int D,
                                   unsigned int* table, unsigned int* mask, size_t mask_words, cudaStream_t s, int* n_launches) {
    cudaError_t e;
    if ((e = cudaMemsetAsync(table, 0xFF, sizeof(unsigned int) * ((size_t)1 << D), s)) != cudaSuccess) return e;
    if ((e = cudaMemsetAsync(mask, 0, sizeof(unsigned int) * mask_words, s)) != cudaSuccess) return e;
    if (n > 0) {
        voxel_min_kernel<<<(n + 255) / 256, 256, 0, s>>>(pts_sorted, nrm_sorted, n, grid, T, D, table);
        voxel_mask_kernel<<<(n + 255) / 256, 256, 0, s>>>(pts_sorted, nrm_sorted, n, grid, T, D, table, mask);
        if (n_launches) *n_launches += 2;
    }
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------- leaf adjacency
// One warp per leaf l: all other leaves whose box meets box(l) inflated by R, found by a box query on the BVH
// (lane = child).  R starts at ADJ_R_FACTOR times the leaf's largest extent and is halved until the list fits in 32 entries.
#define ADJ_WARPS 4
#define ADJ_R_FACTOR 2.0f      // 1.5 / 3 / 4 measured no different (round 2, DESIGN §4)
__device__ __forceinline__ bool boxes_meet(const float* lo, const float* hi, const float4 blo, const float4 bhi) {
    return blo.x <= hi[0] && bhi.x >= lo[0] && blo.y <= hi[1] && bhi.y >= lo[1] && blo.z <= hi[2] && bhi.z >= lo[2];
}

__global__ void __launch_bounds__(ADJ_WARPS * 32) leaf_adjacency_kernel(const BvhDesc* __restrict__ bvh, const float4* __restrict__ box,
                                                                         const unsigned int* __restrict__ child_start,
                                                                         unsigned int* __restrict__ adj, float4* __restrict__ adj_box,
                                                                         int capacity, int lv,
                                                                         const unsigned int* __restrict__ node_rank, const unsigned int* __restrict__ adj1,
                                                                         const float4* __restrict__ adj1_box, int adj1_capacity, float* __restrict__ adj_gap) {
    __shared__ unsigned int s_node[ADJ_WARPS][32 * ICP_BVH_MAX_LEVELS];
    __shared__ unsigned int s_list[ADJ_WARPS][64];
    const BvhDesc b = *bvh;
    const unsigned int FULL = 0xFFFFFFFFu;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, warps = (gridDim.x * blockDim.x) >> 5;
    // lv = 0: lists of leaves (the node itself excluded: a search has scanned it already); lv = 1: lists of level-1 nodes
    // (the node itself included)
    if (lv >= b.n_levels) return;
    const int n_leaves = min(b.count[lv], capacity);
    const int top_level = b.n_levels - 1;
    unsigned int* st = s_node[wid]; unsigned int* list = s_list[wid];
    const unsigned int lt = (1u << lane) - 1u;
    for (int l = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; l < n_leaves; l += warps) {
        const float4 mlo = box[2 * (size_t)(b.offset[lv] + l)], mhi = box[2 * (size_t)(b.offset[lv] + l) + 1];
        float R = ADJ_R_FACTOR * fmaxf(fmaxf(mhi.x - mlo.x, mhi.y - mlo.y), mhi.z - mlo.z);
        int count = 0; bool ok = false;
        // Leaves (lv = 0) with the level-1 lists already built: while the leaf's inflated box lies inside the inflated box of its
        // level-1 node m, every leaf that meets it is a child of a node of m's list -- two rounds of box tests (the <= 32 nodes
        // of the list, then the children of those that meet) instead of a walk from the root.
        int pm = -1, pna = 0; float4 plo = make_float4(0.f, 0.f, 0.f, 0.f), phi = plo;
        if (lv == 0 && adj1 && b.n_levels >= 2) {
            pm = (int)(node_rank[b.coffset[1] + l + 1] - 1u);
            if (pm < adj1_capacity) { plo = adj1_box[2 * (size_t)pm]; phi = adj1_box[2 * (size_t)pm + 1]; pna = __float_as_int(plo.w); } else pm = -1;
        }
        for (int attempt = 0; attempt < 6 && !ok; ++attempt, R *= 0.5f) {
            const float lo[3] = {__fsub_rd(mlo.x, R), __fsub_rd(mlo.y, R), __fsub_rd(mlo.z, R)};
            const float hi[3] = {__fadd_ru(mhi.x, R), __fadd_ru(mhi.y, R), __fadd_ru(mhi.z, R)};
            count = 0; ok = true;
            if (pm >= 0 && lo[0] >= plo.x && lo[1] >= plo.y && lo[2] >= plo.z && hi[0] <= phi.x && hi[1] <= phi.y && hi[2] <= phi.z) {   // never true for the inverted "no list" box
                unsigned int cfirst = 0u, clast = 0u; bool keep1 = false;
                if (lane < pna) {
                    const unsigned int node = adj1[(size_t)pm * 32 + lane];
                    keep1 = boxes_meet(lo, hi, box[2 * (size_t)(b.offset[1] + node)], box[2 * (size_t)(b.offset[1] + node) + 1]);
                    cfirst = child_start[b.coffset[1] + node]; clast = child_start[b.coffset[1] + node + 1];
                }
                unsigned int m1 = __ballot_sync(FULL, keep1);
                // the children of the nodes that meet, one node per round; the next node's boxes are requested before the
                // current ones are used (the rounds are chains of dependent L2 loads: two in flight)
                float4 nlo = make_float4(0.f, 0.f, 0.f, 0.f), nhi = nlo; unsigned int nc = 0u, nlast = 0u;
                bool more = m1 != 0u;                          // warp-uniform: a node's boxes are in flight
                if (more) {
                    const int src = __ffs((int)m1) - 1; m1 &= m1 - 1u;
                    nc = __shfl_sync(FULL, cfirst, src) + lane; nlast = __shfl_sync(FULL, clast, src);
                    if (nc < nlast) { nlo = box[2 * (size_t)nc]; nhi = box[2 * (size_t)nc + 1]; }
                }
                while (more && ok) {
                    const float4 clo = nlo, chi = nhi; const unsigned int c = nc, last = nlast;
                    more = m1 != 0u;
                    if (more) {
                        const int src = __ffs((int)m1) - 1; m1 &= m1 - 1u;
                        nc = __shfl_sync(FULL, cfirst, src) + lane; nlast = __shfl_sync(FULL, clast, src);
                        if (nc < nlast) { nlo = box[2 * (size_t)nc]; nhi = box[2 * (size_t)nc + 1]; }
                    }
                    const bool keep = c < last && c != (unsigned int)l && boxes_meet(lo, hi, clo, chi);
                    const unsigned int mk = __ballot_sync(FULL, keep);
                    if (count + __popc(mk) > 32) { ok = false; break; }
                    if (keep) list[count + __popc(mk & lt)] = c;
                    count += __popc(mk);
                }
                __syncwarp();
                if (ok) break;                                 // R stays the one this list was built with
                continue;
            }
            int top = 0;
            // virtual root over the top level, then depth-first; leaves are appended to the list
            for (unsigned int base = 0; base < (unsigned int)b.count[top_level] && ok; base += 32) {
                int L = top_level; unsigned int first = base, last = min(base + 32u, (unsigned int)b.count[top_level]);
                for (;;) {
                    const unsigned int c = first + lane;
                    bool keep = false;
                    if (c < last) keep = boxes_meet(lo, hi, box[2 * (size_t)(b.offset[L] + c)], box[2 * (size_t)(b.offset[L] + c) + 1]);
                    if (L == lv && lv == 0) keep = keep && c != (unsigned int)l;
                    const unsigned int mk = __ballot_sync(FULL, keep);
                    if (L == lv) {
                        if (count + __popc(mk) > 32) { ok = false; break; }
                        if (keep) list[count + __popc(mk & lt)] = c;
                        count += __popc(mk);
                    } else {
                        if (keep) st[top + __popc(mk & lt)] = ((unsigned int)L << 27) | c;
                        top += __popc(mk);
                    }
                    __syncwarp();
                    if (top == 0) break;
                    --top;
                    const unsigned int id = st[top];
                    __syncwarp();
                    const int lvl = (int)(id >> 27); const unsigned int j = id & 0x7FFFFFFu;
                    first = child_start[b.coffset[lvl] + j]; last = child_start[b.coffset[lvl] + j + 1];
                    L = lvl - 1;
                }
            }
            if (ok) break;
        }
        __syncwarp();
        if (adj_gap && ok) {
            // Entries in the order of their squared box-to-box gap to this node (rounded down), the gaps stored with them: a search
            // whose best candidate p lies in this node's box at distance r from the query needs only the entries with gap <= 2r
            // (a point x within r of the query is within 2r of p, and gap <= |p - x|), and stops at the first one beyond.
            float gq = INFINITY; unsigned int e = 0u;
            if (lane < count) {
                e = list[lane];
                const float4 elo = box[2 * (size_t)(b.offset[lv] + e)], ehi = box[2 * (size_t)(b.offset[lv] + e) + 1];
                const float gx = fmaxf(fmaxf(__fsub_rd(elo.x, mhi.x), __fsub_rd(mlo.x, ehi.x)), 0.f);
                const float gy = fmaxf(fmaxf(__fsub_rd(elo.y, mhi.y), __fsub_rd(mlo.y, ehi.y)), 0.f);
                const float gz = fmaxf(fmaxf(__fsub_rd(elo.z, mhi.z), __fsub_rd(mlo.z, ehi.z)), 0.f);
                gq = __fadd_rd(__fadd_rd(__fmul_rd(gx, gx), __fmul_rd(gy, gy)), __fmul_rd(gz, gz));
            }
            int rank = 0;
#pragma unroll
            for (int k = 0; k < 32; ++k) {
                const float gk = __shfl_sync(FULL, gq, k);
                rank += (gk < gq || (gk == gq && k < lane)) ? 1 : 0;
            }
            if (lane < count) { adj[(size_t)l * 32 + rank] = e; adj_gap[(size_t)l * 32 + rank] = gq; }
        } else if (lane < count && ok) adj[(size_t)l * 32 + lane] = list[lane];
        if (lane == 0) {
            // the inflated box exactly as the query above used it (so that "ball inside this box" implies "every leaf the
            // ball meets is in the list"); inverted when there is no list
            if (ok) {
                adj_box[2 * (size_t)l] = make_float4(__fsub_rd(mlo.x, R), __fsub_rd(mlo.y, R), __fsub_rd(mlo.z, R), __int_as_float(count));
                adj_box[2 * (size_t)l + 1] = make_float4(__fadd_ru(mhi.x, R), __fadd_ru(mhi.y, R), __fadd_ru(mhi.z, R), 0.f);
            } else {
                adj_box[2 * (size_t)l] = make_float4(INFINITY, INFINITY, INFINITY, __int_as_float(0));
                adj_box[2 * (size_t)l + 1] = make_float4(-INFINITY, -INFINITY, -INFINITY, 0.f);
            }
        }
        __syncwarp();
    }
}

// level 1 first; the level-0 call then takes the level-1 lists (node_rank, adj1, adj1_box)
cudaError_t icp_launch_leaf_adjacency(const BvhDesc* bvh_dev, const float4* box, const unsigned int* child_start, unsigned int* adj,
                                      float4* adj_box, int capacity, int level, const unsigned int* node_rank, const unsigned int* adj1,
                                      const float4* adj1_box, int adj1_capacity, int n_sms, cudaStream_t s, int* n_launches, float* adj_gap) {
    long long nb = ((long long)capacity + ADJ_WARPS - 1) / ADJ_WARPS;
    if (nb > 16ll * n_sms) nb = 16ll * n_sms;
    if (nb < 1) nb = 1;
    leaf_adjacency_kernel<<<(int)nb, ADJ_WARPS * 32, 0, s>>>(bvh_dev, box, child_start, adj, adj_box, capacity, level,
                                                             node_rank, adj1, adj1_box, adj1_capacity, adj_gap);
    if (n_launches) *n_launches += 1;
    return cudaGetLastError();
}

size_t icp_bvh_max_nodes(int n) {
    // worst case: every point its own leaf, and every upper level only halves the node count until the cap
    return (size_t)(n > 0 ? n : 1) * 2 + 64;
}

// Tight-box BVH over the sorted cloud.  keys: the sorted keys; nonfinite: device count of the points past the last cell.
// leaf_rank: n + 2 entries (kept: maps a sorted position to its leaf); leaf_start: n + 2; node_rank / child_start:
// icp_bvh_max_nodes(n) + ICP_BVH_MAX_LEVELS entries each; flags: n bytes; tile_count: n / 1024 + 2; delta_a / delta_b: n + 2 each.
cudaError_t icp_launch_bvh_build(float4* pts_sorted, float4* nrm_sorted, int n, int T, const unsigned int* keys,
                                 const unsigned int* nonfinite, unsigned char* flags, unsigned int* tile_count,
                                 int* delta_a, int* delta_b, unsigned int* leaf_rank, unsigned int* leaf_start, unsigned int* node_rank,
                                 unsigned int* child_start, BvhDesc* bvh_dev, float4* box, int n_sms, cudaStream_t s, int* n_launches) {
    int launches = 0;
    const int n1 = n > 0 ? n : 1;
    const int tiles0 = (n1 + LV_TILE - 1) / LV_TILE;
    // level 0: leaves
    level_flags_kernel<true><<<tiles0, LV_THREADS, 0, s>>>(keys, nullptr, nullptr, n, nonfinite, 0, T, flags, tile_count); ++launches;
    level_rank_kernel<true><<<tiles0, LV_THREADS, 0, s>>>(keys, nullptr, nullptr, n, nonfinite, 0, T, flags, tile_count, leaf_rank, leaf_start, delta_a,
                                                          bvh_dev, 0, n); ++launches;
    long long nb0 = ((long long)n1 + 7) / 8; if (nb0 > 8ll * n_sms) nb0 = 8ll * n_sms;
    bvh_level_kernel<<<(int)nb0, 256, 0, s>>>(pts_sorted, nrm_sorted, leaf_start, child_start, bvh_dev, box, 0); ++launches;
    // level 1: elements = leaves (a healthy cloud has ~n/16 of them; the kernels loop if there are more)
    int tiles1 = (n1 / 8 + LV_TILE - 1) / LV_TILE; if (tiles1 < 1) tiles1 = 1; if (tiles1 > 4 * n_sms) tiles1 = 4 * n_sms;
    const int* leaves_dev = &bvh_dev->count[0];
    level_flags_kernel<false><<<tiles1, LV_THREADS, 0, s>>>(nullptr, delta_a, leaves_dev, 0, nullptr, 32, T, flags, tile_count); ++launches;
    level_rank_kernel<false><<<tiles1, LV_THREADS, 0, s>>>(nullptr, delta_a, leaves_dev, 0, nullptr, 32, T, flags, tile_count, node_rank, child_start, delta_b,
                                                           bvh_dev, 1, 0); ++launches;
    const int nb1 = 2 * n_sms;
    bvh_level_kernel<<<nb1, 256, 0, s>>>(pts_sorted, nrm_sorted, leaf_start, child_start, bvh_dev, box, 1); ++launches;
    // levels >= 2: one block
    upper_levels_kernel<<<1, UP_THREADS, 0, s>>>(delta_b, delta_a, node_rank, child_start, bvh_dev, box, T, 2); ++launches;
    if (n_launches) *n_launches += launches;
    return cudaGetLastError();
}
