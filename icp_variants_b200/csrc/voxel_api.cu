// voxel_api.cu -- the host side of voxel-grid downsampling (icp_gpu_voxel_downsample[_dev]): B concatenated clouds filtered in one
// pass of voxel.cu's kernels, the result returned and, in the TARGET / SOURCE roles, made the context's cloud through set_cloud as
// icp_gpu_cloud_from_depth does.  Host code only.
//
//   inputs   the concatenated clouds and offsets (one upload each, or read in place), the offsets read back and checked
//   keys     each point's voxel and each cloud's bounds; the bounds read back (the refusals, the key's field widths)
//   sort     by (cloud, voxel) key, one 32-bit word at a time (one word up to 31 key bits)
//   reduce   voxel heads compacted, one centroid per voxel, off_out; the count read back
#include "context.cuh"
#include <limits.h>
#include <math.h>

// Bits of an unsigned field that holds 0 .. m.
static int field_bits(long long m) { int b = 0; while (b < 63 && (1ll << b) <= m) ++b; return b; }

#define VOX_MAX_SPAN (1ll << 21)         // voxels on an axis of one cloud: three fields and the cloud index stay within three words

static int voxel_downsample(icp_gpu_ctx* ctx, int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off,
                            float voxel_size, int role, float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out, bool dev) {
    if (!ctx) return ICP_GPU_E_ARG;
    if (n_clouds < 0) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: n_clouds %d", n_clouds);
    if (!(isfinite(voxel_size) && voxel_size > 0.f)) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: voxel size %g (finite and > 0)", (double)voxel_size);
    if (role < ICP_GPU_CLOUD_TARGET || role > ICP_GPU_CLOUD_ONLY) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: role %d", role);
    if (role != ICP_GPU_CLOUD_ONLY && n_clouds != 1)
        return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: the TARGET and SOURCE roles take one cloud, not %d", n_clouds);
    if ((nrm_out && !nrm) || (rgba_out && !rgba)) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: nrm_out / rgba_out without nrm / rgba");
    if (n_clouds > 0 && (!xyz || !off || (role == ICP_GPU_CLOUD_ONLY && (!xyz_out || !off_out))))
        return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: xyz and off are required, and with role ONLY xyz_out and off_out");
    if (int rc = enter(ctx)) return rc;
    if (n_clouds == 0) return ICP_GPU_OK;
    const size_t B = (size_t)n_clouds;
    std::vector<int64_t> ho(B + 1);
    if (dev) {
        CU(cudaMemcpyAsync(ho.data(), off, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    } else {
        memcpy(ho.data(), off, (B + 1) * 8);
    }
    if (ho[0] != 0) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: the offsets must start at 0 (%lld)", (long long)ho[0]);
    for (size_t b = 0; b < B; ++b)
        if (ho[b + 1] < ho[b]) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: offsets of cloud %zu are not monotone", b);
    const long long n_all = ho[B];
    if (n_all > 0x7fffffff / 4) return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: %lld points in all (limit %d)", n_all, 0x7fffffff / 4);
    const int n = (int)n_all;
    const size_t n1 = (size_t)(n > 0 ? n : 1);

    // io: inputs (host form), the offsets, outputs (points, normals, colours, off_out); tmp: records, bounds, sort, compaction
    enum { I_XYZ, I_NRM, I_RGBA, I_OFF, O_XYZ, O_NRM, O_RGBA, O_OFF, IO_N };
    size_t isz[IO_N] = {dev ? 0 : n1 * 12, dev || !nrm ? 0 : n1 * 12, dev || !rgba ? 0 : n1 * 4, dev ? 0 : (B + 1) * 8,
                        n1 * 12, nrm ? n1 * 12 : 0, rgba ? n1 * 4 : 0, (B + 1) * 8};
    enum { T_VOX, T_BOUNDS, T_KEYS_A, T_KEYS_B, T_IDX_A, T_IDX_B, T_HIST, T_FLAG, T_BLOCKS, T_RUN, T_N };
    const size_t tsz[T_N] = {n1 * 16, B * 7 * 4 + 4, n1 * 4, n1 * 4, n1 * 4, n1 * 4, icp_radix_hist_words(n, 31) * 4, (n1 + 1) * 4,
                             (n1 / ICP_FLAG_SCAN_BLOCK + 2) * 4, (n1 + 1) * 4};
    size_t io[IO_N], to[T_N];
    if (ensure(ctx, ctx->vox_io, pack_segments(isz, IO_N, io), false) || ensure(ctx, ctx->vox_tmp, pack_segments(tsz, T_N, to), false))
        return ICP_GPU_E_CUDA;
    char* iob = (char*)ctx->vox_io.p; char* tb = (char*)ctx->vox_tmp.p;
    const float* dx = xyz; const float* dn = nrm; const uint8_t* dc = rgba; const long long* doff = (const long long*)off;
    if (!dev) {
        if (n > 0) CU(cudaMemcpyAsync(iob + io[I_XYZ], xyz, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
        if (n > 0 && nrm) CU(cudaMemcpyAsync(iob + io[I_NRM], nrm, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
        if (n > 0 && rgba) CU(cudaMemcpyAsync(iob + io[I_RGBA], rgba, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaMemcpyAsync(iob + io[I_OFF], off, (B + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
        dx = (const float*)(iob + io[I_XYZ]); dn = nrm ? (const float*)(iob + io[I_NRM]) : nullptr;
        dc = rgba ? (const uint8_t*)(iob + io[I_RGBA]) : nullptr; doff = (const long long*)(iob + io[I_OFF]);
    }
    // the device form writes straight into the caller's outputs where there are some
    float* ox = dev && xyz_out ? xyz_out : (float*)(iob + io[O_XYZ]);
    float* on = !nrm ? nullptr : dev && nrm_out ? nrm_out : (float*)(iob + io[O_NRM]);
    uint8_t* oc = !rgba ? nullptr : dev && rgba_out ? rgba_out : (uint8_t*)(iob + io[O_RGBA]);
    long long* oo = dev && off_out ? (long long*)off_out : (long long*)(iob + io[O_OFF]);
    CU(cudaMemsetAsync(oo, 0, (B + 1) * 8, ctx->stream));

    int launches = 0;
    unsigned int n_vox = 0;
    if (n > 0) {
        int4* vox = (int4*)(tb + to[T_VOX]);
        int* bounds = (int*)(tb + to[T_BOUNDS]);
        unsigned int* bad = (unsigned int*)(bounds + 6 * B);
        std::vector<int> hb(B * 7);
        for (size_t b = 0; b < B; ++b) for (int a = 0; a < 6; ++a) hb[6 * b + a] = a < 3 ? INT_MAX : INT_MIN;
        for (size_t b = 0; b < B; ++b) hb[6 * B + b] = 0;
        CU(cudaMemcpyAsync(bounds, hb.data(), B * 7 * 4, cudaMemcpyHostToDevice, ctx->stream));
        const float inv = 1.0f / voxel_size;                       // V1: PCL's inverse_leaf_size_, rounded to fp32
        CU(icp_launch_voxel_coords(dx, n, doff, n_clouds, inv, vox, bounds, bad, ctx->stream, &launches));
        CU(cudaMemcpyAsync(hb.data(), bounds, B * 7 * 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        long long span[3] = {0, 0, 0};
        for (size_t b = 0; b < B; ++b) {
            if (hb[6 * B + b]) { ctx->stats.n_kernel_launches += (uint64_t)launches; return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: cloud %zu has a voxel index outside int32", b); }
            if (hb[6 * b] > hb[6 * b + 3]) continue;               // no finite point
            for (int a = 0; a < 3; ++a) {
                const long long m = (long long)hb[6 * b + 3 + a] - hb[6 * b + a];
                if (m + 1 > VOX_MAX_SPAN) {
                    ctx->stats.n_kernel_launches += (uint64_t)launches;
                    return fail(ctx, ICP_GPU_E_ARG, "voxel_downsample: cloud %zu spans %lld voxels on %c (limit 2^21)", b, m + 1, "xyz"[a]);
                }
                if (m > span[a]) span[a] = m;
            }
        }
        VoxKeyLayout L;
        L.bx = field_bits(span[0]); L.by = field_bits(span[1]); L.bz = field_bits(span[2]); L.bc = field_bits((long long)B - 1);
        const int K = L.bx + L.by + L.bz + L.bc;
        L.n_words = K <= 31 ? 1 : 1 + (K - 31 + 31) / 32;
        L.top_bits = K - 32 * (L.n_words - 1);
        unsigned int* idx = nullptr;
        CU(icp_launch_voxel_sort(vox, n, bounds, L, (unsigned int*)(tb + to[T_KEYS_A]), (unsigned int*)(tb + to[T_KEYS_B]),
                                 (unsigned int*)(tb + to[T_IDX_A]), (unsigned int*)(tb + to[T_IDX_B]), (unsigned int*)(tb + to[T_HIST]), ctx->stream,
                                 &idx, &launches));
        unsigned int* total = (unsigned int*)(tb + to[T_BLOCKS]) + n1 / ICP_FLAG_SCAN_BLOCK + 1;
        CU(icp_launch_voxel_centroids(idx, vox, n, dx, dn, dc, n_clouds, (unsigned int*)(tb + to[T_FLAG]), (unsigned int*)(tb + to[T_BLOCKS]), total,
                                      (unsigned int*)(tb + to[T_RUN]), ox, on, oc, oo, ctx->stream, &launches));
        CU(cudaMemcpyAsync(&n_vox, total, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    }
    ctx->stats.n_kernel_launches += (uint64_t)launches;
    if (!dev) {
        if (n_vox > 0 && xyz_out) CU(cudaMemcpyAsync(xyz_out, ox, (size_t)n_vox * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (n_vox > 0 && nrm_out) CU(cudaMemcpyAsync(nrm_out, on, (size_t)n_vox * 12, cudaMemcpyDeviceToHost, ctx->stream));
        if (n_vox > 0 && rgba_out) CU(cudaMemcpyAsync(rgba_out, oc, (size_t)n_vox * 4, cudaMemcpyDeviceToHost, ctx->stream));
        if (off_out) CU(cudaMemcpyAsync(off_out, oo, (B + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    }
    int rc = ICP_GPU_OK;
    if (role != ICP_GPU_CLOUD_ONLY) rc = set_cloud(ctx, role == ICP_GPU_CLOUD_TARGET, ox, on, oc, (int64_t)n_vox, true);
    CU(cudaStreamSynchronize(ctx->stream));
    return rc;
}

int icp_gpu_voxel_downsample(icp_gpu_ctx* ctx, int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off,
                             float voxel_size, int role, float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out) {
    return voxel_downsample(ctx, n_clouds, xyz, nrm, rgba, off, voxel_size, role, xyz_out, nrm_out, rgba_out, off_out, false);
}
int icp_gpu_voxel_downsample_dev(icp_gpu_ctx* ctx, int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off,
                                 float voxel_size, int role, float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out) {
    return voxel_downsample(ctx, n_clouds, xyz, nrm, rgba, off, voxel_size, role, xyz_out, nrm_out, rgba_out, off_out, true);
}
