/*
 * voxel_reference.c -- CPU restatement of the device's voxel-grid downsampling (icp_gpu_voxel_downsample, csrc/voxel.cu), written
 * from DESIGN.md section 4 rows V1-V5 as literally as C allows.  TEST INFRASTRUCTURE ONLY: tests/voxel_reference.py compiles it with
 * -O2 -ffp-contract=off -fno-fast-math (no contraction of the products into FMAs) and tests/test_voxel_reference.py pins it against a
 * separate numpy / Python-float restatement.
 *
 * Cloud b = points [off[b], off[b+1]); one point per occupied voxel (floorf(x * (1.0f / voxel_size)) per axis, finite points only),
 * clouds in order, voxels in ascending (iz, iy, ix); coordinates = fp64 sequential sum in ascending index / count, normals = fp64 sum
 * of the finite normals / its norm (-inf where none or norm 0), colours (2 sum + k) / 2k.  nrm / rgba (and their outputs) nullable;
 * outputs need room for off[n_clouds] points.  Returns 0, or -1 - b when a voxel index of cloud b does not fit int32.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>

static int finite3(const float* p) { return isfinite(p[0]) && isfinite(p[1]) && isfinite(p[2]); }

typedef struct { int32_t v[3]; int64_t idx; } vref_pt;
static int vref_pt_cmp(const void* a, const void* b) {
    const vref_pt* x = (const vref_pt*)a; const vref_pt* y = (const vref_pt*)b;
    for (int k = 2; k >= 0; --k) if (x->v[k] != y->v[k]) return x->v[k] < y->v[k] ? -1 : 1;     /* (iz, iy, ix), then the index */
    return x->idx < y->idx ? -1 : (x->idx > y->idx ? 1 : 0);
}

int vref_voxel_downsample(int32_t n_clouds, const float* xyz, const float* nrm, const uint8_t* rgba, const int64_t* off, float voxel_size,
                           float* xyz_out, float* nrm_out, uint8_t* rgba_out, int64_t* off_out) {
    const float inv = 1.0f / voxel_size;                           /* V1 */
    int64_t m = 0;
    off_out[0] = 0;
    vref_pt* v = (vref_pt*)malloc(sizeof(vref_pt) * (size_t)(off[n_clouds] > 0 ? off[n_clouds] : 1));
    for (int32_t b = 0; b < n_clouds; ++b) {
        int64_t c = 0;
        for (int64_t i = off[b]; i < off[b + 1]; ++i) {
            const float* p = xyz + 3 * i;
            if (!finite3(p)) continue;
            for (int a = 0; a < 3; ++a) {
                const float f = floorf(p[a] * inv);
                if (!(f >= -2147483648.0f && f < 2147483648.0f)) { free(v); return -1 - b; }
                v[c].v[a] = (int32_t)f;
            }
            v[c].idx = i; ++c;
        }
        qsort(v, (size_t)c, sizeof(vref_pt), vref_pt_cmp);    /* V2 */
        for (int64_t s = 0; s < c;) {
            int64_t e = s + 1;
            while (e < c && v[e].v[0] == v[s].v[0] && v[e].v[1] == v[s].v[1] && v[e].v[2] == v[s].v[2]) ++e;
            double p[3] = {0, 0, 0}, q[3] = {0, 0, 0};
            uint64_t col[4] = {0, 0, 0, 0};
            int any = 0;
            for (int64_t j = s; j < e; ++j) {                      /* ascending original index */
                const int64_t i = v[j].idx;
                for (int a = 0; a < 3; ++a) p[a] += (double)xyz[3 * i + a];                                   /* V3 */
                if (nrm && finite3(nrm + 3 * i)) { for (int a = 0; a < 3; ++a) q[a] += (double)nrm[3 * i + a]; any = 1; }   /* V4 */
                if (rgba) for (int ch = 0; ch < 4; ++ch) col[ch] += rgba[4 * i + ch];                          /* V5 */
            }
            const uint64_t k = (uint64_t)(e - s);
            for (int a = 0; a < 3; ++a) xyz_out[3 * m + a] = (float)(p[a] / (double)k);
            if (nrm) {
                const double len = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2]);
                for (int a = 0; a < 3; ++a) nrm_out[3 * m + a] = (any && len != 0.0) ? (float)(q[a] / len) : -INFINITY;
            }
            if (rgba) for (int ch = 0; ch < 4; ++ch) rgba_out[4 * m + ch] = (uint8_t)((2 * col[ch] + k) / (2 * k));
            ++m; s = e;
        }
        off_out[b + 1] = m;
    }
    free(v);
    return 0;
}
