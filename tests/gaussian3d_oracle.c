/*
 * gaussian3d_oracle.c — per-voxel C restatement of skimage.filters.gaussian / unsharp_mask on 3-D arrays
 * (scipy.ndimage.gaussian_filter over all axes).  TEST INFRASTRUCTURE, loaded by tests/gaussian3d_oracle.py; nothing
 * in the package links it.
 *
 * It includes the CPU oracle whole, so the x and y passes are the 2-D oracle's own (orc_gaussian2d_ex on every plane)
 * and every source index goes through its border_index.  gauss3d.cu follows the result bit for bit.  Compile with the
 * oracle's flags (-ffp-contract=off: nothing is fused).
 */
#include "../oracle/mie_oracle.c"

/* n independent (d, h, w) volumes.  Pass order x, y (orc_gaussian2d_ex on every plane), then z, each with the
 * accumulation rule acc = w[0]*x[0]; acc = fmaf(w[t], x[t], acc); with kz == 1 (weight 1.0) the z pass is exact and
 * the result is orc_gaussian2d_ex's per plane.  Any radius on any axis length.  unsharp: fmaf(amount, x - blur, x),
 * clipped to [0, 1] when clip is set.  One scratch volume of d*h*w floats holds the xy-blurred planes. */
int orc_gaussian3d_ex(const float* in, float* out, int64_t n, int d, int h, int w, const float* wx, int kx,
                      const float* wy, int ky, const float* wz, int kz, int border, int unsharp, float amount, int clip) {
    if (kz <= 0) return 1;
    const size_t plane = (size_t)h * w, vol = (size_t)d * plane;
    float* xy = (float*)malloc(vol * sizeof(float));
    if (!xy) return 1;
    const int rz = kz / 2;
    for (int64_t v = 0; v < n; ++v) {
        const float* src = in + (size_t)v * vol;
        float* dst = out + (size_t)v * vol;
        if (orc_gaussian2d_ex(src, xy, d, h, w, wx, kx, wy, ky, border, 0, 1.0f, 0)) {
            free(xy);
            return 1;
        }
#pragma omp parallel for schedule(dynamic, 1)
        for (int z = 0; z < d; ++z) {
            float* acc = dst + (size_t)z * plane;   /* accumulated in place, tap by tap */
            for (int t = 0; t < kz; ++t) {
                const int sz = border_index(z - rz + t, d, border);
                const float* p = sz < 0 ? NULL : xy + (size_t)sz * plane;
                for (size_t i = 0; i < plane; ++i) {
                    const float x = p ? p[i] : 0.0f;
                    acc[i] = t == 0 ? wz[0] * x : fmaf(wz[t], x, acc[i]);
                }
            }
            if (unsharp) {
                const float* c = src + (size_t)z * plane;
                for (size_t i = 0; i < plane; ++i) {
                    float r = fmaf(amount, c[i] - acc[i], c[i]);
                    acc[i] = clip ? fminf(fmaxf(r, 0.0f), 1.0f) : r;
                }
            }
        }
    }
    free(xy);
    return 0;
}
