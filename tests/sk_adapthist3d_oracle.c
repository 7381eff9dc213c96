/*
 * sk_adapthist3d_oracle.c — per-voxel C restatement of skimage.exposure.equalize_adapthist on ONE 3-D volume
 * (TEST INFRASTRUCTURE, loaded by tests/sk_adapthist3d_oracle.py; nothing in the package links it).
 *
 * It includes the CPU oracle whole, so the volume path reuses that file's numpy 'reflect' index (sk_reflect), the
 * iterative clip redistribution (sk_clip_histogram) and the grey / rescale stages (orc_sk_adapthist_grey,
 * orc_sk_rescale01 on flat buffers of d * h rows) instead of restating them.  The contextual-region stage below is
 * the 3-D form of orc_sk_clahe; sk_exposure.cu's volume kernels follow it bit for bit.  Compile with the oracle's
 * flags (-ffp-contract=off: nothing is fused).
 */
#include "../oracle/mie_oracle.c"

/* _clahe on a 2^14-level VOLUME (skimage on a 3-D array): the per-voxel form of orc_sk_clahe with kernel (kd, kr, kc).
 * ceil(d/kd) x ceil(h/kr) x ceil(w/kc) regions anchored at the origin, completed by 'reflect' padding; a voxel at
 * (z, y, x) lies in block ((z + kd/2) / kd, ...) at position ((z + kd/2) % kd, ...) and blends the 8 mappings of the
 * regions clamp(block - 1) / clamp(block) per axis.  The coefficient of edge (ez, ey, ex) is (wx[ex] * wy[ey]) * wz[ez]
 * (np.prod over the axes reversed, left to right); float32(mapped * coef) is accumulated over the edges in
 * np.ndindex(2, 2, 2) order — z outermost, x innermost — and truncated to uint16. */
int orc_sk_clahe3d(const uint16_t* grey, int d, int h, int w, int kd, int kr, int kc, double clip_limit, int nbins,
                   uint16_t* out, int64_t* maps_out /* optional: nbz * nby * nbx * nbins */) {
    if (kd <= 0 || kr <= 0 || kc <= 0 || nbins <= 0 || nbins > 16384) return -3;
    const int nbz = (d + kd - 1) / kd, nby = (h + kr - 1) / kr, nbx = (w + kc - 1) / kc;
    const int bin_size = 1 + 16384 / nbins;
    const int64_t kernel_elements = (int64_t)kd * kr * kc;
    int64_t clim;
    if (clip_limit > 0.0) {
        double c = clip_limit * (double)kernel_elements;
        if (c < 1.0) c = 1.0;
        clim = (int64_t)c;
    } else {
        clim = 65535; /* np.iinfo(uint16).max: "no clipping" */
    }
    const int64_t nreg = (int64_t)nbz * nby * nbx;
    int64_t* maps = (int64_t*)malloc((size_t)nreg * nbins * sizeof(int64_t));
    if (!maps) return -1;
    const double scale = 16383.0 / (double)kernel_elements;
#pragma omp parallel for schedule(dynamic, 1)
    for (int64_t b = 0; b < nreg; ++b) {
        const int bz = (int)(b / ((int64_t)nby * nbx)), by = (int)(b / nbx % nby), bx = (int)(b % nbx);
        int64_t* hist = maps + (size_t)b * nbins;
        memset(hist, 0, (size_t)nbins * sizeof(int64_t));
        for (int dz = 0; dz < kd; ++dz) {
            const int sz = sk_reflect(bz * kd + dz, d);
            for (int r = 0; r < kr; ++r) {
                const int sy = sk_reflect(by * kr + r, h);
                const uint16_t* row = grey + ((size_t)sz * h + sy) * w;
                for (int c = 0; c < kc; ++c) hist[row[sk_reflect(bx * kc + c, w)] / bin_size] += 1;
            }
        }
        sk_clip_histogram(hist, nbins, clim);
        int64_t cum = 0;
        for (int k = 0; k < nbins; ++k) { /* map_histogram */
            cum += hist[k];
            double v = (double)cum * scale;
            v += 0.0;
            if (v > 16383.0) v = 16383.0;
            hist[k] = (int64_t)v;
        }
    }
    if (maps_out) memcpy(maps_out, maps, (size_t)nreg * nbins * sizeof(int64_t));
#pragma omp parallel for schedule(static) collapse(2)
    for (int z = 0; z < d; ++z) {
        for (int y = 0; y < h; ++y) {
            const int pz = z + kd / 2, bz = pz / kd, rz = pz % kd;
            const double cz = (double)rz / (double)kd;
            int hb_z[2] = {bz - 1, bz};
            for (int e = 0; e < 2; ++e) { if (hb_z[e] < 0) hb_z[e] = 0; if (hb_z[e] > nbz - 1) hb_z[e] = nbz - 1; }
            const double wz[2] = {1.0 - cz, cz};
            const int py = y + kr / 2, by = py / kr, ry = py % kr;
            const double cy = (double)ry / (double)kr;
            int hb_y[2] = {by - 1, by};
            for (int e = 0; e < 2; ++e) { if (hb_y[e] < 0) hb_y[e] = 0; if (hb_y[e] > nby - 1) hb_y[e] = nby - 1; }
            const double wy[2] = {1.0 - cy, cy};
            for (int x = 0; x < w; ++x) {
                const int pxx = x + kc / 2, bx = pxx / kc, rx = pxx % kc;
                const double cx = (double)rx / (double)kc;
                int hb_x[2] = {bx - 1, bx};
                for (int e = 0; e < 2; ++e) { if (hb_x[e] < 0) hb_x[e] = 0; if (hb_x[e] > nbx - 1) hb_x[e] = nbx - 1; }
                const double wx[2] = {1.0 - cx, cx};
                const size_t p = ((size_t)z * h + y) * w + x;
                const int bin = grey[p] / bin_size;
                float acc = 0.0f;
                for (int ez = 0; ez < 2; ++ez)
                    for (int ey = 0; ey < 2; ++ey)
                        for (int ex = 0; ex < 2; ++ex) {
                            const int64_t m = maps[(((size_t)hb_z[ez] * nby + hb_y[ey]) * nbx + hb_x[ex]) * nbins + bin];
                            const double coef = (wx[ex] * wy[ey]) * wz[ez];
                            acc = acc + (float)((double)m * coef);
                        }
                out[p] = (uint16_t)acc;
            }
        }
    }
    free(maps);
    return 0;
}
