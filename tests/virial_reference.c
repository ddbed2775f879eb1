/*
 * virial_reference.c — TEST INFRASTRUCTURE ONLY.  Plain-C fp32 restatement of the pair virial
 *     W = sum_{i<j, r2 < rc2} r_ij . f_ij = sum 24 eps (2 (sigma/r)^12 - (sigma/r)^6)
 * with the arithmetic of oracle/lj_oracle.c's pair_term (the same minimum image d - box*rint(d/box), the
 * same unfused r2 = dx*dx + dy*dy, the same s2 = sig2/r2 by true division): per pair the factor of
 * pair_term's force scalar, in fp32; the pair terms summed in double over ordered pairs and halved (like PE).
 * *wabs_out = sum_{i<j} |w_ij|, the scale of the rounding error any fp32 summation order can make.
 * Compiled by tests/virial_reference.py with -O2 -ffp-contract=off -fno-fast-math (every fp32 operation
 * rounds once).  The product never loads it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static inline float minimg(float d, float box) {
    return d - box * rintf(d / box);
}

static inline float pair_virial(float xi, float yi, float xj, float yj, float box, float sig2, float eps,
                                float rc2, int* inside) {
    float dx = minimg(xi - xj, box);
    float dy = minimg(yi - yj, box);
    float r2 = dx * dx + dy * dy;
    float s2 = sig2 / r2;
    float s6 = (s2 * s2) * s2;
    float s12 = s6 * s6;
    *inside = (r2 < rc2);
    return (24.0f * eps) * (2.0f * s12 - s6);
}

/* dense O(N^2); rc2 = INFINITY: every pair (the reference, no cutoff) */
void vref_virial(int64_t N, const float* R, float box, float sigma, float eps, float rc2,
                 double* w_out, double* wabs_out) {
    float sig2 = sigma * sigma;
    double w_tot = 0.0, a_tot = 0.0;
#pragma omp parallel for schedule(static) reduction(+ : w_tot, a_tot)
    for (int64_t i = 0; i < N; ++i) {
        for (int64_t j = 0; j < N; ++j) {
            if (j == i) continue;
            int in;
            float w = pair_virial(R[2 * i], R[2 * i + 1], R[2 * j], R[2 * j + 1], box, sig2, eps, rc2, &in);
            if (!in) continue;
            w_tot += w;
            a_tot += fabs((double)w);
        }
    }
    if (w_out) *w_out = 0.5 * w_tot;
    if (wabs_out) *wabs_out = 0.5 * a_tot;
}

/* the same through a CPU cell grid of edge >= rc (as orc_forces_cells), for N in the millions */
void vref_virial_cells(int64_t N, const float* R, float box, float sigma, float eps, float rc,
                       double* w_out, double* wabs_out) {
    int32_t nc = (int32_t)floor((double)box / (double)rc);
    if (nc < 5) { vref_virial(N, R, box, sigma, eps, rc * rc, w_out, wabs_out); return; }
    double cell = (double)box / nc;
    size_t ncc = (size_t)nc * nc;
    int32_t* head = (int32_t*)calloc(ncc + 1, sizeof(int32_t));
    int32_t* cid = (int32_t*)malloc(sizeof(int32_t) * N);
    int32_t* order = (int32_t*)malloc(sizeof(int32_t) * N);
    for (int64_t i = 0; i < N; ++i) {
        int32_t cx = (int32_t)floor((double)R[2 * i] / cell), cy = (int32_t)floor((double)R[2 * i + 1] / cell);
        if (cx >= nc) cx = nc - 1;
        if (cy >= nc) cy = nc - 1;
        if (cx < 0) cx = 0;
        if (cy < 0) cy = 0;
        cid[i] = cy * nc + cx;
        head[cid[i] + 1]++;
    }
    for (size_t c = 0; c < ncc; ++c) head[c + 1] += head[c];
    int32_t* fill = (int32_t*)malloc(sizeof(int32_t) * ncc);
    memcpy(fill, head, sizeof(int32_t) * ncc);
    for (int64_t i = 0; i < N; ++i) order[fill[cid[i]]++] = (int32_t)i;
    float sig2 = sigma * sigma, rc2 = rc * rc;
    double w_tot = 0.0, a_tot = 0.0;
    /* +-2 cells: independent of the fp32-vs-double binning of particles on a cell edge */
#pragma omp parallel for schedule(dynamic, 1024) reduction(+ : w_tot, a_tot)
    for (int64_t i = 0; i < N; ++i) {
        float xi = R[2 * i], yi = R[2 * i + 1];
        int32_t cx = cid[i] % nc, cy = cid[i] / nc;
        for (int oy = -2; oy <= 2; ++oy)
            for (int ox = -2; ox <= 2; ++ox) {
                int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
                for (int32_t k = head[c]; k < head[c + 1]; ++k) {
                    int32_t j = order[k];
                    if (j == i) continue;
                    int in;
                    float w = pair_virial(xi, yi, R[2 * j], R[2 * j + 1], box, sig2, eps, rc2, &in);
                    if (!in) continue;
                    w_tot += w;
                    a_tot += fabs((double)w);
                }
            }
    }
    if (w_out) *w_out = 0.5 * w_tot;
    if (wabs_out) *wabs_out = 0.5 * a_tot;
    free(head); free(cid); free(order); free(fill);
}
