/*
 * bond_reference.c — TEST INFRASTRUCTURE ONLY.  CPU restatement of the bond-orientational order psi_m
 * (ljmd_bond_order) and of its pair-correlation histogram (ljmd_bond_corr), with the library's rules:
 *   neighbours   j != i with 0 < r <= r_nb, r = sqrtf(dx*dx + dy*dy), dx = minimg(x_j - x_i) in fp32
 *                (d - box*rintf(d/box): the minimum image of gr_reference.c / oracle/lj_oracle.c)
 *   bond term    in double: r_d = sqrt(dx^2 + dy^2), u = d / r_d, w = u^m by m - 1 products (ac - bd, ad + bc)
 *   fixed point  sum of llrint(w 2^32) in int64; psi = (double)sum * 2^-32 / n (0 when n = 0)
 *   NaN          a particle with a non-finite coordinate: psi = NaN, n = 0, nobody's neighbour
 *   corr         for the pairs i < j of gr_reference.c's histogram: w = a.x b.x + a.y b.y, skipped when not
 *                finite, else counts += 1 and wsum += llrint(w 2^24)
 * Neighbour search: every pair for N <= 65536 (bref_bond_order) or with fewer than 5 cells per side, otherwise
 * an OpenMP grid of cells of edge >= the radius (in double) with a +-2-cell stencil, so the result does not rely
 * on the margin proof of the library's grid.  Compiled by tests/bond_reference.py with -O2 -ffp-contract=off
 * -fno-fast-math (every operation rounds once).  The product never loads it.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

static inline float minimg(float d, float box) {
    return d - box * rintf(d / box);
}

static inline int finite2(const float* R, int64_t i) {
    return isfinite(R[2 * i]) && isfinite(R[2 * i + 1]);
}

/* cells of edge >= radius with a +-2-cell stencil; NULL (every pair) when that grid has fewer than 5 per side */
typedef struct { int32_t nc; int32_t* head; int32_t* cid; int32_t* order; } Grid;

static int grid_build(Grid* g, int64_t N, const float* R, float box, float radius) {
    int32_t nc = (int32_t)floor((double)box / (double)radius);
    if (nc > 4096) nc = 4096;
    if (nc < 5) return 0;
    double cell = (double)box / nc;
    size_t ncc = (size_t)nc * nc;
    g->nc = nc;
    g->head = (int32_t*)calloc(ncc + 1, sizeof(int32_t));
    g->cid = (int32_t*)malloc(sizeof(int32_t) * N);
    g->order = (int32_t*)malloc(sizeof(int32_t) * N);
    for (int64_t i = 0; i < N; ++i) {
        int32_t cx = 0, cy = 0;
        if (finite2(R, i)) {                       /* non-finite particles pair with nobody: any cell will do */
            cx = (int32_t)floor((double)R[2 * i] / cell);
            cy = (int32_t)floor((double)R[2 * i + 1] / cell);
            if (cx >= nc) cx = nc - 1;
            if (cy >= nc) cy = nc - 1;
            if (cx < 0) cx = 0;
            if (cy < 0) cy = 0;
        }
        g->cid[i] = cy * nc + cx;
        g->head[g->cid[i] + 1]++;
    }
    for (size_t c = 0; c < ncc; ++c) g->head[c + 1] += g->head[c];
    int32_t* fill = (int32_t*)malloc(sizeof(int32_t) * ncc);
    memcpy(fill, g->head, sizeof(int32_t) * ncc);
    for (int64_t i = 0; i < N; ++i) g->order[fill[g->cid[i]]++] = (int32_t)i;
    free(fill);
    return 1;
}

static void grid_free(Grid* g) {
    free(g->head); free(g->cid); free(g->order);
}

static inline float pair_r(const float* R, int64_t i, int64_t j, float box, float* dx, float* dy) {
    *dx = minimg(R[2 * j] - R[2 * i], box);
    *dy = minimg(R[2 * j + 1] - R[2 * i + 1], box);
    return sqrtf(*dx * *dx + *dy * *dy);
}

static inline void bond_add(const float* R, int64_t i, int64_t j, float box, int32_t m, float r_nb,
                            int64_t* sx, int64_t* sy, int32_t* n) {
    float dxf, dyf;
    float r = pair_r(R, i, j, box, &dxf, &dyf);
    if (!(r > 0.0f && r <= r_nb)) return;
    double dx = dxf, dy = dyf;
    double rd = sqrt(dx * dx + dy * dy);
    double ux = dx / rd, uy = dy / rd, wx = ux, wy = uy;
    for (int32_t k = 1; k < m; ++k) {
        double a = wx, b = wy;
        wx = a * ux - b * uy;
        wy = a * uy + b * ux;
    }
    *sx += llrint(wx * 4294967296.0);
    *sy += llrint(wy * 4294967296.0);
    ++*n;
}

void bref_bond_order(int64_t N, const float* R, float box, int32_t m, float r_nb, double* psi, int32_t* nnb) {
    Grid g;
    int grid = N > 65536 && grid_build(&g, N, R, box, r_nb);
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t i = 0; i < N; ++i) {
        int64_t sx = 0, sy = 0;
        int32_t n = 0;
        if (!finite2(R, i)) {
            psi[2 * i] = psi[2 * i + 1] = NAN;
            nnb[i] = 0;
            continue;
        }
        if (!grid) {
            for (int64_t j = 0; j < N; ++j) bond_add(R, i, j, box, m, r_nb, &sx, &sy, &n);
        } else {
            int32_t nc = g.nc, cx = g.cid[i] % nc, cy = g.cid[i] / nc;
            for (int oy = -2; oy <= 2; ++oy)
                for (int ox = -2; ox <= 2; ++ox) {
                    int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
                    for (int32_t k = g.head[c]; k < g.head[c + 1]; ++k) bond_add(R, i, g.order[k], box, m, r_nb, &sx, &sy, &n);
                }
        }
        nnb[i] = n;
        psi[2 * i] = n ? (double)sx * 0x1p-32 / n : 0.0;
        psi[2 * i + 1] = n ? (double)sy * 0x1p-32 / n : 0.0;
    }
    if (grid) grid_free(&g);
}

static inline void corr_pair(const float* R, const double* psi, int64_t i, int64_t j, float box, int32_t nbins,
                             const float* edges, float lo, float hi, int64_t* h, int64_t* ws) {
    float dx, dy;
    float r = pair_r(R, j, i, box, &dx, &dy);       /* fl(x_i - x_j), as gr_reference.c */
    if (!(r >= lo && r <= hi)) return;
    double w = psi[2 * i] * psi[2 * j] + psi[2 * i + 1] * psi[2 * j + 1];
    if (!isfinite(w)) return;
    int32_t a = 0, b = nbins;
    while (b - a > 1) { int32_t mid = (a + b) >> 1; if (edges[mid] <= r) a = mid; else b = mid; }
    h[a]++;
    ws[a] += llrint(w * 16777216.0);
}

void bref_bond_corr(int64_t N, const float* R, const double* psi, float box, int32_t nbins, const float* edges,
                    float r_cap, int64_t* counts, int64_t* wsum) {
    memset(counts, 0, sizeof(int64_t) * nbins);
    memset(wsum, 0, sizeof(int64_t) * nbins);
    float lo = edges[0], hi = fminf(edges[nbins], r_cap);
    int nthr = 1;
#ifdef _OPENMP
    nthr = omp_get_max_threads();
#endif
    int64_t* part = (int64_t*)calloc((size_t)nthr * 2 * nbins, sizeof(int64_t));
    Grid g;
    int grid = grid_build(&g, N, R, box, r_cap);
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < N; ++i) {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        int64_t* h = part + (size_t)t * 2 * nbins;
        if (!grid) {
            for (int64_t j = i + 1; j < N; ++j) corr_pair(R, psi, i, j, box, nbins, edges, lo, hi, h, h + nbins);
        } else {
            int32_t nc = g.nc, cx = g.cid[i] % nc, cy = g.cid[i] / nc;
            for (int oy = -2; oy <= 2; ++oy)
                for (int ox = -2; ox <= 2; ++ox) {
                    int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
                    for (int32_t k = g.head[c]; k < g.head[c + 1]; ++k)
                        if (g.order[k] > i) corr_pair(R, psi, i, g.order[k], box, nbins, edges, lo, hi, h, h + nbins);
                }
        }
    }
    if (grid) grid_free(&g);
    for (int t = 0; t < nthr; ++t)
        for (int32_t k = 0; k < nbins; ++k) {
            counts[k] += part[(size_t)t * 2 * nbins + k];
            wsum[k] += part[(size_t)t * 2 * nbins + nbins + k];
        }
    free(part);
}
