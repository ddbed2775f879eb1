/*
 * ref_grid.h — TEST INFRASTRUCTURE ONLY.  The fp32 pair rule and the CPU cell grid that the C references of the
 * snapshot analyses share (gr_reference.c, bond_reference.c, cluster_reference.c, virial_reference.c):
 *   minimg       d - box*rintf(d/box), the minimum image of oracle/lj_oracle.c
 *   pair_r       r = sqrtf(dx*dx + dy*dy) with dx = minimg(x_j - x_i) in fp32
 *   grid_build   a counting sort into cells of edge >= radius (in double), for a +-2-cell stencil, so a result does
 *                not depend on how a particle on a cell edge is binned; returns 0 (visit every pair instead) when
 *                that grid has fewer than 5 cells per side.  At most 4096 cells per side.
 * Compiled with -ffp-contract=off -fno-fast-math (tests/cref.py), so every operation rounds once.
 */
#pragma once
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

static inline float minimg(float d, float box) {
    return d - box * rintf(d / box);
}

static inline int finite2(const float* R, int64_t i) {
    return isfinite(R[2 * i]) && isfinite(R[2 * i + 1]);
}

static inline float pair_r(const float* R, int64_t i, int64_t j, float box, float* dx, float* dy) {
    *dx = minimg(R[2 * j] - R[2 * i], box);
    *dy = minimg(R[2 * j + 1] - R[2 * i + 1], box);
    return sqrtf(*dx * *dx + *dy * *dy);
}

/* head[c] .. head[c + 1]: the particles of cell c in order[]; cid[i]: the cell of particle i */
typedef struct { int32_t nc; int32_t* head; int32_t* cid; int32_t* order; } Grid;

/* floor(x / cell) clamped to [0, nc - 1], in double before the conversion, so no input converts out of range */
static inline int32_t grid_coord(float x, double cell, int32_t nc) {
    double c = floor((double)x / cell);
    return c < 0.0 ? 0 : c >= nc ? nc - 1 : (int32_t)c;
}

static int grid_build(Grid* g, int64_t N, const float* R, float box, float radius) {
    if (!(isfinite(radius) && radius > 0.0f)) return 0;
    double q = floor((double)box / (double)radius);
    int32_t nc = q > 4096.0 ? 4096 : (int32_t)q;
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
            cx = grid_coord(R[2 * i], cell, nc);
            cy = grid_coord(R[2 * i + 1], cell, nc);
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
