/*
 * cluster_reference.c — TEST INFRASTRUCTURE ONLY.  The links of ljmd_clusters, enumerated on the CPU with the grid
 * and the fp32 pair rule of tests/bond_reference.c (included, so there is one grid implementation):
 *   active   finite coordinates and, when a mask is given, mask[i] != 0
 *   links    the pairs i < j of active particles with r <= r_link, r = sqrtf(dx*dx + dy*dy), dx = minimg(x_j - x_i)
 *            in fp32; coincident particles (r = 0) are linked
 * Every pair when the grid of cells of edge >= r_link has fewer than 5 per side, otherwise that grid with its
 * +-2-cell stencil.  tests/cluster_reference.py compiles it (tests/cref.py) and turns the links into components.
 * The product never loads it.
 */
#include "ref_grid.h"

static inline int active(const float* R, const uint8_t* mask, int64_t i) {
    return finite2(R, i) && (!mask || mask[i]);
}

static int64_t links_of(const float* R, const uint8_t* mask, int64_t N, const Grid* g, int grid, int64_t i,
                        float box, float r_link, int32_t* out) {
    int64_t n = 0;
    float dx, dy;
    if (!active(R, mask, i)) return 0;
    if (!grid) {
        for (int64_t j = i + 1; j < N; ++j)
            if (active(R, mask, j) && pair_r(R, i, j, box, &dx, &dy) <= r_link) {
                if (out) { out[2 * n] = (int32_t)i; out[2 * n + 1] = (int32_t)j; }
                ++n;
            }
        return n;
    }
    int32_t nc = g->nc, cx = g->cid[i] % nc, cy = g->cid[i] / nc;
    for (int oy = -2; oy <= 2; ++oy)
        for (int ox = -2; ox <= 2; ++ox) {
            int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
            for (int32_t k = g->head[c]; k < g->head[c + 1]; ++k) {
                int64_t j = g->order[k];
                if (j > i && active(R, mask, j) && pair_r(R, i, j, box, &dx, &dy) <= r_link) {
                    if (out) { out[2 * n] = (int32_t)i; out[2 * n + 1] = (int32_t)j; }
                    ++n;
                }
            }
        }
    return n;
}

/* The links of one snapshot: a count pass, then (pairs != NULL) a fill pass writing (i, j) pairs, i < j, grouped by
 * i in ascending order.  mask may be NULL.  Returns the number of links. */
int64_t bref_links(int64_t N, const float* R, float box, float r_link, const uint8_t* mask, int32_t* pairs) {
    Grid g;
    int grid = grid_build(&g, N, R, box, r_link);
    int64_t* start = (int64_t*)calloc((size_t)N + 1, sizeof(int64_t));
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t i = 0; i < N; ++i) start[i + 1] = links_of(R, mask, N, &g, grid, i, box, r_link, NULL);
    for (int64_t i = 0; i < N; ++i) start[i + 1] += start[i];
    int64_t total = start[N];
    if (pairs) {
#pragma omp parallel for schedule(dynamic, 256)
        for (int64_t i = 0; i < N; ++i) links_of(R, mask, N, &g, grid, i, box, r_link, pairs + 2 * start[i]);
    }
    free(start);
    if (grid) grid_free(&g);
    return total;
}
