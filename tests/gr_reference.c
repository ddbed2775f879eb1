/*
 * gr_reference.c — TEST INFRASTRUCTURE ONLY.  CPU recount of the g(r) pair-distance histogram through a
 * cell grid, for N in the millions: the count of unordered pairs i < j whose fp32 minimum-image distance
 *     r = sqrtf(dx*dx + dy*dy),  dx = d - box*rintf(d/box)   (oracle/lj_oracle.c's orc_gr_hist)
 * lies in [edges[0], min(edges[nbins], r_cap)], binned by binary search against the fp32 edges (last bin
 * right-closed).  The grid of ref_grid.h has cells of edge >= r_cap and a +-2-cell stencil, as
 * orc_neighbor_count; with fewer than 5 cells per side every pair is visited.  Each OpenMP thread counts into
 * its own integer histogram and the histograms are summed.  Compiled by tests/cref.py.  The product never
 * loads it.
 */
#include "ref_grid.h"
#ifdef _OPENMP
#include <omp.h>
#endif

static inline void bin_pair(const float* R, int64_t i, int64_t j, float box, int32_t nbins, const float* edges,
                            float lo, float hi, int64_t* h) {
    float dx, dy;
    float r = pair_r(R, j, i, box, &dx, &dy);   /* fl(x_i - x_j) */
    if (!(r >= lo && r <= hi)) return;
    int32_t a = 0, b = nbins;                   /* largest k with edges[k] <= r ; r == edges[nbins] -> last bin */
    while (b - a > 1) { int32_t m = (a + b) >> 1; if (edges[m] <= r) a = m; else b = m; }
    h[a]++;
}

void gref_gr_hist(int64_t N, const float* R, float box, int32_t nbins, const float* edges, float r_cap,
                  int64_t* counts) {
    memset(counts, 0, sizeof(int64_t) * nbins);
    float lo = edges[0], hi = fminf(edges[nbins], r_cap);
    int nthr = 1;
#ifdef _OPENMP
    nthr = omp_get_max_threads();
#endif
    int64_t* part = (int64_t*)calloc((size_t)nthr * nbins, sizeof(int64_t));
    Grid g;
    int grid = grid_build(&g, N, R, box, r_cap);
#pragma omp parallel for schedule(dynamic, 64)
    for (int64_t i = 0; i < N; ++i) {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        int64_t* h = part + (size_t)t * nbins;
        if (!grid) {
            for (int64_t j = i + 1; j < N; ++j) bin_pair(R, i, j, box, nbins, edges, lo, hi, h);
            continue;
        }
        int32_t nc = g.nc, cx = g.cid[i] % nc, cy = g.cid[i] / nc;
        for (int oy = -2; oy <= 2; ++oy)
            for (int ox = -2; ox <= 2; ++ox) {
                int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
                for (int32_t k = g.head[c]; k < g.head[c + 1]; ++k)
                    if (g.order[k] > i) bin_pair(R, i, g.order[k], box, nbins, edges, lo, hi, h);
            }
    }
    if (grid) grid_free(&g);
    for (int t = 0; t < nthr; ++t)
        for (int32_t k = 0; k < nbins; ++k) counts[k] += part[(size_t)t * nbins + k];
    free(part);
}
