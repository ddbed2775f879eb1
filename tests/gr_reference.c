/*
 * gr_reference.c — TEST INFRASTRUCTURE ONLY.  CPU recount of the g(r) pair-distance histogram through a
 * cell grid, for N in the millions: the count of unordered pairs i < j whose fp32 minimum-image distance
 *     r = sqrtf(dx*dx + dy*dy),  dx = d - box*rintf(d/box)   (oracle/lj_oracle.c's orc_gr_hist)
 * lies in [edges[0], min(edges[nbins], r_cap)], binned by binary search against the fp32 edges (last bin
 * right-closed).  The grid has cells of edge >= r_cap (in double) and a +-2-cell stencil, as
 * orc_neighbor_count, so the recount does not depend on how a particle on a cell edge is binned; with
 * fewer than 5 cells per side every pair is visited.  Each OpenMP thread counts into its own integer
 * histogram and the histograms are summed.  Compiled by tests/gr_reference.py with -O2 -ffp-contract=off
 * -fno-fast-math (every fp32 operation rounds once).  The product never loads it.
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

static inline void bin_pair(const float* R, int64_t i, int64_t j, float box, int32_t nbins, const float* edges,
                            float lo, float hi, int64_t* h) {
    float dx = minimg(R[2 * i] - R[2 * j], box), dy = minimg(R[2 * i + 1] - R[2 * j + 1], box);
    float r = sqrtf(dx * dx + dy * dy);
    if (!(r >= lo && r <= hi)) return;
    int32_t a = 0, b = nbins;                   /* largest k with edges[k] <= r ; r == edges[nbins] -> last bin */
    while (b - a > 1) { int32_t m = (a + b) >> 1; if (edges[m] <= r) a = m; else b = m; }
    h[a]++;
}

void gref_gr_hist(int64_t N, const float* R, float box, int32_t nbins, const float* edges, float r_cap,
                  int64_t* counts) {
    memset(counts, 0, sizeof(int64_t) * nbins);
    float lo = edges[0], hi = fminf(edges[nbins], r_cap);
    int32_t nc = (isfinite(r_cap) && r_cap > 0.0f) ? (int32_t)floor((double)box / (double)r_cap) : 1;
    if (nc > 4096) nc = 4096;
    int nthr = 1;
#ifdef _OPENMP
    nthr = omp_get_max_threads();
#endif
    int64_t* part = (int64_t*)calloc((size_t)nthr * nbins, sizeof(int64_t));
    if (nc < 5) {
#pragma omp parallel for schedule(dynamic, 64)
        for (int64_t i = 0; i < N; ++i) {
            int t = 0;
#ifdef _OPENMP
            t = omp_get_thread_num();
#endif
            for (int64_t j = i + 1; j < N; ++j) bin_pair(R, i, j, box, nbins, edges, lo, hi, part + (size_t)t * nbins);
        }
    } else {
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
#pragma omp parallel for schedule(dynamic, 1024)
        for (int64_t i = 0; i < N; ++i) {
            int t = 0;
#ifdef _OPENMP
            t = omp_get_thread_num();
#endif
            int64_t* h = part + (size_t)t * nbins;
            int32_t cx = cid[i] % nc, cy = cid[i] / nc;
            for (int oy = -2; oy <= 2; ++oy)
                for (int ox = -2; ox <= 2; ++ox) {
                    int32_t c = ((cy + oy + nc) % nc) * nc + ((cx + ox + nc) % nc);
                    for (int32_t k = head[c]; k < head[c + 1]; ++k) {
                        int64_t j = order[k];
                        if (j > i) bin_pair(R, i, j, box, nbins, edges, lo, hi, h);
                    }
                }
        }
        free(head); free(cid); free(order); free(fill);
    }
    for (int t = 0; t < nthr; ++t)
        for (int32_t k = 0; k < nbins; ++k) counts[k] += part[(size_t)t * nbins + k];
    free(part);
}
