// voronoi.cu — the Voronoi cell of every particle of S snapshots on the periodic box (ljmd_voronoi), through the
// periodic cell grid of g(r) (gr.cu): neighbour count, area, angle-ordered adjacency and edge-weighted psi_m.
//
// Displacements.  d_ij = x_j - x_i of the fp32 coordinates taken in double, then shifted by -box if > box / 2 and by
// +box if < -box / 2.  Both steps are exact in double unless a coordinate is a tiny non-zero value (below about
// 2^-29 box; the error is then <= 2^-53 box), so d_ji = -d_ij bit for bit and neighbouring particles see their
// shared vertices in frames that agree to the rounding of the clipping alone.  r2 = fl(fl(dx^2) + fl(dy^2)).
//
// Cell.  V_i = { p : p.d_ij <= r2_ij / 2 for every active j with d_ij != 0 }, a convex polygon around the origin
// (site i), in double.  It starts as the square [-box/2, box/2]^2 and is clipped by one candidate j at a time in
// the total order (r2, original index) ascending; a candidate whose bisector misses the polygon changes nothing.
// Coincident sites: i ignores those at d = 0 (so coincident particles get the same cell), and of several sites at
// one point only the smallest index clips (the others give the same half-plane): it alone is the neighbour.
//
// Security radius.  Let R be the largest distance from the origin to a vertex of the current polygon.  A site at
// |d| >= 2R cannot cut it (its bisector is >= R from the origin), and once every site with |d| < 2R has been
// applied the polygon is V_i (a ray from the origin leaves V_i at a point q of the bisector of some j with
// |d_j| <= 2|q| <= 2R).  So the walk stops at the first candidate with r2 >= min(4R^2, box^2/4); the cell is
// COMPLETE when then 2R < box / 2.  Every image of j other than the minimum one is >= box / 2 from i, and so is
// every image of i itself, so then no other image can cut V_i either, and the cell is the cell on the torus.
// Otherwise (2R >= box / 2: a tiny box or a void of comparable size), or when the polygon would need more than
// VOR_CAP vertices, the particle is INCOMPLETE: nvor = -1, area = psi = NaN, adjacency row -1.
//
// Degeneracy.  An edge of the final polygon counts when its length l > VOR_TAU R.  Four co-circular sites (the
// square lattice) leave edges of ~1e-16 R from rounding; VOR_TAU = 2^-30 keeps them out with ~7 orders of
// magnitude to spare.  nvor = the number of counted edges; each has one generating neighbour.
//
// Rings (coverage margin, after gr_grid_side).  The walk visits the (2k+1)^2 cells around i's cell of the nc x nc
// grid of edge w = box / nc.  gr_cell puts a particle of x / w in [c - 2u nc, c + 1 + 2u nc] (u = 2^-24, the two
// roundings of fl(x fl(nc / box)); the clamp moves only x == box into the last cell), so a site outside the rings
// is, on one axis, at least (k + 1 - 1 - 4u nc) w = k w - 4u box from i in every periodic image.  With
// rho_k = k w - 2^-20 box every site with |d| < rho_k (hence r2 < rho_k^2, double rounding included) is in the
// rings.  The next candidate is selected by a scan of the rings for the smallest key above the last one; it is the
// global next one when its r2 < rho_k^2.  If not, and rho_k^2 < the stop bound, the rings grow by one; once
// 2k + 1 >= nc the scan covers every particle of the snapshot (rho = infinity).  nc < 3: one cell, all particles.
//
// Determinism.  The sequence of clips is the global (r2, index) order up to the stop, whatever the cell order the
// atomic ranks of gr_count_kernel give, and every output is computed by one thread from that sequence: results are
// bit-identical run to run, across batches, handles and the other snapshots of the call.
//
// Outputs (original order, one thread per particle in cell order, grid.y = snapshot in the batch): nvor; area by
// the shoelace formula over all vertices; adjacency = the counted neighbours' original indices ordered by the angle
// of d_ij ascending in (-pi, pi] (the polygon is counter-clockwise, so its edge normals already are in angular
// order up to the start), first adj_cap of them, -1 padded; psi = sum_j (l_j / L) (d_j / |d_j|)^m in that order,
// L = sum of the counted l_j, u^m by unit_pow (m - 1 sequential complex products), every operation rounded once.
#include "ljmd_device.cuh"

#include <algorithm>
#include <cmath>

namespace ljmd {

namespace {

constexpr int    VOR_THREADS = 128;
constexpr int    VOR_CAP     = LJMD_VORONOI_MAX_VERTICES;   // polygon vertices held per thread (local memory)
constexpr double VOR_TAU     = 0x1p-30;
#ifndef VOR_CELL
#define VOR_CELL 2.0   // cell edge in mean spacings box / sqrt(N) (measured, DESIGN.md 4.8)
#endif

__device__ __forceinline__ double nan_d() { return __longlong_as_double(0x7ff8000000000000ll); }

// exact minimum-image displacement (see the top of the file)
__device__ __forceinline__ double vor_disp(float xj, float xi, double box, double half) {
    double d = __dsub_rn((double)xj, (double)xi);
    if (d > half) d = __dsub_rn(d, box);
    else if (d < -half) d = __dadd_rn(d, box);
    return d;
}

struct Poly {
    double x[VOR_CAP], y[VOR_CAP];
    int    g[VOR_CAP];   // generator of edge k (vertex k -> k + 1): the site's index in cell order, -1 = the square
    int    n;
};

__device__ __forceinline__ double vor_f(const Poly& P, int k, double dx, double dy, double h) {
    return __dsub_rn(__dadd_rn(__dmul_rn(P.x[k], dx), __dmul_rn(P.y[k], dy)), h);
}

// Clip P by { p : p.d <= h } (h = r2 / 2), the new edge generated by q.  The vertices outside form one cyclic run
// around the farthest one (a convex polygon and a line); a vertex outside only by rounding elsewhere is kept.
// The run [r0 .. e] is replaced by P1 on edge (r0 - 1, r0) and P2 on edge (e, e + 1).  false: more than VOR_CAP.
__device__ bool vor_clip(Poly& P, double dx, double dy, double h, int q) {
    const int n = P.n;
    double fmax = 0.0;
    int imax = -1;
    for (int k = 0; k < n; ++k) {
        const double f = vor_f(P, k, dx, dy, h);
        if (f > fmax) { fmax = f; imax = k; }
    }
    if (imax < 0) return true;                                      // the bisector misses the polygon
    int r0 = imax, e = imax, cnt = 1;
    while (cnt < n) {
        const int k = r0 == 0 ? n - 1 : r0 - 1;
        if (!(vor_f(P, k, dx, dy, h) > 0.0)) break;
        r0 = k;
        ++cnt;
    }
    while (cnt < n) {
        const int k = e + 1 == n ? 0 : e + 1;
        if (!(vor_f(P, k, dx, dy, h) > 0.0)) break;
        e = k;
        ++cnt;
    }
    if (cnt == n) return false;   // cannot happen (the origin is inside); reported as incomplete, never as a cell
    if (cnt == 1 && n == VOR_CAP) return false;
    const int a = r0 == 0 ? n - 1 : r0 - 1, b = e + 1 == n ? 0 : e + 1;
    const double fa = vor_f(P, a, dx, dy, h), fr = vor_f(P, r0, dx, dy, h);
    const double fe = vor_f(P, e, dx, dy, h), fb = vor_f(P, b, dx, dy, h);
    const double t1 = __ddiv_rn(fa, __dsub_rn(fa, fr)), t2 = __ddiv_rn(fb, __dsub_rn(fb, fe));
    const double p1x = __dadd_rn(P.x[a], __dmul_rn(t1, __dsub_rn(P.x[r0], P.x[a])));
    const double p1y = __dadd_rn(P.y[a], __dmul_rn(t1, __dsub_rn(P.y[r0], P.y[a])));
    const double p2x = __dadd_rn(P.x[b], __dmul_rn(t2, __dsub_rn(P.x[e], P.x[b])));
    const double p2y = __dadd_rn(P.y[b], __dmul_rn(t2, __dsub_rn(P.y[e], P.y[b])));
    const int ge = P.g[e];
    int s1, s2;                                                     // slots of P1 and P2
    if (r0 <= e) {                                                  // [0, r0) P1 P2 [e + 1, n)
        const int delta = 2 - cnt;
        if (delta > 0) {
            for (int k = n - 1; k > e; --k) { P.x[k + 1] = P.x[k]; P.y[k + 1] = P.y[k]; P.g[k + 1] = P.g[k]; }
        } else if (delta < 0) {
            for (int k = e + 1; k < n; ++k) { P.x[k + delta] = P.x[k]; P.y[k + delta] = P.y[k]; P.g[k + delta] = P.g[k]; }
        }
        P.n = n + delta;
        s1 = r0;
        s2 = r0 + 1;
    } else {                                                        // the run wraps: P2 [e + 1, r0) P1
        for (int k = e + 1; k < r0; ++k) { P.x[k - e] = P.x[k]; P.y[k - e] = P.y[k]; P.g[k - e] = P.g[k]; }
        P.n = r0 - e + 1;
        s1 = P.n - 1;
        s2 = 0;
    }
    P.x[s1] = p1x; P.y[s1] = p1y; P.g[s1] = q;
    P.x[s2] = p2x; P.y[s2] = p2y; P.g[s2] = ge;
    return true;
}

__device__ __forceinline__ double vor_r2max(const Poly& P) {
    double m = 0.0;
    for (int k = 0; k < P.n; ++k) m = fmax(m, __dadd_rn(__dmul_rn(P.x[k], P.x[k]), __dmul_rn(P.y[k], P.y[k])));
    return m;
}

__device__ __forceinline__ double vor_len(const Poly& P, int k) {
    const int k1 = k + 1 == P.n ? 0 : k + 1;
    const double ex = __dsub_rn(P.x[k1], P.x[k]), ey = __dsub_rn(P.y[k1], P.y[k]);
    return __dsqrt_rn(__dadd_rn(__dmul_rn(ex, ex), __dmul_rn(ey, ey)));
}

struct VorArgs {
    const float2* P;      // (ns, N) positions in cell order
    const int* idx;       // (ns, N) original index in cell order
    const int* cs;        // (ns, stride) cell starts
    long long stride;
    int N, nc, m, adj_cap;
    float inv_cell;
    double box, w;        // box, cell edge box / nc
    int* nvor;            // (ns, N) original order
    double* area;         // (ns, N) or null
    int* adj;             // (ns, N, adj_cap) or null
    double2* psi;         // (ns, N) or null
};

__global__ void __launch_bounds__(VOR_THREADS)
voronoi_kernel(const VorArgs a) {
    const int p = blockIdx.x * VOR_THREADS + threadIdx.x;
    if (p >= a.N) return;
    const size_t s = blockIdx.y;
    const float2* Ps = a.P + s * a.N;
    const int* ids = a.idx + s * a.N;
    const int* cs = a.cs + s * a.stride;
    const int nc = a.nc;
    const double box = a.box, half = 0.5 * box;
    const double stop_box = __dmul_rn(half, half);                  // (box / 2)^2
    const float2 ri = Ps[p];
    const int id = ids[p];
    const size_t o = s * a.N + id;

    Poly P;
    bool ok = isfinite(ri.x) && isfinite(ri.y);
    double R2 = 0.0;
    if (ok) {
        P.n = 4;
        P.x[0] = -half; P.y[0] = -half; P.x[1] = half; P.y[1] = -half;
        P.x[2] = half;  P.y[2] = half;  P.x[3] = -half; P.y[3] = half;
        P.g[0] = P.g[1] = P.g[2] = P.g[3] = -1;
        R2 = vor_r2max(P);
        const int c = gr_cell(ri, a.inv_cell, nc);
        const int cx = c % nc, cy = c / nc;
        int k = 1;
        bool all = nc < 3;
        double last_r2 = -1.0;
        int last_id = -1;
        while (true) {
            // smallest key (r2, id) above the last one among the sites of the rings (or of the snapshot)
            double best_r2 = INFINITY;
            int best_id = 0x7fffffff, best_q = -1;
            const int kk = all ? 0 : k;
            for (int oy = -kk; oy <= kk; ++oy) {
                const int y = all ? 0 : (cy + oy + nc) % nc;
                for (int ox = -kk; ox <= kk; ++ox) {
                    int j0 = 0, j1 = a.N;
                    if (!all) {
                        const int cc = y * nc + (cx + ox + nc) % nc;
                        j0 = cs[cc];
                        j1 = cs[cc + 1];
                    }
                    for (int j = j0; j < j1; ++j) {
                        const float2 rj = Ps[j];
                        if (!(isfinite(rj.x) && isfinite(rj.y))) continue;
                        const double dx = vor_disp(rj.x, ri.x, box, half), dy = vor_disp(rj.y, ri.y, box, half);
                        const double r2 = __dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy));
                        if (r2 == 0.0 || r2 > best_r2) continue;             // i itself and coincident sites
                        const int jd = ids[j];
                        if (r2 < last_r2 || (r2 == last_r2 && jd <= last_id)) continue;
                        if (r2 < best_r2 || jd < best_id) {    // r2 <= best_r2 here
                            best_r2 = r2; best_id = jd; best_q = j; }
                    }
                }
            }
            const double stop = fmin(__dmul_rn(4.0, R2), stop_box);
            const double rho = all ? INFINITY : __dsub_rn(__dmul_rn((double)k, a.w), ldexp(box, -20));
            const double cover = all ? INFINITY : (rho > 0.0 ? __dmul_rn(rho, rho) : 0.0);
            if (best_q >= 0 && best_r2 < cover) {
                if (best_r2 >= stop) break;                          // no further site can cut the cell
                const float2 rj = Ps[best_q];
                const double dx = vor_disp(rj.x, ri.x, box, half), dy = vor_disp(rj.y, ri.y, box, half);
                // a site coincident with an earlier one (the same d, so the same r2 and one of the candidates just
                // before) is the same half-plane: it adds nothing, and the neighbour stays the smaller index
                bool twin = false;
                if (best_r2 == last_r2) {
                    for (int t = 0; t < P.n && !twin; ++t) {
                        if (P.g[t] < 0) continue;
                        const float2 rt = Ps[P.g[t]];
                        twin = vor_disp(rt.x, ri.x, box, half) == dx && vor_disp(rt.y, ri.y, box, half) == dy;
                    }
                }
                if (!twin && !vor_clip(P, dx, dy, __dmul_rn(0.5, best_r2), best_q)) { ok = false; break; }
                R2 = vor_r2max(P);
                last_r2 = best_r2;
                last_id = best_id;
                continue;
            }
            if (cover >= stop) break;                                // every site below the stop bound was seen
            ++k;
            if (2 * k + 1 >= nc) all = true;
        }
        ok = ok && __dmul_rn(16.0, R2) < __dmul_rn(box, box);
    }

    int* arow = a.adj ? a.adj + o * a.adj_cap : nullptr;
    if (!ok) {
        a.nvor[o] = -1;
        if (a.area) a.area[o] = nan_d();
        if (a.psi) a.psi[o] = make_double2(nan_d(), nan_d());
        if (arow) for (int t = 0; t < a.adj_cap; ++t) arow[t] = -1;
        return;
    }
    const double lmin = __dmul_rn(VOR_TAU, __dsqrt_rn(R2));
    const int n = P.n;
    // counted edges, their count, the area, and the first counted edge whose normal is in the lower half-plane
    // (dy < 0) after one in the upper one: the start of the order by angle in (-pi, pi]
    double area2 = 0.0;
    int cnt = 0, start = -1, first = -1;
    bool prev_low = false;
    for (int k = n - 1; k >= 0; --k) {
        if (P.g[k] >= 0 && vor_len(P, k) > lmin) {
            prev_low = vor_disp(Ps[P.g[k]].y, ri.y, box, half) < 0.0;
            break;
        }
    }
    for (int k = 0; k < n; ++k) {
        const int k1 = k + 1 == n ? 0 : k + 1;
        area2 = __dadd_rn(area2, __dsub_rn(__dmul_rn(P.x[k], P.y[k1]), __dmul_rn(P.x[k1], P.y[k])));
        if (P.g[k] < 0 || !(vor_len(P, k) > lmin)) continue;
        const bool low = vor_disp(Ps[P.g[k]].y, ri.y, box, half) < 0.0;
        if (first < 0) first = k;
        if (start < 0 && low && !prev_low) start = k;
        prev_low = low;
        ++cnt;
    }
    if (start < 0) start = first < 0 ? 0 : first;
    a.nvor[o] = cnt;
    if (a.area) a.area[o] = __dmul_rn(0.5, area2);
    double L = 0.0;
    int t = 0;
    for (int c = 0; c < n; ++c) {
        const int k = start + c < n ? start + c : start + c - n;
        if (P.g[k] < 0) continue;
        const double l = vor_len(P, k);
        if (!(l > lmin)) continue;
        L = __dadd_rn(L, l);
        if (arow && t < a.adj_cap) arow[t] = ids[P.g[k]];
        ++t;
    }
    if (arow) for (; t < a.adj_cap; ++t) arow[t] = -1;
    if (a.psi) {
        double sx = 0.0, sy = 0.0;
        for (int c = 0; c < n; ++c) {
            const int k = start + c < n ? start + c : start + c - n;
            if (P.g[k] < 0) continue;
            const double l = vor_len(P, k);
            if (!(l > lmin)) continue;
            const float2 rj = Ps[P.g[k]];
            const double dx = vor_disp(rj.x, ri.x, box, half), dy = vor_disp(rj.y, ri.y, box, half);
            const double2 w = unit_pow(dx, dy, a.m);
            const double c_l = __ddiv_rn(l, L);
            sx = __dadd_rn(sx, __dmul_rn(c_l, w.x));
            sy = __dadd_rn(sy, __dmul_rn(c_l, w.y));
        }
        a.psi[o] = make_double2(sx, sy);
    }
}

}  // namespace

int voronoi(ljmd_handle* h, const float2* R_hist, long long S, int* nvor, double* area, int* adj, int adj_cap,
            int m, double2* psi) {
    const long long N = h->p.N;
    if (S == 0) return 0;
    const double box = (double)h->p.box;
    long long nc = (long long)std::floor(std::sqrt((double)N) / VOR_CELL);
    if (nc < 3) nc = 1;                                    // fewer than 3 cells per side: one cell, all particles
    GrGrid g;
    if (int e = gr_grid_alloc(h, S, (int)nc, true, false, &g)) return e;
    VorArgs a{};
    a.P = g.P; a.idx = g.idx; a.cs = g.cs; a.stride = g.stride;
    a.N = (int)N; a.nc = (int)nc; a.m = m; a.adj_cap = adj ? adj_cap : 0;
    a.inv_cell = g.inv_cell;
    a.box = box; a.w = box / (double)nc;
    const unsigned pblocks = (unsigned)((N + VOR_THREADS - 1) / VOR_THREADS);
    for (long long s0 = 0; s0 < S; s0 += g.nb) {
        const unsigned ns = (unsigned)std::min(g.nb, S - s0);
        const size_t off = (size_t)s0 * N;
        if (int e = gr_grid_bin(h, g, R_hist + off, nullptr, ns)) return e;
        a.nvor = nvor + off;
        a.area = area ? area + off : nullptr;
        a.adj = adj ? adj + off * adj_cap : nullptr;
        a.psi = psi ? psi + off : nullptr;
        voronoi_kernel<<<dim3(pblocks, ns), VOR_THREADS, 0, h->stream>>>(a);
        LJ_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    return 0;
}

}  // namespace ljmd
