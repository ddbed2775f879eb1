// bond.cu — bond-orientational order psi_m(i) = (1/n_i) sum_{j in nb(i)} exp(i m theta_ij) of every particle of
// S snapshots (ljmd_bond_order), through the periodic cell grid of g(r) (gr.cu).
//
// Neighbours.  j != i with 0 < r_ij <= r_nb, where r_ij is exactly the fp32 r that g(r) bins (min_image of
// __fsub_rn, __fmul_rn / __fadd_rn, __fsqrt_rn), so the neighbour set is defined in fp32 and a CPU restatement
// reproduces it bit for bit.  A particle with a non-finite coordinate has r = NaN or inf to everyone: it is no
// particle's neighbour, and it gets psi = NaN, n = 0.
//
// Bond term.  d = min_image(fl(x_j - x_i)) from i to j (the sign matters for odd m), converted to double (exact);
// then in double, every operation rounded once (no contraction): r_d = sqrt(d_x^2 + d_y^2), u = d / r_d, and
// w = u^m by m - 1 sequential complex products w <- w u = (ac - bd, ad + bc).
//
// Fixed-point sum.  q = llrint(w 2^32) per component, summed in int64: exact (N < 2^31 terms of |q| <= 2^32 + 1)
// and independent of the order of the terms, hence of the cell order that the atomic ranks of gr_count_kernel
// produce.  psi_i = (double)(sum q) 2^-32 / n_i, and 0 when n_i = 0.
//
// Bound, per component of psi_i, against exact arithmetic on the fp32 bond vectors (u = 2^-53):
//   |u_x - d_x / |d|| <= 3u (r_d: <= 2u relative; the quotient one more rounding), so |u| - 1 <= 5u;
//   each complex product adds <= 3u (two products and a sum, |terms| <= 1) and carries the error of u:
//   |w - (d/|d|)^m| <= 9 m u;  quantisation <= 2^-33;  (double) of the sum and the division: <= 2u (1 + 2^-32).
// So |psi_i - exact| <= 2^-33 + (9m + 3) 2^-53 per component, below 1.2e-10 for every m in [1, 12].
//
// Layout (measured, DESIGN.md 4.6): one thread per particle in cell order, grid.y = snapshot in the batch.  Each
// thread walks the full 9-cell stencil of its own cell (cells of edge >= r_nb + the gr_grid_side margin: ~1.8
// particles per cell at r_nb = 1.5 and rho = 0.8, so ~16 candidates) and writes psi and n to its ORIGINAL index.
// Neighbouring threads hold neighbouring cells, so the candidates' loads hit L1.  With fewer than 3 cells per
// side (r_nb > box / 3: tiny N) the grid is one cell and every thread visits all N particles.
#include "ljmd_device.cuh"

#include <algorithm>

namespace ljmd {

namespace {

constexpr int BO_THREADS = 256;

__device__ __forceinline__ void bond_term(float dxf, float dyf, int m, long long& sx, long long& sy) {
    const double dx = (double)dxf, dy = (double)dyf;
    const double r = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    const double ux = __ddiv_rn(dx, r), uy = __ddiv_rn(dy, r);
    double wx = ux, wy = uy;
    for (int k = 1; k < m; ++k) {
        const double a = wx, b = wy;
        wx = __dsub_rn(__dmul_rn(a, ux), __dmul_rn(b, uy));
        wy = __dadd_rn(__dmul_rn(a, uy), __dmul_rn(b, ux));
    }
    sx += llrint(__dmul_rn(wx, 4294967296.0));
    sy += llrint(__dmul_rn(wy, 4294967296.0));
}

__global__ void __launch_bounds__(BO_THREADS)
bond_order_kernel(const float2* __restrict__ P, const int* __restrict__ idx, const int* __restrict__ cstart,
                  long long stride, int N, int nc, float inv_cell, float box, float timg, float r_nb, int m,
                  double2* __restrict__ psi, int* __restrict__ nnb) {
    const int p = blockIdx.x * BO_THREADS + threadIdx.x;
    if (p >= N) return;
    const size_t s = blockIdx.y;
    const float2* Ps = P + s * N;
    const int* cs = cstart + s * stride;
    const float2 ri = Ps[p];
    const bool ok = isfinite(ri.x) && isfinite(ri.y);
    long long sx = 0, sy = 0;
    int n = 0;
    if (ok) {
        const int c = gr_cell(ri, inv_cell, nc);
        const int cx = c % nc, cy = c / nc;
        const int o = nc >= 3 ? 1 : 0;                 // nc < 3 only as nc == 1: one cell, all pairs
        for (int oy = -o; oy <= o; ++oy) {
            const int y = (cy + oy + nc) % nc;
            for (int ox = -o; ox <= o; ++ox) {
                const int cc = y * nc + (cx + ox + nc) % nc;
                const int j1 = cs[cc + 1];
                for (int j = cs[cc]; j < j1; ++j) {
                    const float2 rj = Ps[j];
                    const float dx = min_image(__fsub_rn(rj.x, ri.x), box, timg);
                    const float dy = min_image(__fsub_rn(rj.y, ri.y), box, timg);
                    const float r = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
                    if (!(r > 0.0f && r <= r_nb)) continue;   // also drops j == i and non-finite j
                    bond_term(dx, dy, m, sx, sy);
                    ++n;
                }
            }
        }
    }
    double2 v = make_double2(0.0, 0.0);
    if (!ok) {
        v.x = v.y = __longlong_as_double(0x7ff8000000000000ll);
    } else if (n > 0) {
        v.x = __ddiv_rn(__dmul_rn(__ll2double_rn(sx), 0x1p-32), (double)n);
        v.y = __ddiv_rn(__dmul_rn(__ll2double_rn(sy), 0x1p-32), (double)n);
    }
    const size_t o = s * N + idx[s * N + p];
    psi[o] = v;
    if (nnb) nnb[o] = n;
}

}  // namespace

int bond_order(ljmd_handle* h, const float2* R_hist, long long S, int m, float r_nb, double2* psi, int* nnb) {
    const long long N = h->p.N;
    if (S == 0) return 0;
    int nc = gr_grid_side(N, h->p.box, r_nb);
    if (nc < 3) nc = 1;                                   // the 9-cell stencil needs 3 distinct cells per side
    GrGrid g;
    if (int e = gr_grid_alloc(h, S, nc, true, false, &g)) return e;
    const unsigned pblocks = (unsigned)((N + BO_THREADS - 1) / BO_THREADS);
    for (long long s0 = 0; s0 < S; s0 += g.nb) {
        const unsigned ns = (unsigned)std::min(g.nb, S - s0);
        if (int e = gr_grid_bin(h, g, R_hist + (size_t)s0 * N, nullptr, ns)) return e;
        bond_order_kernel<<<dim3(pblocks, ns), BO_THREADS, 0, h->stream>>>(
            g.P, g.idx, g.cs, g.stride, (int)N, nc, g.inv_cell, h->pc.box, h->pc.timg, r_nb, m,
            psi + (size_t)s0 * N, nnb ? nnb + (size_t)s0 * N : nullptr);
        LJ_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    return 0;
}

}  // namespace ljmd
