// gr.cu — the pair-distance histogram of calculate_g_r (get_histogram, MD:117-124) through a cell grid:
// only pairs in neighbouring cells of a periodic nc x nc grid of edge >= r_max are visited, so a histogram
// that ends at r_max costs O(S N rho pi r_max^2) instead of the O(S N^2) of gr_hist_kernel (allpairs.cu).
// The counts are those of gr_hist_kernel bit for bit: the same fp32 r of every pair, the same binning
// (gr_bin), exact integer counts.  ljmd_gr_hist_rmax (api.cu) decides which of the two kernels runs.
//
// Per batch of snapshots (blockIdx.y = snapshot in the batch), four launches:
//   gr_count_kernel    cell of every particle, atomic per-cell count; the returned slot is its rank in the cell
//   gr_scan_kernel     in-place exclusive scan of the counts -> cell_start[nc^2 + 1] (one CTA per snapshot)
//   gr_scatter_kernel  positions in cell order
//   gr_cells_kernel    the half stencil of every cell into a per-CTA shared histogram
// Snapshots are batched up to GR_BATCH_BYTES of scratch: at N = 4096 all 100 snapshots of the driver take
// one batch (four launches per call); at N = 16 M a batch holds two.
//
// The same grid serves the bond order (bond.cu: the first three launches, then its own kernel) and the
// weighted histogram g_m(r) of ljmd_bond_corr (the W instantiations).  The scatter's W instantiation also
// records each particle's original index (bond order: 16 B of scratch per particle instead of 12) or its psi
// in cell order (g_m(r): 28 B).
#include "ljmd_device.cuh"

#include <algorithm>
#include <cmath>

namespace ljmd {

struct Gr {
    void*  buf = nullptr;   // one batch of snapshots binned into the grid (GrGrid, gr_grid_alloc)
    size_t bytes = 0;
};

namespace {

constexpr size_t   GR_BATCH_BYTES  = size_t(512) << 20;
constexpr int      GRB_THREADS     = 256;           // count / scatter
constexpr int      GRS_THREADS     = 1024;          // scan
constexpr int      GRC_THREADS     = 256;           // pair kernel: one warp per home cell
constexpr int      GRC_WARPS       = GRC_THREADS / 32;
constexpr int      GRC_CELLS       = 64;            // home cells per CTA
// A CTA's shared counters are 32-bit.  A warp bins at most GRC_WARP_BUDGET pairs into them (counted
// conservatively, 32 per staged target); beyond that (a clumped state) it adds to the global counts
// directly, so the CTA's counters stay below GRC_WARPS * (2^28 + 1024) < 2^32.
constexpr long long GRC_WARP_BUDGET = 1ll << 28;

__global__ void __launch_bounds__(GRB_THREADS)
gr_count_kernel(const float2* __restrict__ R, int N, float inv_cell, int nc, int* __restrict__ cstart,
                long long stride, int* __restrict__ rank) {
    const int i = blockIdx.x * GRB_THREADS + threadIdx.x;
    if (i >= N) return;
    const size_t s = blockIdx.y;
    const int c = gr_cell(R[s * N + i], inv_cell, nc);
    rank[s * N + i] = atomicAdd(&cstart[s * stride + c], 1);
}

// In-place exclusive scan of the L counts of snapshot blockIdx.y (L = nc^2 + 1: the last count is 0, so
// cstart[nc^2] ends as N).  stride is a multiple of 4 and the padding past L is zero.
__global__ void __launch_bounds__(GRS_THREADS)
gr_scan_kernel(int* __restrict__ cstart, long long stride, int L) {
    __shared__ int swarp[GRS_THREADS / 32];
    __shared__ int stotal;
    int4* p = reinterpret_cast<int4*>(cstart + (size_t)blockIdx.y * stride);
    const int n4 = (L + 3) / 4;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int carry = 0;
    for (int base = 0; base < n4; base += GRS_THREADS) {
        const int k = base + threadIdx.x;
        const int4 v = (k < n4) ? p[k] : make_int4(0, 0, 0, 0);
        const int sum = v.x + v.y + v.z + v.w;
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) swarp[w] = incl;
        __syncthreads();
        if (w == 0) {
            const int x = swarp[lane];
            int xi = x;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, xi, o);
                if (lane >= o) xi += t;
            }
            swarp[lane] = xi - x;
            if (lane == 31) stotal = xi;
        }
        __syncthreads();
        if (k < n4) {
            int4 o;
            o.x = carry + swarp[w] + incl - sum;
            o.y = o.x + v.x;
            o.z = o.y + v.y;
            o.w = o.z + v.z;
            p[k] = o;
        }
        carry += stotal;
        __syncthreads();                       // swarp / stotal are rewritten by the next chunk
    }
}

// W: also, where the pointers are given, the original index of every particle in cell order (idx) and its psi (Ppsi)
template <bool W>
__global__ void __launch_bounds__(GRB_THREADS)
gr_scatter_kernel(const float2* __restrict__ R, int N, float inv_cell, int nc, const int* __restrict__ cstart,
                  long long stride, const int* __restrict__ rank, float2* __restrict__ P,
                  int* __restrict__ idx, const double2* __restrict__ psi, double2* __restrict__ Ppsi) {
    const int i = blockIdx.x * GRB_THREADS + threadIdx.x;
    if (i >= N) return;
    const size_t s = blockIdx.y;
    const float2 r = R[s * N + i];
    const int c = gr_cell(r, inv_cell, nc);
    const size_t o = s * N + cstart[s * stride + c] + rank[s * N + i];
    P[o] = r;
    if constexpr (W) {
        if (idx) idx[o] = i;
        if (psi) Ppsi[o] = psi[s * N + i];
    }
}

struct GrCellsArgs {
    const float2* P;              // (ns, N) positions in cell order
    const int* cstart;            // (ns, stride) cell starts
    long long stride;
    int N, nc, nbins;
    float box, timg, cap;
    const float* edges;           // nbins + 1
    unsigned long long* counts;   // (ns, nbins)
    const double2* psi;           // W: (ns, N) psi in cell order
    unsigned long long* wsum;     // W: (ns, nbins) sums of llrint(w 2^24) (two's complement)
};

// W: byte offset of the CTA's 64-bit weight sums, after the pair kernel's other shared arrays (8-aligned)
__host__ __device__ constexpr size_t grc_wsum_offset(int nbins) {
    return (sizeof(float2) * GRC_WARPS * 32 + sizeof(float) * (2 * (size_t)nbins + 1) + 7) / 8 * 8;
}

// One warp per home cell c: its particles, 32 at a time one per lane, against the targets of the half
// stencil - c itself (j > i), E, NE, N and NW, periodic - staged 32 at a time in the warp's shared slots.
// Cells of any occupancy are walked in these chunks.  For nc >= 3 the five cells are distinct and every
// unordered pair of particles in adjacent cells is visited exactly once.
// W (ljmd_bond_corr): a counted pair with a finite weight w_ij (bond_pair_weight) also adds llrint(w 2^24) to
// wsum; a pair whose weight is not finite is neither counted nor summed.
template <bool W>
__global__ void __launch_bounds__(GRC_THREADS)
gr_cells_kernel(const GrCellsArgs a) {
    extern __shared__ unsigned char smem_raw[];
    float2*   stage  = reinterpret_cast<float2*>(smem_raw);                  // GRC_WARPS x 32
    float*    sedges = reinterpret_cast<float*>(stage + GRC_WARPS * 32);     // nbins + 1
    unsigned* shist  = reinterpret_cast<unsigned*>(sedges + a.nbins + 1);    // nbins
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nbins = a.nbins, nc = a.nc;
    const size_t s = blockIdx.y;
    const float2* P = a.P + s * a.N;
    const int* cs = a.cstart + s * a.stride;
    unsigned long long* out = a.counts + s * nbins;
    unsigned long long* swsum = nullptr;
    unsigned long long* wout = nullptr;
    const double2* psi = nullptr;
    if constexpr (W) {
        swsum = reinterpret_cast<unsigned long long*>(smem_raw + grc_wsum_offset(nbins));   // nbins
        wout = a.wsum + s * nbins;
        psi = a.psi + s * a.N;
        for (int k = tid; k < nbins; k += GRC_THREADS) swsum[k] = 0ull;
    }
    for (int k = tid; k <= nbins; k += GRC_THREADS) sedges[k] = a.edges[k];
    for (int k = tid; k < nbins; k += GRC_THREADS) shist[k] = 0u;
    __syncthreads();
    const float lo = sedges[0], hi = fminf(sedges[nbins], a.cap);
    const float scale = (float)nbins / (sedges[nbins] - lo);
    float2* sj = stage + warp * 32;
    long long used = 0;
    const int c_end = min(nc * nc, (int)(blockIdx.x + 1) * GRC_CELLS);
    for (int c = blockIdx.x * GRC_CELLS + warp; c < c_end; c += GRC_WARPS) {
        const int cx = c % nc, cy = c / nc;
        const int xe = (cx + 1 == nc) ? 0 : cx + 1, xw = (cx == 0) ? nc - 1 : cx - 1;
        const int yn = (cy + 1 == nc) ? 0 : cy + 1;
        const int a0 = cs[c], a1 = cs[c + 1];
        for (int ib = a0; ib < a1; ib += 32) {
            const int i = ib + lane;
            const bool has_i = i < a1;
            const float2 ri = has_i ? P[i] : make_float2(0.0f, 0.0f);
            double2 pi = make_double2(0.0, 0.0);
            if constexpr (W) pi = has_i ? psi[i] : pi;
            for (int t = 0; t < 5; ++t) {
                int b0 = ib, b1 = a1;                                       // t == 0: own cell, j > i
                if (t > 0) {
                    const int nx = (t == 1 || t == 2) ? xe : (t == 3 ? cx : xw);
                    const int nb = (t == 1 ? cy : yn) * nc + nx;
                    b0 = cs[nb];
                    b1 = cs[nb + 1];
                }
                for (int jb = b0; jb < b1; jb += 32) {
                    const int n = min(32, b1 - jb);
                    __syncwarp();
                    if (lane < n) sj[lane] = P[jb + lane];
                    __syncwarp();
                    const bool direct = used > GRC_WARP_BUDGET;
                    used += 32 * n;
                    if (!has_i) continue;
                    for (int q = 0; q < n; ++q) {
                        if (t == 0 && jb + q <= i) continue;
                        const float dx = min_image(__fsub_rn(ri.x, sj[q].x), a.box, a.timg);
                        const float dy = min_image(__fsub_rn(ri.y, sj[q].y), a.box, a.timg);
                        const float r = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
                        const int b = gr_bin(r, sedges, nbins, lo, hi, scale);
                        if (b < 0) continue;
                        if constexpr (W) {
                            long long wq;
                            if (!bond_pair_weight(pi, psi[jb + q], wq)) continue;
                            if (direct) atomicAdd(&wout[b], (unsigned long long)wq);
                            else        atomicAdd(&swsum[b], (unsigned long long)wq);
                        }
                        if (direct) atomicAdd(&out[b], 1ull);
                        else        atomicAdd(&shist[b], 1u);
                    }
                }
            }
        }
    }
    __syncthreads();
    for (int k = tid; k < nbins; k += GRC_THREADS)
        if (shist[k]) atomicAdd(&out[k], (unsigned long long)shist[k]);
    if constexpr (W) {
        for (int k = tid; k < nbins; k += GRC_THREADS)
            if (swsum[k]) atomicAdd(&wout[k], swsum[k]);
    }
}

}  // namespace

// Cells per side of the g(r) grid for pairs up to r_max.  Every pair with fp32 r <= r_max must lie in
// cells at most one apart on each axis.  Margin: with the cell width w = box / nc and inv_cell =
// fl(nc / box), t = fl(x * inv_cell) differs from x / w by at most (2u + u^2)(x / w), about 2u nc cells
// (u = 2^-24; two roundings; x in [0, box]) and the cell is trunc(t), clamped to nc - 1 (the clamp only moves x == box,
// or t rounded up to nc, into the last cell, which holds x / w in [nc - 1, nc]).  So a particle in cell
// k has x / w in [k - 2u nc, k + 1 + 2u nc], and two particles whose cells are >= 2 apart (periodically)
// are at least w - 4u box apart in every periodic image.  The fp32 dx = min_image(fl(xi - xj)) is within
// 2u box of the exact difference of that image (two roundings of values <= box), and r = fl(sqrt(fl(
// fl(dx^2) + fl(dy^2)))) >= |dx| (1 - 2u) (monotone roundings).  Together r >= w - 8u box = w - 2^-21 box.
// With r_max_eff = r_max + 2^-20 box and w >= r_max_eff such a pair has r > r_max and is never binned.
// Larger cells are always correct, so nc is also capped at sqrt(N): a tiny r_max must not ask for more
// cells than particles.
int gr_grid_side(long long N, float box, float r_max) {
    const double eff = (double)r_max + std::ldexp((double)box, -20);
    long long nc = (long long)std::floor((double)box / eff);
    while (nc > 0 && (double)box / (double)nc < eff) --nc;
    long long cap = (long long)std::sqrt((double)N);
    while (cap * cap > N) --cap;
    while ((cap + 1) * (cap + 1) <= N) ++cap;
    return (int)std::max<long long>(0, std::min(nc, cap));
}

int gr_grid_alloc(ljmd_handle* h, long long S, int nc, bool with_idx, bool with_psi, GrGrid* g) {
    const long long N = h->p.N;
    const long long ncell = (long long)nc * nc;
    const long long stride = (ncell + 1 + 3) / 4 * 4;                       // int4-aligned rows of cell starts
    const size_t extra = (with_psi ? sizeof(double2) : 0) + (with_idx ? sizeof(int) : 0);
    const size_t per = sizeof(int) * stride + (sizeof(float2) + sizeof(int) + extra) * (size_t)N;
    const long long nb = std::max<long long>(1, std::min<long long>(std::min<long long>(S, 65535),
                                                                    (long long)(GR_BATCH_BYTES / per)));
    const size_t need = per * (size_t)nb;
    if (!h->gr) h->gr = new Gr();
    Gr* b = h->gr;
    if (b->bytes < need) {
        LJ_CUDA(cudaFree(b->buf));
        b->buf = nullptr;
        b->bytes = 0;
        LJ_CUDA(cudaMalloc(&b->buf, need));
        b->bytes = need;
    }
    // cell starts (rows of 16 B) | psi (with_psi) | positions | ranks | original indices (with_idx)
    g->cs = reinterpret_cast<int*>(b->buf);
    double2* after_cs = reinterpret_cast<double2*>(g->cs + nb * stride);
    g->psi = with_psi ? after_cs : nullptr;
    g->P = reinterpret_cast<float2*>(with_psi ? after_cs + nb * N : after_cs);
    g->rank = reinterpret_cast<int*>(g->P + nb * N);
    g->idx = with_idx ? g->rank + nb * N : nullptr;
    g->stride = stride;
    g->nb = nb;
    g->nc = nc;
    g->inv_cell = (float)nc / h->p.box;
    return 0;
}

int gr_grid_bin(ljmd_handle* h, const GrGrid& g, const float2* R, const double2* psi, unsigned ns) {
    const long long N = h->p.N;
    cudaStream_t st = h->stream;
    const long long ncell = (long long)g.nc * g.nc;
    const unsigned pblocks = (unsigned)((N + GRB_THREADS - 1) / GRB_THREADS);
    LJ_CUDA(cudaMemsetAsync(g.cs, 0, sizeof(int) * g.stride * ns, st));
    gr_count_kernel<<<dim3(pblocks, ns), GRB_THREADS, 0, st>>>(R, (int)N, g.inv_cell, g.nc, g.cs, g.stride, g.rank);
    LJ_CUDA(cudaGetLastError());
    gr_scan_kernel<<<dim3(1, ns), GRS_THREADS, 0, st>>>(g.cs, g.stride, (int)(ncell + 1));
    LJ_CUDA(cudaGetLastError());
    if (g.idx || g.psi)
        gr_scatter_kernel<true><<<dim3(pblocks, ns), GRB_THREADS, 0, st>>>(R, (int)N, g.inv_cell, g.nc, g.cs, g.stride,
                                                                          g.rank, g.P, g.idx, psi, g.psi);
    else
        gr_scatter_kernel<false><<<dim3(pblocks, ns), GRB_THREADS, 0, st>>>(R, (int)N, g.inv_cell, g.nc, g.cs, g.stride,
                                                                           g.rank, g.P, nullptr, nullptr, nullptr);
    LJ_CUDA(cudaGetLastError());
    h->launches += 3;
    return 0;
}

int gr_cells_hist(ljmd_handle* h, const float2* R_hist, long long S, int nbins, const float* edges,
                  float r_max, int nc, long long* counts, const double2* psi, long long* wsum) {
    const long long N = h->p.N;
    const bool W = psi != nullptr;
    cudaStream_t st = h->stream;
    LJ_CUDA(cudaMemsetAsync(counts, 0, sizeof(long long) * S * nbins, st));
    if (W) LJ_CUDA(cudaMemsetAsync(wsum, 0, sizeof(long long) * S * nbins, st));
    if (S == 0) return 0;
    GrGrid g;
    if (int e = gr_grid_alloc(h, S, nc, false, W, &g)) return e;

    GrCellsArgs a{};
    a.P = g.P; a.cstart = g.cs; a.stride = g.stride;
    a.N = (int)N; a.nc = nc; a.nbins = nbins;
    a.box = h->pc.box; a.timg = h->pc.timg; a.cap = r_max;
    a.edges = edges;
    a.psi = g.psi;
    const size_t smem = W ? grc_wsum_offset(nbins) + sizeof(long long) * nbins
                          : sizeof(float2) * GRC_WARPS * 32 + sizeof(float) * (nbins + 1) + sizeof(unsigned) * nbins;
    void (*kernel)(const GrCellsArgs) = W ? gr_cells_kernel<true> : gr_cells_kernel<false>;
    LJ_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const unsigned cblocks = (unsigned)(((long long)nc * nc + GRC_CELLS - 1) / GRC_CELLS);
    for (long long s0 = 0; s0 < S; s0 += g.nb) {
        const unsigned ns = (unsigned)std::min(g.nb, S - s0);
        if (int e = gr_grid_bin(h, g, R_hist + (size_t)s0 * N, W ? psi + (size_t)s0 * N : nullptr, ns)) return e;
        a.counts = reinterpret_cast<unsigned long long*>(counts) + (size_t)s0 * nbins;
        if (W) a.wsum = reinterpret_cast<unsigned long long*>(wsum) + (size_t)s0 * nbins;
        kernel<<<dim3(cblocks, ns), GRC_THREADS, smem, st>>>(a);
        LJ_CUDA(cudaGetLastError());
        h->launches += 1;
    }
    return 0;
}

void gr_destroy(ljmd_handle* h) {
    if (!h->gr) return;
    cudaFree(h->gr->buf);
    delete h->gr;
    h->gr = nullptr;
}

}  // namespace ljmd
