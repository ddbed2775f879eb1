// ljmd_internal.cuh — shared declarations of the B200-native LJ-MD library (sm_100a only).
// The public C ABI is include/ljmd.h; nothing here is exported.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include <vector>

#include "../../include/ljmd.h"

#define LJMD_MAX_RANKS 8
#define LJMD_GR_MAXBINS 8192      // bins of a g(r) histogram: one 32-bit counter each in a CTA's shared memory

namespace ljmd {

void set_error(const char* fmt, ...);

#define LJ_CUDA(expr)                                                                  \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            ljmd::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                            __FILE__, __LINE__);                                       \
            return (int)_e;                                                            \
        }                                                                              \
    } while (0)

// ----------------------------------------------------------------------------------------
// Pair-interaction constants, precomputed on the host once per handle.
//   timg : exact minimum-image threshold.  The reference computes n = round(d / box) with a
//          true fp32 division and round-half-even (MD:46-48).  For |d| <= box that n is -1, 0
//          or +1, and n != 0  <=>  |d| >= timg where timg is the smallest fp32 with
//          fl(timg / box) > 0.5 (fp32 division is monotone).  One compare therefore
//          reproduces div+round bit for bit, and d - box*n is a single rounded subtract
//          (box*n is exact) exactly as in the reference.
//   c12,c6 : 48 eps sigma^12, 24 eps sigma^6   (force scalar  f = (c12*ir6 - c6) * ir6 * ir2)
//   d12,d6 :  4 eps sigma^12,  4 eps sigma^6   (pair energy   e = (d12*ir6 - d6) * ir6)
struct PairConsts {
    float box, timg, rc2;
    float c12, c6, d12, d6;
    float one;      // 1.0f passed at run time (blocks an unwanted FMA contraction, see pair2_eval)
    int   cutoff;   // 0 = none (the reference), 1 = plain truncation at rc
};

PairConsts make_pair_consts(float box, float sigma, float eps, float rc);

// ----------------------------------------------------------------------------------------
// Run-control block shared by the all-pairs and the cell-list step loops.
struct RunCtl {
    long long nsteps;
    long long sample_every;   // 0 = no trajectory
    long long S;              // number of trajectory rows = nsteps / sample_every  (MD:88)
    long long energy_every;   // 0 = no energies
    long long thermo_every;   // 0 = NVE
    float     thermo_kT;
    float2*   traj;           // (S,N,2)
    float*    ke_pe;          // (ceil(nsteps/energy_every),2)
    int       blocked;        // multi-GPU: R/V pointers address the rank's INDEX BLOCK [rank N/P, (rank+1) N/P)
                              // only (ljmd_run_blocked) instead of the full replicated arrays
};

struct AllPairs;   // allpairs.cu
struct Cells;      // cells.cu
struct Dist;       // dist.cu
struct Gr;         // gr.cu
struct Sk;         // sk.cu

}  // namespace ljmd

struct ljmd_handle {
    ljmd_params      p;
    ljmd::PairConsts pc;
    int              path;        // resolved LJMD_PATH_*
    cudaStream_t     stream;
    int              num_sms;
    ljmd::AllPairs*  ap;
    ljmd::Cells*     cells;
    ljmd::Dist*      dist;
    ljmd::Gr*        gr;          // cell-grid scratch of g(r), psi_m, g_m(r), clusters and Voronoi (allocated on the first call that uses it)
    cudaEvent_t      ev0, ev1;
    bool             timed;
    long long        launches;
    int              rank, nranks;
    long long        spin_limit;  // clocks a device-side spin wait may last (0 = unlimited)
    float2*          blk_full[4]; // all-pairs ljmd_run_blocked: replicated in / out arrays (allocated on first use)
    ljmd::Sk*        sk;          // density-mode partial sums (allocated on the first ljmd_density_modes)
};

namespace ljmd {

// allpairs.cu
int  ap_create(ljmd_handle* h);
void ap_destroy(ljmd_handle* h);
// nsteps == 0: evaluate F (optional), PE (optional) and the virial W (optional) of R_in only.
// vir_out != nullptr selects the virial kernels: W of R_in (nsteps == 0), else vir_out[i / energy_every]
// = W of the post-step state on every row that ke_pe receives (single GPU only).
int  ap_run(ljmd_handle* h, const float2* R_in, const float2* V_in, float2* R_out, float2* V_out,
            float2* F_out, float* pe_out, const RunCtl& rc, float* vir_out);
int  ap_check_error(ljmd_handle* h);
int  ap_mode(ljmd_handle* h);

// cells.cu
int  cells_create(ljmd_handle* h);
void cells_destroy(ljmd_handle* h);
int  cells_run(ljmd_handle* h, const float2* R_in, const float2* V_in, float2* R_out,
               float2* V_out, float2* F_out, float* pe_out, const RunCtl& rc, float* vir_out);   // as ap_run
int  cells_geometry(ljmd_handle* h, int* nrows, int* nbx, int* kbins, float* inv_hy, float* inv_wx);
int  cells_assign(ljmd_handle* h, const float2* R, int* cell_id, int* cell_count);
int  cells_neighbor_count(ljmd_handle* h, const float2* R, float radius, int* nbr_count);
long long cells_last_rebuilds(ljmd_handle* h);
int  cells_check_error(ljmd_handle* h);

// gr.cu: the g(r) pair-distance histogram, over all pairs or through a periodic nc x nc cell grid of edge >= r_max.
// psi != nullptr: the weighted histogram of ljmd_bond_corr (psi (S,N) in particle order, wsum (S,nbins)).
// Every pair; cap: pairs with r > cap are dropped too (+INFINITY: the plain histogram of ljmd_gr_hist)
int  gr_allpairs_hist(ljmd_handle* h, const float2* R_hist, long long S, int nbins, const float* edges,
                      float cap, long long* counts, const double2* psi = nullptr, long long* wsum = nullptr);
// The pairs with r <= r_max, through the grid when it has >= 3 cells per side, else gr_allpairs_hist
int  gr_pair_hist(ljmd_handle* h, const float2* R_hist, long long S, int nbins, const float* edges,
                  float r_max, long long* counts, const double2* psi = nullptr, long long* wsum = nullptr);
int  gr_grid_side(long long N, float box, float r_max);   // nc for this r_max
// One batch of snapshots binned into the nc x nc grid, in the handle's Gr scratch (rows of the batch: nb).
// with_idx: also idx (original index of each particle in cell order, for the bond order);
// with_psi: also psi (its psi in cell order, for the weighted histogram of ljmd_bond_corr).
struct GrGrid {
    int*      cs;        // (nb, stride) cell starts; cs[c + 1] - cs[c] particles in cell c
    float2*   P;         // (nb, N) positions in cell order
    int*      rank;      // (nb, N) rank of each particle in its cell
    int*      idx;       // with_idx: (nb, N) original index in cell order, else nullptr
    double2*  psi;       // with_psi: (nb, N) psi in cell order, else nullptr
    long long stride, nb;
    int       nc;
    float     inv_cell;  // fl(nc / box), the multiplier of gr_cell
};
int  gr_grid_alloc(ljmd_handle* h, long long S, int nc, bool with_idx, bool with_psi, GrGrid* g);
// count / scan / scatter of ns <= nb snapshots R (ns, N); psi (ns, N) is permuted too when given (with_psi)
int  gr_grid_bin(ljmd_handle* h, const GrGrid& g, const float2* R, const double2* psi, unsigned ns);
void gr_destroy(ljmd_handle* h);

// bond.cu: bond-orientational order psi_m of every particle (see ljmd_bond_order)
int  bond_order(ljmd_handle* h, const float2* R_hist, long long S, int m, float r_nb, double2* psi, int* nnb);

// cluster.cu: connected components within r_link of every snapshot (see ljmd_clusters); mask and sizes may be null
int  clusters(ljmd_handle* h, const float2* R_hist, long long S, float r_link, const unsigned char* mask,
              int* labels, int* sizes);

// voronoi.cu: Voronoi cell of every particle (see ljmd_voronoi); area, adj and psi may be null
int  voronoi(ljmd_handle* h, const float2* R_hist, long long S, int* nvor, double* area, int* adj, int adj_cap,
             int m, double2* psi);

// sk.cu: density modes rho_k of S snapshots for K integer wave vectors (see ljmd_density_modes)
int  sk_density_modes(ljmd_handle* h, const float2* R_hist, long long S, const int2* nvec, long long K,
                      double2* rho);
void sk_destroy(ljmd_handle* h);

// api.cu
int  create_common(ljmd_t** out, const ljmd_params* p, int rank, int nranks, const void* nccl_uid);

// dist.cu (NCCL over NVLink for bootstrap / final replication; IPC peer mapping)
int  dist_init(ljmd_handle* h, const void* nccl_unique_id);
void dist_destroy(ljmd_handle* h);
int  dist_share(ljmd_handle* h, void* local_base, void** peer_bases /*[nranks]*/);
int  dist_allgather(ljmd_handle* h, void* buf, size_t bytes_per_rank);   // in place, slab `rank`
int  dist_allgather_from(ljmd_handle* h, const void* send, void* recv, size_t bytes_per_rank);
int  dist_allreduce_f32(ljmd_handle* h, float* buf, size_t n);
int  dist_barrier(ljmd_handle* h);                      // cross-rank barrier in stream order

// pairlaw.cu
int  pairlaw_accel(int law, const float2* pos, const float* mass, long long n, float G, float2* acc,
                   cudaStream_t stream);

// probe.cu
int  fp32_peak_probe(int device, int packed, float* tflops);

}  // namespace ljmd
