/*
 * ljmd.h — C ABI of the B200-native 2-D Lennard-Jones molecular-dynamics hot path.
 *
 * This is the drop-in boundary for the per-step hot path of the reference script
 *   molecular_dynamics_jax_single-host_workload.py   (cited below as MD:<line>)
 * The reference has no FFI of its own: its "interface" is the set of Python closures
 * defined inside main() (MD:46-131).  Every entry point below names the closure it
 * replaces.  The reference-side binding a maintainer would add is the ctypes stub
 * shown in INTEGRATION.md (and shipped as jax_tpus_benchmark_physics_simulation_b200/_lib.py).
 *
 * Conventions
 *   - plain C: pointers + sizes, no C++/torch types.
 *   - all `*_dev` / R / V / F / traj / ke_pe pointers are DEVICE pointers owned by the
 *     caller, contiguous row-major (N,2) float32 (== float2 AoS), 8-byte aligned.
 *   - every call enqueues work on the stream given to ljmd_create() and returns
 *     without synchronising (JAX-style async dispatch; MD:145 block_until_ready maps
 *     to a stream synchronise done by the caller).
 *   - inputs are never modified (the reference closures are pure); R_out/V_out may
 *     alias R_in/V_in.
 *   - return value 0 = success; >0 = cudaError_t; <0 = LJMD_E_* library code.
 *     Nothing throws or aborts across the ABI.  ljmd_last_error() gives text.
 *   - a handle is not thread-safe: one per device, driven by one host thread.
 */
#ifndef LJMD_H_
#define LJMD_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LJMD_ABI_VERSION 1

/* library (negative) error codes */
#define LJMD_E_INVALID   (-1)   /* bad argument                                   */
#define LJMD_E_STATE     (-2)   /* call not valid for this handle's configuration */
#define LJMD_E_NCCL      (-3)   /* NCCL failure (see ljmd_last_error)             */
#define LJMD_E_NOMEM     (-4)
#define LJMD_E_UNSUPPORTED (-5)
#define LJMD_E_OVERFLOW  (-6)   /* device flag: neighbour list / slab capacity exceeded - results invalid */
#define LJMD_E_TIMEOUT   (-7)   /* device flag: a grid barrier or cross-GPU wait timed out - results invalid */

/* force-path selection */
#define LJMD_PATH_AUTO      0   /* all-pairs for N <= 131072, else cell list      */
#define LJMD_PATH_ALLPAIRS  1   /* dense N x N, the reference's formulation MD:50-62 */
#define LJMD_PATH_CELLS     2   /* sorted strip cells, 3 contiguous ranges / particle (requires rc) */

typedef struct ljmd_handle ljmd_t;

/* Parameters captured by the reference's closures (MD:16-31). */
typedef struct ljmd_params {
    int64_t N;          /* particles                              MD:16          */
    float   box;        /* fp32 box edge = sqrt(N/rho)            MD:30          */
    float   sigma;      /* MD:26 (1.0 in the reference)                           */
    float   epsilon;    /* MD:27 (1.0 in the reference)                           */
    float   rc;         /* cutoff radius; INFINITY (or <=0) = none = reference    */
    float   dt;         /* time step                              MD:19          */
    float   skin;       /* cell-list skin (ignored by all-pairs); <=0 -> 0.3*sigma */
    int32_t path;       /* LJMD_PATH_*                                            */
    int32_t device;     /* CUDA device ordinal                                    */
    void*   stream;     /* cudaStream_t (NULL = legacy default stream)            */
} ljmd_params;

int         ljmd_abi_version(void);
const char* ljmd_last_error(void);

/* Positions handed to ljmd_energy / ljmd_forces / ljmd_run / ljmd_neighbor_count may lie anywhere:
 * coordinates outside the closed interval [0, box] are wrapped with jnp.mod semantics (MD:72) when
 * they are loaded (the reference's closures are periodic in R, MD:46-48), coordinates inside it
 * - everything a previous step can produce - are used bit for bit.  ljmd_gr_hist and
 * ljmd_cell_assign expect positions in [0, box] (what production_fn returns).                    */

/* closure capture of N, box_size, sigma, epsilon, dt (MD:16-31).  All scratch
 * (partial sums, cell arrays, ping-pong state) is allocated here, never per call. */
int  ljmd_create(ljmd_t** out, const ljmd_params* p);
void ljmd_destroy(ljmd_t* h);

/* total_energy_fn(R) -> scalar                                   MD:50-62
 * pe_dev: device float[1].                                                        */
int ljmd_energy(ljmd_t* h, const float* R, float* pe_dev);

/* force_fn(R) -> (N,2)                                           MD:64
 * F: device (N,2).  pe_dev may be NULL.                                           */
int ljmd_forces(ljmd_t* h, const float* R, float* F, float* pe_dev);

/* verlet_step (nsteps=1) MD:66-75, equilibrate_fn MD:77-83, production_fn MD:85-106.
 *   sample_every > 0 and traj != NULL: after step i (0-based), if i % sample_every == 0
 *     and i / sample_every < S (S = nsteps / sample_every) the new positions are stored in
 *     traj[i / sample_every]  — exactly MD:88-100, including the silently dropped
 *     out-of-range sample.  traj is (S,N,2) float32 and is fully overwritten
 *     (rows never sampled are zero, MD:89).
 *   energy_every > 0 and ke_pe != NULL: after step i, if i % energy_every == 0,
 *     ke_pe[i / energy_every] = {KE, PE} of the post-step state
 *     (KE = 0.5*sum|V|^2, PE = total_energy_fn(R)); buffer is (ceil(nsteps/energy_every),2).
 *     On a step that also rescales (thermostat), KE is the value BEFORE the rescale (the one the
 *     rescale factor is computed from); the returned V is after it.
 *     Not in the reference (it never reports energies) — see DESIGN.md.
 *   thermostat_kT > 0: velocity-rescale thermostat, V *= sqrt(kT_target / (KE/N)) after every
 *     `thermostat_every`-th step.  Default off (<= 0) = the reference's pure NVE.
 * No host synchronisation inside; all nsteps are enqueued in one call (MD:82,103).  */
int ljmd_run(ljmd_t* h, const float* R_in, const float* V_in, float* R_out, float* V_out,
             int64_t nsteps, int64_t sample_every, float* traj,
             int64_t energy_every, float* ke_pe,
             float thermostat_kT, int64_t thermostat_every);

/* ---- pair virial and pressure (new; the reference has neither - see DESIGN.md) ---------- */
/* W(R) = sum over unordered pairs i<j with r^2 < rc^2 of r_ij . f_ij = sum 24 eps (2 (sigma/r)^12 - (sigma/r)^6),
 * with the minimum image, the fp32 pair set {r^2 < rc^2} and the 1/r^2 (MUFU.RCP) of the force that moves the
 * particles: per pair w = t * (1/r^2)^3 with t = c12 (1/r^2)^3 - c6 the force's own factor, accumulated where and
 * with the weight that PE is, and finished with PE's 1/2.  rc = none: all pairs, as the reference.  No tail and
 * no impulsive correction for the truncation at rc (PE has neither): W is the virial of exactly the forces the
 * integrator applies.  The pressure of the 2-D fluid (unit mass, k_B = 1) is P = (KE + W/2) / box^2.
 * Single-GPU handles only: multi-GPU handles return LJMD_E_UNSUPPORTED from both calls.
 *
 * ljmd_virial: W of R as one device float, like ljmd_energy.  w_dev: device float[1].                    */
int ljmd_virial(ljmd_t* h, const float* R, float* w_dev);

/* ljmd_run plus the virial trace: w[i / energy_every] = W of the post-step state on exactly the rows where
 * ke_pe is written (the KE of a thermostat step there is the value before the rescale, as for ke_pe).
 * w: device float[ceil(nsteps/energy_every)].  w == NULL: this is ljmd_run.  w != NULL without ke_pe and
 * energy_every > 0: LJMD_E_INVALID.  The trajectory, the final state and ke_pe are bit for bit those of
 * ljmd_run: W is summed on the energy steps only, by a separate instantiation of the step kernel.        */
int ljmd_run_virial(ljmd_t* h, const float* R_in, const float* V_in, float* R_out, float* V_out,
                    int64_t nsteps, int64_t sample_every, float* traj,
                    int64_t energy_every, float* ke_pe,
                    float thermostat_kT, int64_t thermostat_every, float* w);

/* calculate_g_r histogram stage (get_histogram, MD:117-124) for S snapshots:
 * counts[s*nbins + k] = number of unordered pairs (i<j) of snapshot s whose minimum-image
 * distance r satisfies edges[k] <= r < edges[k+1] (last bin right-closed, values outside
 * [edges[0], edges[nbins]] dropped — numpy/jnp.histogram semantics).  edges: device
 * float32[nbins+1], ascending (the caller passes linspace(0, r_max, nbins+1), MD:110);
 * counts: device int64 (S,nbins).  The normalisation (MD:111-115,126-128) is host-side
 * arithmetic on nbins numbers.                                                     */
int ljmd_gr_hist(ljmd_t* h, const float* R_hist, int64_t S, int32_t nbins,
                 const float* edges, int64_t* counts);

/* ljmd_gr_hist for callers that know on the host an upper bound r_max of the histogram range:
 * counts exactly the pairs ljmd_gr_hist counts that also have r <= r_max, so with r_max >= edges[nbins]
 * the result is ljmd_gr_hist's, bit for bit.  r_max: finite, > 0.  The library bins each snapshot into a
 * periodic cell grid of edge >= r_max (at most N cells) and visits only neighbouring cells when that grid
 * has >= 3 cells per side: O(S N rho pi r_max^2) work, which is what makes g(r) affordable for millions of
 * particles.  Otherwise it runs the all-pairs histogram of ljmd_gr_hist.  nbins in [1, 8192].  S == 0 does
 * nothing, and R_hist and counts may then be NULL.  Scratch for the grid is allocated on the first call
 * that uses it and kept until ljmd_destroy.                                                          */
int ljmd_gr_hist_rmax(ljmd_t* h, const float* R_hist, int64_t S, int32_t nbins,
                      const float* edges, float r_max, int64_t* counts);

/* ---- density modes and the static structure factor (new; the reference has no S(k) - see DESIGN.md) ---- */
/* Density modes rho_k(s) = sum_j exp(i 2pi (n_x x_j + n_y y_j) / box) of S snapshots for K integer wave vectors
 * n = (n_x, n_y), k = (2pi / box) n; the structure factor is S(k) = <|rho_k|^2> / N.
 * R_hist: device (S,N,2) float32, 8-byte aligned; nvec: device int32 (K,2), any integers, 8-byte aligned;
 * rho: device float64 (S,K,2) = (Re, Im), 16-byte aligned.
 *   - Fixed-point phase: each coordinate is converted once to the 32-bit phase word rint(x / box * 2^32) mod 2^32
 *     and the phase of a term is n_x q_x + n_y q_y in uint32 arithmetic, exact modulo one revolution.  Positions
 *     may lie anywhere: a coordinate outside [0, box] is taken periodically (x and x + box give the same bits).
 *   - Accuracy, for each of Re and Im: |rho_k - exact| <= N eps_term + N 16.5 2^-24 + (N/32 + 1024) N 2^-53 with
 *     eps_term = (|n_x| + |n_y|) pi 2^-32 + 1.074e-6 (phase words, fp32 angle, MUFU sin/cos; the second term is
 *     the fp32 sum over chunks of 32 particles; derivation in csrc/sk.cu and DESIGN.md 4.5), for |x| <= 1024 box.
 *   - NaN: a snapshot with a non-finite coordinate gets NaN in every rho_k of its row; other rows are unaffected.
 *   - Deterministic: the same bits on every run, and rho_k of a (snapshot, vector) does not depend on the other
 *     snapshots and vectors of the call (the particle split depends on N only).
 *   - Any handle works, the multi-GPU ones included; there is no communication: each rank computes on the
 *     snapshots it was given.  Two launches per batch; partial-sum scratch (<= 512 MiB, snapshots and vectors
 *     batched to fit) is allocated on the first call and kept until ljmd_destroy.
 * S < 0, K < 0 or a NULL array: LJMD_E_INVALID.  S == 0 or K == 0 does nothing, and the arrays may then be NULL. */
int ljmd_density_modes(ljmd_t* h, const float* R_hist, int64_t S, const int32_t* nvec, int64_t K, double* rho);

/* ---- bond-orientational order (new; the reference has neither - see DESIGN.md) ----------------------------- */
/* psi_m(i) = (1/n_i) sum_{j in nb(i)} exp(i m theta_ij) of every particle of S snapshots.
 * R_hist: device (S,N,2) float32 in [0, box] (what production_fn returns; other input does not fault), 8-byte
 * aligned; psi: device float64 (S,N,2) = (Re, Im) in ORIGINAL particle order, 16-byte aligned; nnb: device int32
 * (S,N) = n_i, or NULL.  m in [1, 12]; r_nb finite and > 0.
 *   - Neighbours: j != i with 0 < r_ij <= r_nb, r_ij exactly the fp32 minimum-image r that ljmd_gr_hist bins, so
 *     sum_i n_i = 2 x the ljmd_gr_hist_rmax count with edges [0, r_nb] when no two particles coincide.
 *   - Bond term: d = min_image(fl(x_j - x_i)) (from i to j) in double, u = d / |d| and w = u^m by m - 1 sequential
 *     complex products, every double operation rounded once.
 *   - Fixed point: each component of w is added as llrint(w 2^32) in int64 (exact, order-free), and
 *     psi_i = (double)sum 2^-32 / n_i; psi_i = 0 when n_i = 0.  |psi_i - exact| <= 2^-33 + (9m + 3) 2^-53 per
 *     component (derivation in csrc/bond.cu).
 *   - NaN: a particle with a non-finite coordinate gets psi = NaN and n = 0 and is no particle's neighbour; other
 *     particles are unaffected.
 *   - Deterministic: the same bits on every run, whatever the other snapshots of the call or the batching.
 *   - Through the periodic cell grid of ljmd_gr_hist_rmax (cells of edge >= r_nb, full 9-cell stencil; one cell,
 *     i.e. all pairs, when r_nb > box / 3).  Four launches per batch of snapshots; the scratch is the grid's (16 B
 *     per particle and snapshot, batches <= 512 MiB), allocated on first use and kept until ljmd_destroy.
 *   - Any handle works, the multi-GPU ones included; there is no communication: each rank computes on the
 *     snapshots it was given.
 * S < 0, m or r_nb out of range, a NULL or misaligned array: LJMD_E_INVALID.  S == 0 does nothing, and the
 * arrays may then be NULL.                                                                                       */
int ljmd_bond_order(ljmd_t* h, const float* R_hist, int64_t S, int32_t m, float r_nb,
                    double* psi, int32_t* nnb);

/* Pair correlation of psi: the histogram of ljmd_gr_hist_rmax (same edges, r_max, pairs and selection of the
 * cell grid or the all-pairs kernel) with a weight per pair.  For every pair it counts,
 * w_ij = Re psi_i Re psi_j + Im psi_i Im psi_j (two products and the sum, each rounded once); a pair with a
 * non-finite w_ij is skipped, any other adds 1 to counts[s*nbins + k] and llrint(w_ij 2^24) to wsum[s*nbins + k].
 * g_m(r) = wsum / (2^24 counts).  psi: device float64 (S,N,2) as ljmd_bond_order writes it (|psi| <= 1),
 * 16-byte aligned; counts, wsum: device int64 (S,nbins).  wsum is exact and order-free while every count is
 * below 2^38 (|llrint(w 2^24)| <= 2^24 + 1), which a count can only reach for N > 741,455.  The counts equal
 * ljmd_gr_hist_rmax's bit for bit when every psi is finite.  Scratch: the grid's (28 B per particle
 * and snapshot, batches <= 512 MiB).
 * Validation as ljmd_gr_hist_rmax, plus psi 16-byte aligned; S == 0 does nothing and accepts NULL arrays.        */
int ljmd_bond_corr(ljmd_t* h, const float* R_hist, const double* psi, int64_t S, int32_t nbins,
                   const float* edges, float r_max, int64_t* counts, int64_t* wsum);

/* ---- cluster analysis (new; the reference has none - see DESIGN.md) ------------------------------------------ */
/* Connected components ("clusters") of the link graph of every snapshot of S.
 * R_hist: device (S,N,2) float32 in [0, box], 8-byte aligned; mask: device uint8 (S,N) or NULL (every particle);
 * labels: device int32 (S,N), 4-byte aligned; sizes: device int32 (S,N), 4-byte aligned, or NULL.  r_link finite
 * and > 0.
 *   - Active: particle i of snapshot s is active when both its coordinates are finite and, if mask is given,
 *     mask[s*N + i] != 0.
 *   - Link: two distinct active particles i != j are linked when r_ij <= r_link, r_ij exactly the fp32
 *     minimum-image r that ljmd_gr_hist bins and ljmd_bond_order uses (min_image of fl(x_j - x_i), fl(dx^2),
 *     fl(dy^2), their rounded sum, rounded sqrt).  Coincident particles (r = 0) are linked.  With every particle
 *     active, the number of links is the ljmd_gr_hist_rmax count on edges [0, r_link].
 *   - Clusters: the connected components of that graph, periodic through the minimum image.
 *   - labels[s*N + i] (ORIGINAL particle order) = the smallest original index in i's cluster; -1 for an inactive
 *     particle; an isolated active particle is its own cluster.  sizes[s*N + k] = the number of particles labelled
 *     k: non-zero exactly at the cluster roots (labels[s*N + k] == k).
 *   - Deterministic: the canonical label does not depend on the order of any atomic operation, so the output is
 *     bit-identical on every run, whatever the other snapshots of the call, the batching or the handle.
 *   - Through the periodic cell grid of ljmd_gr_hist_rmax (cells of edge >= r_link, full 9-cell stencil; one cell,
 *     i.e. all pairs, when r_link > box / 3) and a lock-free union-find whose forest lives in labels (derivation in
 *     csrc/cluster.cu).  Six launches per batch of snapshots (three of the grid, init, hook, flatten).  The only
 *     scratch is the grid's (16 B per particle and snapshot, batches <= 512 MiB), allocated on first use and kept
 *     until ljmd_destroy.
 *   - Any handle works, the multi-GPU ones included; there is no communication: each rank computes on the
 *     snapshots it was given.
 * S < 0, r_link out of range, a NULL R_hist or labels, or a misaligned array: LJMD_E_INVALID.  S == 0 does nothing,
 * and the arrays may then be NULL.                                                                               */
int ljmd_clusters(ljmd_t* h, const float* R_hist, int64_t S, float r_link, const uint8_t* mask,
                  int32_t* labels, int32_t* sizes);

/* ---- Voronoi tessellation (new; the reference has none - see DESIGN.md 4.8) ---------------------------------- */
#define LJMD_VORONOI_MAX_VERTICES 64   /* polygon vertices a cell may need while it is built */
/* The Voronoi cell of every particle of S snapshots on the periodic box.
 * R_hist: device (S,N,2) float32 in [0, box], 8-byte aligned.  nvor: device int32 (S,N), required; area: device
 * float64 (S,N), 8-byte aligned, or NULL; adj: device int32 (S,N,adj_cap), or NULL; psi: device float64 (S,N,2),
 * 16-byte aligned, or NULL.  Integer arrays 4-byte aligned.  adj_cap in [1, 64] when adj is given; m in [1, 12]
 * when psi is given (read only then).
 *   - Sites: every particle with finite coordinates.  d_ij is the minimum-image difference of the fp32
 *     coordinates computed in double (x_j - x_i, then -box if > box/2, +box if < -box/2): exact unless a
 *     coordinate is a non-zero value below about 2^-29 box, and within 2^-53 box even then.  So d_ji = -d_ij.
 *   - Cell: V_i = { p : p.d_ij <= |d_ij|^2 / 2 for every site j with d_ij != 0 }, relative to site i, in double.
 *     Coincident sites (d_ij = 0) are ignored: two coincident particles get the same cell.
 *   - Complete: with R_i the largest distance from i to a vertex of V_i, the cell is exact on the torus once
 *     2 R_i < box / 2 (only minimum images can then cut it).  A particle whose cell does not meet that, or would
 *     need more than LJMD_VORONOI_MAX_VERTICES vertices while it is clipped, is INCOMPLETE; so is a particle with a
 *     non-finite coordinate, which is also nobody's neighbour.  Such a particle gets nvor = -1, area = psi = NaN
 *     and an adjacency row of -1; the other particles are unaffected, and ljmd_check stays clean.
 *   - Neighbours: j is a Voronoi neighbour of i when its half-plane gives V_i an edge of length l_ij > 2^-30 R_i
 *     (rounding at a degenerate vertex - four co-circular sites, e.g. the exact square lattice - leaves edges of
 *     ~1e-16 R_i, so the square lattice has 4 neighbours).  nvor[s*N + i] = their number.
 *   - area[s*N + i]: the shoelace area of the final polygon, in double.
 *   - adj[(s*N + i)*adj_cap + t]: the neighbours' original indices ordered by the angle of d_ij ascending in
 *     (-pi, pi], padded with -1; with nvor > adj_cap the first adj_cap of them (nvor still counts all).
 *   - psi[s*N + i]: sum_j (l_ij / L_i) (d_ij / |d_ij|)^m over the neighbours in adjacency order, L_i = sum_j l_ij;
 *     the power by m - 1 sequential complex products as ljmd_bond_order, each operation rounded once.
 *   - Deterministic: one thread per particle clips the cell by the sites in the order (double r^2, original index)
 *     ascending, so the output is bit-identical on every run, whatever the other snapshots of the call, the
 *     batching or the handle.
 *   - Through the periodic cell grid of ljmd_gr_hist_rmax (cells of about two mean spacings; the rings around a
 *     particle's cell grow until they cover its security radius 2 R_i; derivation in csrc/voronoi.cu).  Four
 *     launches per batch of snapshots; the scratch is the grid's (16 B per particle and snapshot, batches <= 512
 *     MiB), allocated on first use and kept until ljmd_destroy.
 *   - Any handle works, the multi-GPU ones included; there is no communication.
 * S < 0, a NULL R_hist or nvor, adj_cap or m out of range for a requested output, or a misaligned array:
 * LJMD_E_INVALID.  S == 0 does nothing, and the arrays may then be NULL.                                         */
int ljmd_voronoi(ljmd_t* h, const float* R_hist, int64_t S, int32_t* nvor, double* area,
                 int32_t* adj, int32_t adj_cap, int32_t m, double* psi);

/* ---- the other dense pairwise kernels of the reference repo (SURVEY.md 8f) -------- */
/* All-pairs acceleration with the pair law as a functor: gravity r^-3 in an open plane.
 *   LJMD_LAW_GRAVITY_NBODY  pairwise_forces(positions, masses) of nbody_bh_merger_sim (NBODY:54-67):
 *       a_i = sum_{j != i} where(r >= 1e-6, G m_j / r^3, 0) (pos_j - pos_i), summed in j order
 *   LJMD_LAW_GRAVITY_EM3    the gravity term of acceleration() of three_particles_em_nonuni (EM3:25-38):
 *       a_i = sum_j G m_j (pos_j - pos_i) max(r^2 + [i == j], 1e-12)^(-3/2)
 * pos, acc: device (n,2) float32; mass: device float32[n]; enqueued on `stream` (cudaStream_t, may be
 * NULL), no handle needed.  fp32 with every operation rounded once, as in the reference.            */
#define LJMD_LAW_GRAVITY_NBODY 0
#define LJMD_LAW_GRAVITY_EM3   1
int ljmd_pair_accel(int32_t law, const float* pos, const float* mass, int64_t n, float G, float* acc,
                    void* stream);

/* ---- cell-list introspection (for the bit-exact CPU recount, north_star) -------- */
/* geometry chosen at create: the box is cut into `nrows` rows of height >= rc+skin and each row
 * into `nbins_x` bins of width >= (rc+skin)/kbins; cell id = row * nbins_x + bin with
 * row = min((int)(y * inv_row_height), nrows-1), bin = min((int)(x * inv_bin_width), nbins_x-1)
 * (one fp32 multiply, truncation).  A particle's candidates are bins [bin-kbins, bin+kbins] of
 * rows row-1, row, row+1 (periodic).                                                      */
int ljmd_cell_geometry(ljmd_t* h, int32_t* nrows, int32_t* nbins_x, int32_t* kbins,
                       float* inv_row_height, float* inv_bin_width);
/* bins R, returns per-particle cell id (device int32[N]) and per-cell counts
 * (device int32[nrows*nbins_x]).  Either pointer may be NULL.                            */
int ljmd_cell_assign(ljmd_t* h, const float* R, int32_t* cell_id, int32_t* cell_count);
/* per-particle number of neighbours with minimum-image r^2 < radius^2 (j != i), found
 * through the cell list.  nbr_count: device int32[N] in ORIGINAL particle order.     */
int ljmd_neighbor_count(ljmd_t* h, const float* R, float radius, int32_t* nbr_count);
/* number of cell-list rebuilds performed by the last ljmd_run (host value; syncs).   */
int ljmd_last_rebuilds(ljmd_t* h, int64_t* rebuilds);

/* ---- multi-GPU (new; the reference is single-device) ---------------------------- */
/* One handle per rank/device.  nccl_unique_id: the 128 bytes of an ncclUniqueId made
 * by rank 0 and broadcast by the caller (e.g. over torch.distributed/gloo).
 * Atom decomposition for all-pairs (position all-gather each step, plus a reduce-scatter
 * of partial forces when the Newton's-third-law tiles are dealt to the ranks), row-slab
 * decomposition with halo-row exchange for the cell list (all as in-kernel NVLink peer
 * stores); one all-reduce for energies.  Cell list on several GPUs: no thermostat, outputs
 * must not alias inputs, neighbor_count is single-GPU.
 * R/V arguments of ljmd_run etc. are then the FULL (N,2) arrays on every rank
 * (replicated in, replicated out) so the Python closures keep their signatures.     */
int ljmd_get_unique_id(void* id128);
int ljmd_create_dist(ljmd_t** out, const ljmd_params* p, const void* nccl_unique_id,
                     int32_t rank, int32_t nranks);

/* Block-distributed state for multi-GPU handles (the replicated convention above makes every rank
 * move the whole (N,2) arrays through PCIe and NVLink on every call): rank p passes and receives only
 * the particles of its INDEX block [p N/P, (p+1) N/P) - pointers to (N/P,2) device arrays; N must be
 * divisible by P.  Same physics as ljmd_run without trajectory sampling and thermostat.  Inside, the
 * blocks are all-gathered once (NCCL over NVLink) and every owner stores the final state of its
 * particles straight into the staging block of the rank that holds their index (in-kernel peer stores
 * on the cell path).  With one rank this is ljmd_run.                                              */
int ljmd_run_blocked(ljmd_t* h, const float* R_blk, const float* V_blk, float* R_blk_out, float* V_blk_out,
                     int64_t nsteps, int64_t energy_every, float* ke_pe);

/* ---- run status -------------------------------------------------------------------- */
/* The calls above only ENQUEUE work (JAX-style async dispatch), so conditions that a persistent
 * kernel detects on the device cannot come back through their return value: a Verlet list or a
 * slab that overflowed its buffers (LJMD_E_OVERFLOW: too dense for rc + skin, or too uneven over
 * the GPUs), a grid barrier or a cross-GPU wait that timed out (LJMD_E_TIMEOUT).  ljmd_check blocks
 * until everything enqueued on the handle's stream has finished and returns 0, a cudaError_t, or
 * one of those codes for the most recent call (the flags are cleared when a call starts).  The
 * outputs of a call that failed the check are invalid.  This is what block_until_ready (MD:145,
 * 152,163) maps to in the host wrapper.  Spin waits give up after LJMD_SPIN_TIMEOUT_S seconds
 * (environment, default 4; 0 = never: for cuda-gdb / compute-sanitizer sessions).              */
int ljmd_check(ljmd_t* h);

/* ---- measurement helpers --------------------------------------------------------- */
/* device time (ms) of the last ljmd_run's step loop, measured with CUDA events on the
 * handle's stream (blocks until that run has finished; also performs ljmd_check).   */
int ljmd_last_run_ms(ljmd_t* h, float* ms);
/* all-pairs evaluation mode chosen at create: 1 / 2 = every ORDERED pair is evaluated (one / two
 * i-particles per thread), 3 = Newton's-third-law tiles: every UNORDERED pair is evaluated once and
 * applied to both particles (atomic-free; N >= 2048, slabs of >= 2048 particles per GPU), 4 = ordered pairs inside ONE
 * thread-block cluster with the state resident in distributed shared memory (single GPU, N <= 640).
 * 0 on the cell-list path.                                                                        */
int ljmd_allpairs_mode(ljmd_t* h, int32_t* mode);
/* number of kernel launches issued by this handle since creation                    */
int ljmd_launch_count(ljmd_t* h, int64_t* launches);
/* FP32 issue-rate micro-benchmarks (FFMA / FFMA2 dependent chains): returns achieved
 * TFLOP/s so bench.py can state the measured CUDA-core ceiling next to the nominal. */
int ljmd_fp32_peak_probe(int32_t device, int32_t packed, float* tflops);

#ifdef __cplusplus
}
#endif
#endif /* LJMD_H_ */
