// cells.cu — sorted strip-cell / byte-Verlet-list path for large N (BASELINE configs 4-5).
//
// Not in the reference (it only has the dense O(N^2) form, MD:51): the pair arithmetic is the
// same as the all-pairs path (subtract, exact min-image, unfused r2, r2 < rc^2), so on identical
// fp32 inputs it evaluates exactly the pair set of the all-pairs+cutoff oracle.
//
// Geometry.  The box is cut into `nrows` horizontal rows of height >= rc + skin and every row into
// `nbx` narrow bins of width >= (rc + skin) / K  (K = 4).  Cells (row, bin) are numbered row-major
// and the particle state is kept SORTED by cell ("slots").  Everything within rc + skin of a particle
// of cell (r, b) lies in bins [b-K, b+K] of rows r-1, r, r+1, i.e. in THREE CONTIGUOUS SLOT RANGES
// (42 candidates at rho 0.8, against 57 for square 3x3 cells).
//
// Neighbour list.  A unit = 32 consecutive slots = one warp.  All neighbours of a unit lie in three
// contiguous slot WINDOWS (<= 84 slots each), which the per-step pass stages in shared memory; a
// particle's Verlet list is ONE BYTE per neighbour - its index in the staged windows - built at a
// rebuild from the same fp32 r2 as the force loop.  The per-step pass walks the bytes four per word: two
// neighbours of one particle fill the two lanes of the packed FP32x2 instructions.  Units that straddle
// a row or touch the periodic edge keep (first slot, 32-bit mask) entries and gather from global memory.
//
// Data layout in HBM (all in slot order, permuted only at a rebuild):
//   R[2]     float2  positions, ping-pong by step (the buffer being read is never written in a step)
//   V[2]     float2  velocities (buffers swap at a rebuild)
//   orig[2]  int32   original particle index of each slot
//   Rb       float2  positions at the last rebuild (max-displacement test against skin/2)
//   meta     uint32  number of list entries | edge flag << 8 (particle needs the minimum image)
//   ent      uint2   list entries, ELL layout ent[k * Nalloc + i] = (first slot, mask)
//   wplan    int4    per warp of 32 slots ("unit"): the three contiguous slot windows that hold every
//                    neighbour of the warp's particles (even start, even length: 16-byte granules)
//                    and the list length.  The per-step pass fetches them with ONE bulk copy each
//                    (cp.async.bulk -> UBLKCP, completion on an mbarrier), so the gathers of the pair
//                    loop are LDS, not scattered global loads.
//   nb4      uint32  for such a warp the list is stored EXPANDED: one byte per neighbour = its index
//                    in the staged windows (<= 252 slots), four per word, [unit][word][lane] so that a
//                    unit's words are ONE contiguous block (one more bulk copy), padded with a
//                    sentinel index to the warp's longest list: decode is a byte extract, there is no
//                    per-lane trip count.  (first slot, mask) entries remain for the other warps.
//   cell_start int32 prefix-sum cell index over nrows*nbx cells (+1)
//
// One PERSISTENT cooperative kernel runs a whole ljmd_run(): per step ONE pass over the state
// (thread = particle: list forces + velocity-Verlet + energies + displacement test; state read once,
// written once) and one grid barrier.  The rebuild (bin + histogram with rank capture -> row-wise
// prefix sum -> scatter -> deterministic in-cell order by original index + gather -> list build)
// runs inside the same kernel under a grid-uniform condition: no host round trip (MD:82,103).
#include "ljmd_device.cuh"

#include <algorithm>
#include <cstdio>

namespace ljmd {

namespace {

#ifndef CL_B5_
#define CL_B5_ 3
#endif
constexpr int CL_B5 = CL_B5_;     // slots per thread per trip of the rebuild gather (B5)
#ifndef CL_THREADS_
#define CL_THREADS_ 512
#endif
constexpr int CL_THREADS   = CL_THREADS_;
constexpr int CL_K         = 4;     // bins per (rc + skin)
constexpr int CL_E         = 8;     // list entries per particle (3 when every range fits 32 slots)
constexpr int CL_WIN       = 84;    // staged window capacity per stencil row and warp (slots):
                                    // 3 * CL_WIN = 252 slots fit a one-byte neighbour index
constexpr int CL_WSLOTS    = 256;   // a warp's staging buffer: three windows + 4 sentinel slots
constexpr int CL_DUMMY     = 255;   // byte index of a sentinel slot (pads the byte lists)
constexpr int CL_NW        = 24;    // byte-list words per particle (96 neighbours)
constexpr int CL_NWS       = 10;    // list words per lane that are staged in shared memory (40 neighbours;
                                    // longer lists read their tail from global memory)
constexpr int CL_BROW      = 4 * CL_NW + 4;   // a lane's byte row while a list is built (17 words:
                                              // rows of different lanes start in different banks)
// per-warp shared memory: two window buffers and two word buffers (the per-step pass double-buffers
// them with bulk copies, cp.async.bulk + mbarrier); the list build uses window buffer 0 and lays its
// byte rows over the rest
constexpr int CL_WINBYTES  = CL_WSLOTS * 8;                 // 2048
constexpr int CL_SWBYTES   = CL_NWS * 32 * 4;               // 1280
constexpr int CL_WARP_SMEM = 2 * CL_WINBYTES + 2 * CL_SWBYTES;   // bytes per warp (6656)
#ifndef CL_UNROLL
#define CL_UNROLL 2
#endif
// how a unit's windows and list words reach shared memory: 0 = bulk copies (cp.async.bulk / UBLKCP issued by
// four lanes, completion on an mbarrier), 1 = per-lane 16-byte cp.async (LDGSTS.128, commit / wait groups)
#ifndef CL_COPY
#define CL_COPY 0
#endif
#ifndef CL_DEPTH3
#define CL_DEPTH3 0     // 1 = a warp holds three units in flight (the schedule before the two-unit pipeline)
#endif

constexpr int CL_WORD_UNROLL = CL_UNROLL;                   // list words per trip of the pair loop
constexpr int CL_UNITWORDS = CL_NW * 32;                    // list words of one 32-slot unit in nb4
static_assert(CL_WINBYTES + 32 * CL_BROW <= CL_WARP_SMEM, "byte rows must fit behind window buffer 0");
static_assert(CL_WARP_SMEM % 16 == 0 && CL_WIN % 2 == 0, "bulk copies need 16-byte granularity");
constexpr int CL_WARPS     = CL_THREADS / 32;
constexpr int CL_QMAX      = 1024;  // unit queues: one per SM in use (indexed by a compact SM number)
constexpr int CL_ORDER_MAX = 64;    // cells denser than this keep arrival order (see B5)

enum { ST_PR = 0, ST_PV = 1, ST_REBUILDS = 2, ST_ERR = 3, ST_FLAG = 4, ST_NHELD = 5, ST_OWN_S = 6,
       ST_OWN_E = 7, ST_LOADCNT = 8, ST_XEPOCH = 9, ST_LMOVED = 10, ST_ABORT = 11, ST_WORDS = 16 };
// ST_ERR: conditions that void the RESULT (the kernel itself keeps running in lockstep);
// ST_ABORT: a spin wait gave up (1 = grid barrier, 2 = peer GPU) - later waits fall through
enum { CERR_LIST_OVERFLOW = 2, CERR_CAPACITY = 8, CERR_DEBUG = 16 };
// -DLJMD_DEBUG_CHECKS: in-kernel bounds assertions on every window, list index and bulk copy (the stand-in for
// compute-sanitizer memcheck, which is closed on the measurement pool); a violation raises CERR_DEBUG
#ifdef LJMD_DEBUG_CHECKS
#define CL_ASSERT(cond) do { if (!(cond)) atomicOr(a.state + ST_ERR, CERR_DEBUG); } while (0)
#else
#define CL_ASSERT(cond) do { } while (0)
#endif
// mailbox words a neighbour writes (slab decomposition)
enum { MB_HI_START = 0, MB_WORDS = 8 };

struct CellsArgs {
    PairConsts pc;
    int   N, Nalloc, G, nchunks;    // global particle count; local slot capacity; grid; chunk capacity
    int   nrows, nbx, ncells;       // global rows; bins per row; LOCAL cells = nlr * nbx
    // slab decomposition over P GPUs (P == 1: one slab = the whole box, rows wrap around):
    // this rank owns global rows [g0, g0 + nloc) = local rows [own_lo, own_lo + nloc) and, for P > 1,
    // holds one halo row on each side (local rows 0 and nlr - 1)
    int   P, me, g0, nloc, nlr, own_lo;    // me = this rank
    float2*   peerR[2][LJMD_MAX_RANKS];      // every rank's position / velocity / index buffers,
    float2*   peerV[2][LJMD_MAX_RANKS];      // cell counters, arrival words and mailbox (IPC-mapped)
    int*      peerO[2][LJMD_MAX_RANKS];
    int*      peer_cc[LJMD_MAX_RANKS];
    unsigned* peer_flags[LJMD_MAX_RANKS];
    int*      peer_mail[LJMD_MAX_RANKS];
    int*      mail;                 // = peer_mail[rank]
    int       nloc_of[LJMD_MAX_RANKS];       // owned rows of every rank
    float inv_hy, inv_wx, rlist2, half_skin2, dt;
    float static_frac;              // share of a warp's units that is dealt statically (the rest: dynamic queues)
    float2* R[2];
    float2* V[2];
    int*    orig[2];
    float2* Rb;
    float2* Fs;                     // forces held across the thermostat barrier
    int *key, *rank, *tmpk, *tmpo, *tmpc, *cell_count, *cell_start, *row_tot;
    unsigned* meta;
    uint2*    ent;
    unsigned* nb4;                  // byte lists of staged units, nb4[(unit * CL_NW + w) * 32 + lane]
    int4*     wplan;                // per unit: (ws0, ws1, ws2, wn0 | wn1 << 8 | wn2 << 16 | nw << 24 | staged << 31)
    float  *pe_part, *ke_part;      // [2*nchunks] per-unit partials (by step parity); nchunks = unit capacity
    int*      sched;                // [2][CL_QMAX] unit counters (by step parity, per SM queue) | [CL_QMAX] SM id ->
                                    // queue table | queue count (see the kernel prologue)
    int*      state;                // ST_* words
    unsigned* bar;
    const float2* R_in;
    const float2* V_in;
    long long s_begin, s_end;
    long long spin_limit;           // clocks a spin wait may last (0 = unlimited)
    RunCtl rc;
    float2 *R_out, *V_out, *F_out;
    // block-distributed output (ljmd_run_blocked): the owner of a particle stores its final state straight
    // into the staging block of the rank that owns its ORIGINAL index (NVLink peer store)
    int     blk;                    // particles per index block (0 = replicated output)
    float2* peer_stageR[LJMD_MAX_RANKS];
    float2* peer_stageV[LJMD_MAX_RANKS];
    float*  pe_out;
    int*    count_out;              // count mode: neighbour counts in original order
    int     mode;                   // 0 = run, 1 = build + count only
    long long* prof;                // optional [G][12] phase clocks (debug: LJMD_CELLS_PROF=1)
    float   count_r2;
    // virial kernel: per-unit partial virial like pe_part, and the output: W of R_in when nsteps == 0,
    // else one float per ke_pe row
    float*  vir_part;               // [2*nchunks]
    float*  vir_out;
};

// one fp32 multiply then truncation (x >= 0); the clamp handles x == box (MD:72 closed range)
__device__ __forceinline__ int strip_coord(float x, float inv, int n) {
    const int c = (int)(x * inv);
    return max(0, min(c, n - 1));
}

// local row of a y coordinate (may be >= nlr: not held by this rank)
__device__ __forceinline__ int local_row(const CellsArgs& a, float y) {
    const int gr = strip_coord(y, a.inv_hy, a.nrows);
    if (a.P == 1) return gr;
    int lr = gr - a.g0 + 1;
    lr += (lr < 0) ? a.nrows : 0;
    lr -= (lr >= a.nrows) ? a.nrows : 0;
    return lr;
}
__device__ __forceinline__ bool owned_row(const CellsArgs& a, int lr) {
    return lr >= a.own_lo && lr < a.own_lo + a.nloc;
}
// stencil neighbour of an owned local row: wraps around for one slab, plain offset with halo rows
__device__ __forceinline__ int nbr_row(const CellsArgs& a, int lr, int dr) {
    int rr = lr + dr;
    if (a.P == 1) {
        rr += (rr < 0) ? a.nrows : 0;
        rr -= (rr >= a.nrows) ? a.nrows : 0;
    }
    return rr;
}
// the particle needs the minimum image: first / last GLOBAL row, or within K bins of the x edges
__device__ __forceinline__ bool edge_cell(const CellsArgs& a, int lr, int b) {
    int gr = lr;
    if (a.P > 1) { gr = a.g0 - 1 + lr; gr += (gr < 0) ? a.nrows : 0; gr -= (gr >= a.nrows) ? a.nrows : 0; }
    return (gr == 0) | (gr == a.nrows - 1) | (b < CL_K) | (b > a.nbx - 1 - CL_K);
}

// block-wide exclusive scan of one int per thread; returns the exclusive prefix, *total = block sum
__device__ __forceinline__ int block_exscan(int v, int* swarp /* CL_THREADS/32 + 1 */, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) swarp[w] = inc;
    __syncthreads();
    if (w == 0) {
        int t = (lane < CL_THREADS / 32) ? swarp[lane] : 0;
        int ti = t;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int u = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= o) ti += u;
        }
        if (lane < CL_THREADS / 32) swarp[lane] = ti - t;   // exclusive warp offsets
        if (lane == 31) swarp[CL_THREADS / 32] = ti;
    }
    __syncthreads();
    *total = swarp[CL_THREADS / 32];
    return inc - v + swarp[w];
}

// sum of n floats in fixed order by the whole CTA, in double; result valid in every thread
__device__ __forceinline__ double block_sum_array(const float* p, int n, double* sdbl /* CL_THREADS/32 */) {
    double t = 0.0;
    for (int k = threadIdx.x; k < n; k += CL_THREADS) t += (double)__ldcg(p + k);
    t = warp_sum(t);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sdbl[threadIdx.x >> 5] = t;
    __syncthreads();
    double tot = 0.0;
#pragma unroll
    for (int k = 0; k < CL_THREADS / 32; ++k) tot += sdbl[k];
    return tot;
}

struct Ctx {
    unsigned epoch;     // grid-barrier epoch
    unsigned xepoch;    // cross-GPU sync epoch
    int pr, pv;
    int nheld;          // local slots in use (owned rows + halo rows)
    int own_s, own_e;   // slot range of the owned rows
    long long* pt;      // shared-memory phase clocks (thread 0), or nullptr
    int q, nq;          // this SM's unit queue and the number of queues
};

// ---- cross-GPU synchronisation (slab decomposition) -----------------------------------------------
// All ranks run the same steps in lockstep.  sync: every rank stamps an arrival word (epoch, plus one
// payload bit) into every peer over NVLink after a system-scope fence, then every CTA waits until
// all P local words carry the epoch.  Returns the OR of the payload bits.  Call after a grid barrier
// (all of this rank's peer stores are then ordered before the stamp).
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ bool peer_sync(const CellsArgs& a, Ctx& ctx, bool payload) {
    const unsigned xe = ++ctx.xepoch;
    const int slot = (int)(xe & 1u) * a.P;          // words alternate by epoch: a peer that is already one
                                                    // sync ahead does not overwrite a word still being read
    if (blockIdx.x == 0 && threadIdx.x < a.P && (int)threadIdx.x != a.me) {
        __threadfence_system();
        volatile unsigned* f = a.peer_flags[threadIdx.x] + slot + a.me;
        *f = (xe << 1) | (payload ? 1u : 0u);
    }
    __shared__ int s_any;
    if (threadIdx.x < 32) {
        // lane q polls the word of rank q: all P words are in flight together, so a sync whose words
        // have already landed costs ONE round trip to L2 (it used to be P - 1 dependent ones)
        const int q = (int)threadIdx.x;
        const bool mine_too = (q < a.P) && (q != a.me);
        const unsigned* word = a.peer_flags[a.me] + slot + (mine_too ? q : 0);
        unsigned w = (q == a.me && payload) ? 1u : 0u;
        const long long t0 = clock64();
        for (;;) {
            bool done = true;
            if (mine_too) { w = ld_acquire_sys(word); done = (w >> 1) == xe; }
            if (__all_sync(0xffffffffu, done)) break;
            const bool giveup = (a.spin_limit > 0 && clock64() - t0 > 2 * a.spin_limit) || __ldcg(a.state + ST_ABORT) != 0;
            if (__any_sync(0xffffffffu, giveup)) {           // (warp-uniform exit)
                if (q == 0) atomicExch(a.state + ST_ABORT, 2);
                w = 0u;
                break;
            }
        }
        const bool any = __any_sync(0xffffffffu, (q < a.P) && (w & 1u) != 0u);
        if (q == 0) s_any = any ? 1 : 0;
    }
    __syncthreads();
    const bool r = s_any != 0;
    __syncthreads();
    // the peers' halo stores are read by bulk copies (async proxy) from here on
    asm volatile("fence.proxy.async.global;" ::: "memory");
    return r;
}

#define CL_PROF(k)                                                          \
    do {                                                                    \
        if (ctx.pt && threadIdx.x == 0) {                                   \
            long long _t = clock64();                                       \
            ctx.pt[k] += _t - ctx.pt[11];                                   \
            ctx.pt[11] = _t;                                                \
        }                                                                   \
    } while (0)

// (the proxy fences order this thread's global stores against the bulk copies other CTAs issue after
//  the barrier, see fence_proxy_async)
#define CL_BARRIER()                                                                                  \
    do {                                                                                              \
        asm volatile("fence.proxy.async.global;" ::: "memory");                                              \
        grid_barrier(a.bar, (++ctx.epoch) * (unsigned)a.G, a.state + ST_ABORT, a.spin_limit);         \
        asm volatile("fence.proxy.async.global;" ::: "memory");                                              \
    } while (0)

// ---- rebuild: counting sort by cell, deterministic in-cell order, bitmask Verlet list --------------
// lim2: list radius squared (rc + skin for a run, the caller's radius in count mode)
__device__ void cells_rebuild(const CellsArgs& a, Ctx& ctx, int* sscan, float2* win /* this warp's CL_WSLOTS slots */,
                              unsigned char* sbytes /* this warp's 32 byte rows */, float lim2) {
    const int tid = threadIdx.x, gtid = blockIdx.x * CL_THREADS + tid, gsz = a.G * CL_THREADS;
    const float2* __restrict__ Rc = a.R[ctx.pr];
    const int* __restrict__ orig_old = a.orig[ctx.pv];
    const int nheld = ctx.nheld;
    const int lo_cell = a.own_lo * a.nbx, hi_cell = (a.own_lo + a.nloc) * a.nbx;   // owned local cells
    CL_PROF(0);
    // B1: cell of every held particle + histogram; the atomic's return value is the particle's
    //     (arbitrary) arrival rank inside its cell, so the scatter needs no second atomic pass.  Four
    //     particles per thread keep four atomics in flight.
    //     Slabs: a rank re-bins the particles of its owned rows AND of its two halo rows (whose
    //     positions and velocities the owners push every step) and keeps those that are now in an
    //     owned row.  A particle moves less than one row between rebuilds, so whoever owns it next
    //     already holds it: migration needs no message.
    //     (cell_count is all-zero on entry: cleared at create and again by B3 of every rebuild.)
    for (int k0 = gtid; k0 < nheld; k0 += 4 * gsz) {
        int c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * gsz;
            c[u] = -1;
            if (k < nheld) {
                const float2 r = Rc[k];
                const int lr = local_row(a, r.y);
                if (owned_row(a, lr)) c[u] = lr * a.nbx + strip_coord(r.x, a.inv_wx, a.nbx);
            }
        }
        int rk[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) rk[u] = (c[u] >= 0) ? atomicAdd(&a.cell_count[c[u]], 1) : 0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + u * gsz;
            if (k < nheld) { a.key[k] = c[u]; a.rank[k] = rk[u]; }
        }
    }
    CL_BARRIER();
    if (a.P > 1) {
        // H1: the bin populations of my first / last owned row are the populations of the lower
        //     neighbour's upper halo row / the upper neighbour's lower halo row
        const int dn = (a.me + a.P - 1) % a.P, up = (a.me + 1) % a.P;
        int* cc_dn = a.peer_cc[dn] + (a.nloc_of[dn] + 1) * a.nbx;      // its local row nlr-1
        int* cc_up = a.peer_cc[up];                                      // its local row 0
        const int* mine_first = a.cell_count + lo_cell;
        const int* mine_last  = a.cell_count + hi_cell - a.nbx;
        for (int b = gtid; b < a.nbx; b += gsz) { cc_dn[b] = mine_first[b]; cc_up[b] = mine_last[b]; }
        __threadfence_system();
        CL_BARRIER();
        (void)peer_sync(a, ctx, false);
    }
    CL_PROF(2);
    // B2: population of every local row
    for (int r = blockIdx.x; r < a.nlr; r += a.G) {
        int s = 0;
        for (int b = tid; b < a.nbx; b += CL_THREADS) s += __ldcg(&a.cell_count[r * a.nbx + b]);
        int tot;
        (void)block_exscan(s, sscan, &tot);
        if (tid == 0) a.row_tot[r] = tot;
    }
    CL_BARRIER();
    CL_PROF(3);
    // B3: row offsets + in-row exclusive scan -> cell_start; the row's counters are cleared for the
    //     next rebuild.
    for (int r = blockIdx.x; r < a.nlr; r += a.G) {
        int s = 0;
        for (int q = tid; q < r; q += CL_THREADS) s += a.row_tot[q];
        int carry;
        (void)block_exscan(s, sscan, &carry);
        // eight 512-bin pieces of the row are loaded before the first scan (one memory latency per 4096
        // bins instead of one per piece)
        for (int bb0 = 0; bb0 < a.nbx; bb0 += 8 * CL_THREADS) {
            int v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int b = bb0 + u * CL_THREADS + tid;
                v[u] = (b < a.nbx) ? __ldcg(&a.cell_count[r * a.nbx + b]) : 0;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (bb0 + u * CL_THREADS >= a.nbx) break;              // block-uniform
                const int b = bb0 + u * CL_THREADS + tid;
                int tot;
                const int ex = block_exscan(v[u], sscan, &tot);
                if (b < a.nbx) { a.cell_start[r * a.nbx + b] = carry + ex; a.cell_count[r * a.nbx + b] = 0; }
                carry += tot;
            }
        }
        if (r == a.nlr - 1 && tid == 0) {
            a.cell_start[a.ncells] = carry;
            if (carry > a.Nalloc) atomicOr(a.state + ST_ERR, CERR_CAPACITY);
        }
    }
    CL_BARRIER();
    CL_PROF(4);
    const int own_s = a.cell_start[lo_cell], own_e = a.cell_start[hi_cell], nheld_new = a.cell_start[a.ncells];
    if (a.P > 1 && gtid == 0) {
        // H2: tell the upper neighbour where my upper halo row starts (it fills that row)
        a.peer_mail[(a.me + 1) % a.P][MB_HI_START] = own_e;
        __threadfence_system();
    }
    // B4: scatter (source slot, original index, cell) into the cell's slot range, arrival order
    for (int k0 = gtid; k0 < nheld; k0 += 4 * gsz) {
        int c[4], rk[4], og[4], cs0[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {                       // stage 1: four independent streams
            const int k = k0 + u * gsz;
            c[u] = -1; rk[u] = 0; og[u] = 0;
            if (k < nheld) { c[u] = a.key[k]; rk[u] = a.rank[k]; og[u] = orig_old[k]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) cs0[u] = (c[u] >= 0) ? a.cell_start[c[u]] : 0;   // stage 2: four gathers
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (c[u] >= 0) {
                const int d = min(cs0[u] + rk[u], a.Nalloc - 1);
                a.tmpk[d] = k0 + u * gsz;
                a.tmpo[d] = og[u];
                a.tmpc[d] = c[u];
            }
        }
    }
    CL_BARRIER();
    CL_PROF(5);
    // B5: each new owned slot picks the member of its cell whose ORIGINAL index has the slot's rank,
    //     so the sorted order (cell, orig) is a pure function of the positions (bit-reproducible
    //     summation order downstream), then gathers that member's state (coalesced writes).
    //     (A bin holds ~1.6 particles at liquid density; a bin with more than CL_ORDER_MAX members
    //     keeps its arrival order: still correct, no longer run-to-run bit-reproducible.)
    {
        float2* Rn = a.R[ctx.pr ^ 1];
        const float2* Vo = a.V[ctx.pv];
        float2* Vn = a.V[ctx.pv ^ 1];
        int* on = a.orig[ctx.pv ^ 1];
        // CL_B5 slots per thread per trip: the chain slot -> cell -> cell range -> member -> state is four
        // dependent loads long; independent chains divide the exposed latency (1 -> 2 chains: -27 %)
        for (int d0 = own_s + gtid; d0 < own_e; d0 += CL_B5 * gsz) {
            int dd[CL_B5], c[CL_B5], b[CL_B5], n[CL_B5], msel[CL_B5], ksel[CL_B5], osel[CL_B5];
            bool ok[CL_B5];
            float2 r[CL_B5], v[CL_B5];
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) {
                dd[u] = d0 + u * gsz;
                ok[u] = dd[u] < own_e;
                c[u] = ok[u] ? a.tmpc[dd[u]] : 0;
            }
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) {
                b[u] = a.cell_start[c[u]];
                n[u] = a.cell_start[c[u] + 1] - b[u];
            }
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) {
                const int p = dd[u] - b[u];
                msel[u] = p;
                if (ok[u] && n[u] > 1 && n[u] <= CL_ORDER_MAX) {
                    for (int m = 0; m < n[u]; ++m) {
                        const int om = a.tmpo[b[u] + m];
                        int rk = 0;
                        for (int q = 0; q < n[u]; ++q) rk += (a.tmpo[b[u] + q] < om);
                        if (rk == p) { msel[u] = m; break; }
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) {
                ksel[u] = ok[u] ? a.tmpk[b[u] + msel[u]] : 0;
                osel[u] = ok[u] ? a.tmpo[b[u] + msel[u]] : 0;
            }
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) { r[u] = Rc[ksel[u]]; v[u] = Vo[ksel[u]]; }
#pragma unroll
            for (int u = 0; u < CL_B5; ++u) {
                if (ok[u]) {
                    Rn[dd[u]] = r[u];
                    a.Rb[dd[u]] = r[u];
                    Vn[dd[u]] = v[u];
                    on[dd[u]] = osel[u];
                }
            }
        }
    }
    ctx.pr ^= 1;
    ctx.pv ^= 1;
    ctx.nheld = nheld_new;
    ctx.own_s = own_s;
    ctx.own_e = own_e;
    if (blockIdx.x == 0 && tid == 0) a.state[ST_REBUILDS] += 1;
    CL_BARRIER();
    if (a.P > 1) {
        // H3: my first / last owned row, freshly sorted, becomes the neighbours' halo row: positions,
        //     velocities and original indices (a halo particle may become theirs at the next
        //     rebuild).  One sync before, so that every rank has
        //     published where its upper halo row starts and is done reading its old buffers.
        (void)peer_sync(a, ctx, false);
        const int dn = (a.me + a.P - 1) % a.P, up = (a.me + 1) % a.P;
        const int first_s = own_s, first_e = a.cell_start[lo_cell + a.nbx];
        const int last_s = a.cell_start[hi_cell - a.nbx], last_e = own_e;
        const int peer_hi_start = __ldcg(&a.mail[MB_HI_START]);   // mailed by the lower neighbour (H2)
        const float2* Rn = a.R[ctx.pr];
        const float2* Vn = a.V[ctx.pv];
        const int* on = a.orig[ctx.pv];
        // my first owned row -> lower neighbour's upper halo row (starts at the slot it mailed me)
        {
            float2* pR = a.peerR[ctx.pr][dn]; float2* pV = a.peerV[ctx.pv][dn]; int* pO = a.peerO[ctx.pv][dn];
            for (int i = first_s + gtid; i < first_e; i += gsz) {
                const int j = peer_hi_start + (i - first_s);
                pR[j] = Rn[i]; pV[j] = Vn[i]; pO[j] = on[i];
            }
        }
        // my last owned row -> upper neighbour's lower halo row (starts at its slot 0)
        {
            float2* pR = a.peerR[ctx.pr][up]; float2* pV = a.peerV[ctx.pv][up]; int* pO = a.peerO[ctx.pv][up];
            for (int i = last_s + gtid; i < last_e; i += gsz) {
                const int j = i - last_s;
                pR[j] = Rn[i]; pV[j] = Vn[i]; pO[j] = on[i];
            }
        }
        __threadfence_system();
        CL_BARRIER();
        (void)peer_sync(a, ctx, false);
    }
    CL_PROF(6);
    // B6: bitmask Verlet list.  For each stencil row the candidate bins [b-K, b+K] (periodic: up to
    //     two pieces) form contiguous slot ranges; every 32 slots of a range with at least one
    //     neighbour (min-image r2 < lim2, same unfused fp32 r2 as the force loop, j != i) become one
    //     (first slot, mask) entry.  Count mode only counts.
    //     A warp = 32 consecutive slots.  If they share a row and none needs a wrapped range, all their
    //     neighbours lie in three windows (bins [b_first-K, b_last+K] of rows r-1, r, r+1): the warp's
    //     plan records them and its entries are stored relative to the staged copy of the windows.
    {
        const float2* __restrict__ R = a.R[ctx.pr];
        const int* __restrict__ cs = a.cell_start;
        const PairConsts pc = a.pc;
        const int lane = tid & 31;
        // (position, cell) of the NEXT unit's slot are requested a whole unit ahead
        float2 rnext = make_float2(0.0f, 0.0f);
        int cnext = 0;
        {
            const int i = (ctx.own_s & ~31) + (gtid & ~31) + lane;
            if (i >= ctx.own_s && i < ctx.own_e) { rnext = R[i]; cnext = a.tmpc[i]; }
        }
        for (int i0 = (ctx.own_s & ~31) + (gtid & ~31); i0 < ctx.own_e; i0 += gsz) {
            const int i = i0 + lane;
            const bool live = (i >= ctx.own_s) & (i < ctx.own_e);
            const float2 ri = rnext;
            const int c = cnext;
            {
                const int in = i + gsz;
                rnext = make_float2(0.0f, 0.0f); cnext = 0;
                if (in >= ctx.own_s && in < ctx.own_e) { rnext = R[in]; cnext = a.tmpc[in]; }
            }
            const int r = c / a.nbx, b = c - r * a.nbx;           // local row, bin
            const bool edge = edge_cell(a, r, b);
            // warp plan
            const int l_first = max(ctx.own_s - i0, 0), l_last = min(31, ctx.own_e - 1 - i0);
            const int r_first = __shfl_sync(0xffffffffu, r, l_first), r_last = __shfl_sync(0xffffffffu, r, l_last);
            const int b_first = __shfl_sync(0xffffffffu, b, l_first), b_last = __shfl_sync(0xffffffffu, b, l_last);
            bool staged = (a.mode == 0) && (r_first == r_last) && !__any_sync(0xffffffffu, live && edge);
            int ws[3] = {0, 0, 0}, wn[3] = {0, 0, 0};
            int cs_s[3] = {0, 0, 0}, cs_e[3] = {0, 0, 0};           // this lane's three candidate ranges
            if (staged) {
                // the window bounds and the lane's own range bounds are independent loads: all twelve are
                // in flight together (they used to be four dependent round trips per unit)
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    ws[k] = cs[(r_first + k - 1) * a.nbx + b_first - CL_K];
                    wn[k] = cs[(r_first + k - 1) * a.nbx + b_last + CL_K + 1];
                    if (live) {
                        cs_s[k] = cs[(r + k - 1) * a.nbx + b - CL_K];
                        cs_e[k] = cs[(r + k - 1) * a.nbx + b + CL_K + 1];
                    }
                }
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    // 16-byte granules for the bulk copies of the per-step pass: even first slot, even
                    // length (the extra slots are real slots of the array; the list never names them)
                    const int e = wn[k];
                    ws[k] &= ~1;
                    wn[k] = (e - ws[k] + 1) & ~1;
                    staged = staged && (wn[k] <= CL_WIN);
                }
            }
            if (staged) {
                for (int k = 0; k < 3; ++k) {
                    CL_ASSERT(ws[k] >= 0 && wn[k] >= 0 && ws[k] + wn[k] <= a.Nalloc && (ws[k] & 1) == 0 && (wn[k] & 1) == 0);
                    CL_ASSERT(!live || (cs_s[k] >= ws[k] && cs_e[k] <= ws[k] + wn[k] && cs_s[k] <= cs_e[k]));
                }
                CL_ASSERT(!live || (i >= ws[1] && i < ws[1] + wn[1]));
            }
            int plan_w = staged ? (int)(0x80000000u | (unsigned)wn[0] | ((unsigned)wn[1] << 8) | ((unsigned)wn[2] << 16)) : 0;
            int n = 0, cnt = 0;
            if (staged) {
                // fast path: the warp's windows in shared memory (coalesced copy), every lane scans its
                // three ranges there, two candidates per step on the packed pipe; no minimum image
                // (identity this far from the box edge)
                __syncwarp();
#pragma unroll
                for (int j = 0; j < CL_WIN; j += 32) {
                    if (j + lane < wn[0]) win[j + lane] = R[ws[0] + j + lane];
                    if (j + lane < wn[1]) win[CL_WIN + j + lane] = R[ws[1] + j + lane];
                    if (j + lane < wn[2]) win[2 * CL_WIN + j + lane] = R[ws[2] + j + lane];
                }
                __syncwarp();
                // neighbour indices are appended branch-free to this lane's byte row in shared
                // memory (a rejected candidate is overwritten by the next one), then written out as
                // coalesced words
                unsigned char* myb = sbytes + lane * CL_BROW;
                int nn = 0;                                             // neighbours appended so far
                if (live) {
                    const float2 nri = make_float2(-ri.x, -ri.y);
#pragma unroll
                    for (int k = 0; k < 3; ++k) {
                        const int s = cs_s[k] - ws[k];
                        const int e = cs_e[k] - ws[k];
                        const float2* __restrict__ w = win + k * CL_WIN;
                        const int iself = (k == 1) ? i - ws[k] : -1;    // own slot (own row only)
#pragma unroll 2
                        for (int t = s; t < e; t += 2) {
                            // (slot t + 1 == e is read but never taken: it lies inside the staged buffer;
                            //  one clamp per pair: the byte row has four bytes of slack)
                            const float2 d0 = __fadd2_rn(w[t], nri);
                            const float2 d1 = __fadd2_rn(w[t + 1], nri);
                            const float2 q0 = __fmul2_rn(d0, d0), q1 = __fmul2_rn(d1, d1);
                            const float r20 = __fadd_rn(q0.x, q0.y), r21 = __fadd_rn(q1.x, q1.y);
                            const bool in0 = (r20 < lim2) & (t != iself);
                            const bool in1 = (r21 < lim2) & (t + 1 < e) & (t + 1 != iself);
                            unsigned char* dst = myb + min(nn, 4 * CL_NW);
                            const int a0 = in0 ? 1 : 0;
                            dst[0] = (unsigned char)(k * CL_WIN + t);
                            dst[a0] = (unsigned char)(k * CL_WIN + t + 1);
                            nn += a0 + (in1 ? 1 : 0);
                        }
                    }
                }
                // pad to the warp's longest list with the sentinel index: the per-step loop needs no
                // per-lane trip count
                const int nw = (nn + 3) >> 2;
                int nwmax = nw;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) nwmax = max(nwmax, __shfl_xor_sync(0xffffffffu, nwmax, o));
                nwmax = min(nwmax, CL_NW);
                if (live) {
                    for (int q = min(nn, 4 * CL_NW); q < 4 * nwmax; ++q) myb[q] = (unsigned char)CL_DUMMY;
                    if (nw > CL_NW) atomicOr(a.state + ST_ERR, CERR_LIST_OVERFLOW);
                    const unsigned* myw = reinterpret_cast<const unsigned*>(myb);
                    CL_ASSERT((size_t)(i0 >> 5) * CL_UNITWORDS + (size_t)(nwmax - 1) * 32 + lane < (size_t)a.Nalloc * CL_NW || nwmax == 0);
                    unsigned* dst = a.nb4 + (size_t)(i0 >> 5) * CL_UNITWORDS + lane;
                    for (int u = 0; u < nwmax; ++u) dst[u * 32] = myw[u];
                }
                plan_w |= nwmax << 24;
                n = 0;
            } else if (live) {
                const int lo = b - CL_K, hi = b + CL_K;
                for (int k = 0; k < 3; ++k) {
                    const int rr = nbr_row(a, r, k - 1);
                    const int* __restrict__ csr = cs + rr * a.nbx;
                    for (int piece = 0; piece < 3; ++piece) {
                        int bl, bh;
                        if (piece == 0)      { bl = max(lo, 0); bh = min(hi, a.nbx - 1); }
                        else if (piece == 1) { if (lo >= 0) continue; bl = lo + a.nbx; bh = a.nbx - 1; }
                        else                 { if (hi < a.nbx) continue; bl = 0; bh = hi - a.nbx; }
                        const int s = csr[bl], e = csr[bh + 1];
                        for (int c0 = s; c0 < e; c0 += 32) {
                            const int cnum = min(32, e - c0);
                            unsigned mask = 0u;
                            for (int t0 = 0; t0 < cnum; t0 += 4) {          // four position loads in flight
                                float2 rj[4];
#pragma unroll
                                for (int u = 0; u < 4; ++u) rj[u] = R[c0 + min(t0 + u, cnum - 1)];
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    const float dx = min_image(__fsub_rn(ri.x, rj[u].x), pc.box, pc.timg);
                                    const float dy = min_image(__fsub_rn(ri.y, rj[u].y), pc.box, pc.timg);
                                    const float r2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
                                    if (t0 + u < cnum && r2 < lim2 && c0 + t0 + u != i) mask |= 1u << (t0 + u);
                                }
                            }
                            if (mask) {
                                if (a.mode == 0 && n < CL_E) a.ent[(size_t)n * a.Nalloc + i] = make_uint2((unsigned)c0, mask);
                                ++n;
                                cnt += __popc(mask);
                            }
                        }
                    }
                }
            }
            if (lane == 0) a.wplan[i0 >> 5] = make_int4(ws[0], ws[1], ws[2], plan_w);
            if (!live) continue;
            if (a.mode == 0) {
                if (n > CL_E) atomicOr(a.state + ST_ERR, CERR_LIST_OVERFLOW);
                a.meta[i] = (unsigned)min(n, CL_E) | (edge ? 0x100u : 0u);
            } else {
                a.key[i] = cnt;
            }
        }
    }
    CL_BARRIER();
    CL_PROF(7);
}

// ---- per-step pass ----------------------------------------------------------------------------------
// Two neighbours j0, j1 of ONE particle.  Each displacement (dx, dy) is one packed FP32x2 value made
// directly from the loaded float2 (no register shuffling); from r2 on, the two NEIGHBOURS share the
// packed instructions.  d is formed as rj - ri (= -(ri - rj) exactly), so the accumulator holds -F
// bit for bit; r2 = fl(fl(dx*dx) + fl(dy*dy)) unfused => the pair set {r2 < rc2} is the oracle's.
// The cutoff is a select on the ALU pipe (FSETP + SEL); `two` masks the second neighbour when the
// entry had an odd number of neighbours left.  (Measured: folding the cutoff in as a 1.0f / 0.0f mask with
// one packed multiply saves an instruction but costs two FMA-pipe cycles: 166.4 vs 165.5 us/step.)
// VIR: also accumulate the pair virial t * ir6 (t = c12*ir6 - c6, the force's own factor) into vir2.
template <bool PE, bool EDGE, bool VIR>
__device__ __forceinline__ void eval_two(const PairConsts& pc, const PairConsts2& c2, float2 nri,
                                         float2 rj0, float2 rj1, bool two, float2& acc, float2& pe2,
                                         float2& vir2) {
    float2 d0 = __fadd2_rn(rj0, nri);
    float2 d1 = __fadd2_rn(rj1, nri);
    if (EDGE) {
        d0.x = min_image(d0.x, pc.box, pc.timg); d0.y = min_image(d0.y, pc.box, pc.timg);
        d1.x = min_image(d1.x, pc.box, pc.timg); d1.y = min_image(d1.y, pc.box, pc.timg);
    }
    const float2 q0 = __fmul2_rn(d0, d0), q1 = __fmul2_rn(d1, d1);
    const float r20 = __fadd_rn(q0.x, q0.y), r21 = __fadd_rn(q1.x, q1.y);
    float2 ir2 = make_float2(rcp_approx(r20), rcp_approx(r21));
    ir2.x = (r20 < pc.rc2) ? ir2.x : 0.0f;
    ir2.y = (two & (r21 < pc.rc2)) ? ir2.y : 0.0f;
    const float2 ir6 = __fmul2_rn(__fmul2_rn(ir2, ir2), ir2);
    const float2 t = __ffma2_rn(ir6, c2.c12, c2.nc6);
    const float2 f = __fmul2_rn(t, __fmul2_rn(ir6, ir2));
    acc = __ffma2_rn(d0, make_float2(f.x, f.x), acc);
    acc = __ffma2_rn(d1, make_float2(f.y, f.y), acc);
    if (PE) pe2 = __ffma2_rn(ir6, __ffma2_rn(ir6, c2.d12, c2.nd6), pe2);
    if (VIR) vir2 = __ffma2_rn(t, ir6, vir2);
}

// all neighbours of particle i: the entries are walked as ONE sequence of set bits (a lane that
// finishes an entry moves on to its next one at once), so a warp runs for the longest LIST, not for
// the sum of the longest entries.  Every stored entry has a non-empty mask.
// R = the array the entries index: the staged windows (shared memory) or the global positions
template <bool PE, bool EDGE, bool VIR>
__device__ __forceinline__ void list_force(const CellsArgs& a, const float2* R, int i, int n,
                                           float2 ri, float& Fx, float& Fy, float& pe, float& vir) {
    const PairConsts pc = a.pc;
    const PairConsts2 c2 = make_pair_consts2(pc);
    const uint2* __restrict__ ep = a.ent + i;
    const size_t stride = (size_t)a.Nalloc;
    // the first three entries (all of them, normally) are requested before the loop
    uint2 e0 = make_uint2(0u, 0u), e1 = e0, e2 = e0;
    if (n > 0) e0 = ep[0];
    if (n > 1) e1 = ep[stride];
    if (n > 2) e2 = ep[2 * stride];
    const float2 nri = make_float2(-ri.x, -ri.y);
    float2 acc = make_float2(0.0f, 0.0f), pe2 = acc, vir2 = acc;
    unsigned m = e0.y;
    const float2* base = R + e0.x;
    int k = 1;
    for (;;) {
        if (m == 0u) {
            if (k >= n) break;
            const uint2 e = (k == 1) ? e1 : ((k == 2) ? e2 : ep[(size_t)k * stride]);
            m = e.y;
            base = R + e.x;
            ++k;
        }
        const int b0 = 31 - __clz(m);
        m ^= 1u << b0;
        const bool two = (m != 0u);
        const int b1 = two ? 31 - __clz(m) : b0;
        m &= ~(1u << b1);
        eval_two<PE, EDGE, VIR>(pc, c2, nri, base[b0], base[b1], two, acc, pe2, vir2);
    }
    Fx = -acc.x;
    Fy = -acc.y;
    if (PE) pe = pe2.x + pe2.y;
    if (VIR) vir = vir2.x + vir2.y;
}

// ---- bulk copies (cp.async.bulk = UBLKCP, the 1-D TMA path) completing on an mbarrier ---------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void* src, unsigned bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// (generic-proxy writes - st.global of the integrate epilogue / the rebuild / peer GPUs - are ordered against
//  the async-proxy reads of later bulk copies by one fence.proxy.async.global on each side of every grid
//  barrier and after every cross-GPU sync: CL_BARRIER, peer_sync)

__device__ __forceinline__ void cp_async16(unsigned dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ float2 lds64(unsigned addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned lds32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

// staged units: the list is one byte per neighbour (index into the staged windows), four per word,
// padded with the sentinel index to the warp's longest list (nw words, warp-uniform).  `win` is the
// 32-bit shared-memory address of the staged windows: byte extract + scaled add + LDS.64 per neighbour.
template <bool PE, bool VIR>
__device__ __forceinline__ void word_eval(const PairConsts& pc, const PairConsts2& c2, unsigned win,
                                          unsigned word, float2 nri, float2& acc, float2& pe2, float2& vir2) {
    const float2 r0 = lds64(win + (__byte_perm(word, 0u, 0x4440u) << 3));
    const float2 r1 = lds64(win + (__byte_perm(word, 0u, 0x4441u) << 3));
    const float2 r2 = lds64(win + (__byte_perm(word, 0u, 0x4442u) << 3));
    const float2 r3 = lds64(win + (__byte_perm(word, 0u, 0x4443u) << 3));
    eval_two<PE, false, VIR>(pc, c2, nri, r0, r1, true, acc, pe2, vir2);
    eval_two<PE, false, VIR>(pc, c2, nri, r2, r3, true, acc, pe2, vir2);
}

// all listed neighbours of one particle of a staged unit: the first CL_NWS words of every lane arrived
// in shared memory with the windows, longer lists continue from global memory
template <bool PE, bool VIR>
__device__ __forceinline__ void bytes_force_staged(const CellsArgs& a, unsigned win, unsigned sw, int unit,
                                                   int nw, float2 ri, float& Fx, float& Fy, float& pe, float& vir) {
    const PairConsts pc = a.pc;
    const PairConsts2 c2 = make_pair_consts2(pc);
    const int lane = threadIdx.x & 31;
    const float2 nri = make_float2(-ri.x, -ri.y);
    float2 acc = make_float2(0.0f, 0.0f), pe2 = acc, vir2 = acc;
    const int nws = min(nw, CL_NWS);
    const unsigned swl = sw + lane * 4;
#pragma unroll CL_WORD_UNROLL
    for (int w = 0; w < nws; ++w) word_eval<PE, VIR>(pc, c2, win, lds32(swl + w * 128), nri, acc, pe2, vir2);
    if (nw > CL_NWS) {
        const unsigned* __restrict__ gw = a.nb4 + (size_t)unit * CL_UNITWORDS + lane;
        for (int w = CL_NWS; w < nw; ++w) word_eval<PE, VIR>(pc, c2, win, gw[w * 32], nri, acc, pe2, vir2);
    }
    Fx = -acc.x;
    Fy = -acc.y;
    if (PE) pe = pe2.x + pe2.y;
    if (VIR) vir = vir2.x + vir2.y;
}

// slow path of a buffer wait (try_wait itself sleeps in hardware; this is only reached after its time
// limit): kept out of line so that the unit loop carries one SYNCS + one branch
__device__ __noinline__ void mbar_wait_slow(const CellsArgs& a, unsigned bar, unsigned par) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, par)) {
        if (a.spin_limit > 0 && clock64() - t0 > a.spin_limit) { atomicExch(a.state + ST_ABORT, 3); break; }
    }
}

struct StepFlags {
    long long s;
    int  par;
    bool kick1, final, want_e, want_pe, want_ke, thermo, sample;
};

// per-warp pipeline state that outlives a step: shared-memory addresses and the mbarrier phases
struct WarpPipe {
    unsigned base;      // this warp's block: window buffer 0 | window buffer 1 | word buffer 0 | word buffer 1
    unsigned bar;       // two mbarriers (8 bytes each), one per buffer
    unsigned phase;     // bit b = parity the next wait on buffer b expects
};

// ---- one step's pass of one warp --------------------------------------------------------------------
// A unit = 32 consecutive slots = one warp.  Warp gw evaluates units u_lo + gw + k * W (interleaved:
// every warp sees units of ~28 different rows, which evens out density and edge effects; warps never
// wait for each other inside a step).  Software pipeline, driven by bulk copies: while unit k is
// evaluated out of one shared-memory buffer, FOUR bulk copies of unit k+1 are in flight into the other
// one (three neighbour windows + the unit's list words, issued by lanes 0-3, completion counted in
// bytes on the buffer's mbarrier) and the copy plan of unit k+2 is on its way to registers.
// PLAIN = an ordinary step of a run (second kick of the previous step, first kick + drift of this one;
// no sample, no energies, no thermostat, not the last step): the flag tests are compiled out.
// VIR (with PE): the per-unit virial partials ride along with the energy partials.
template <bool PE, bool PLAIN, bool VIR>
__device__ __forceinline__ void warp_pass(const CellsArgs& a, const Ctx& ctx, const StepFlags& fl,
                                          WarpPipe& wp, int& moved) {
    const RunCtl& rc = a.rc;
    const int lane = threadIdx.x & 31;
    const int W = a.G * CL_WARPS, gw = blockIdx.x * CL_WARPS + (threadIdx.x >> 5);
    const int u_lo = ctx.own_s >> 5, u_hi = (ctx.own_e + 31) >> 5;
    const float2* __restrict__ R = a.R[ctx.pr];
    float2* Rnext = a.R[ctx.pr ^ 1];
    float2* V = a.V[ctx.pv];
    const int* og = a.orig[ctx.pv];
    const bool kick1  = PLAIN ? true  : fl.kick1;
    const bool final  = PLAIN ? false : fl.final;
    const bool thermo = PLAIN ? false : fl.thermo;
    const bool sample = PLAIN ? false : fl.sample;
    const bool want_ke = PLAIN ? false : fl.want_ke;
    // halo pushes (slabs): slots of my first / last owned row and where they live in the neighbours
    const int dn = (a.me + a.P - 1) % a.P, up = (a.me + 1) % a.P;
    int first_e = 0, last_s = 0, peer_hi_start = 0;
    if (a.P > 1) {
        first_e = a.cell_start[(a.own_lo + 1) * a.nbx];
        last_s = a.cell_start[(a.own_lo + a.nloc - 1) * a.nbx];
        peer_hi_start = __ldcg(&a.mail[MB_HI_START]);
    }
    // the sentinel slots behind the staged windows (never within rc of anything; the list build uses
    // this memory for its byte rows, so they are rewritten every step)
    if (lane >= 28) {
        asm volatile("st.shared.v2.f32 [%0], {%1, %1};" ::"r"(wp.base + (3 * CL_WIN + (lane & 3)) * 8), "f"(1.0e9f) : "memory");
        asm volatile("st.shared.v2.f32 [%0], {%1, %1};" ::"r"(wp.base + CL_WINBYTES + (3 * CL_WIN + (lane & 3)) * 8), "f"(1.0e9f) : "memory");
    }
    // this warp's shared memory was last written through the generic proxy (the list build's byte rows):
    // order those writes before the bulk copies that now land in the same bytes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();

    // copy plan of a unit: (ws0, ws1, ws2, wn0 | wn1 << 8 | wn2 << 16 | nw << 24 | staged << 31).
    // Lane k < 3 copies window k, lane 3 the list words; lane 0 arms the mbarrier with the byte total.
    const char* Rbytes = reinterpret_cast<const char*>(R);
    const char* Lbytes = reinterpret_cast<const char*>(a.nb4);
    const unsigned my_dst = wp.base + (lane < 3 ? lane * (CL_WIN * 8) : 2 * CL_WINBYTES);   // + buf * stride
    const unsigned my_stride = lane < 3 ? CL_WINBYTES : CL_SWBYTES;
#if CL_COPY == 1
    const unsigned l16 = lane * 16;
    auto issue = [&](int u, const int4& p, int buf) {
        if (u < u_hi && p.w < 0) {
            const unsigned pw = (unsigned)p.w;
            const unsigned win = wp.base + buf * CL_WINBYTES + l16, sw = wp.base + 2 * CL_WINBYTES + buf * CL_SWBYTES + l16;
            const int wsk[3] = {p.x, p.y, p.z};
#pragma unroll
            for (int k = 0; k < 3; ++k) {           // a window is at most 84 slots = 672 bytes: chunks l16 and l16 + 512
                const unsigned bytes = ((pw >> (8 * k)) & 0xffu) * 8u;
                const char* src = Rbytes + (size_t)wsk[k] * 8 + l16;
                if (l16 < bytes) cp_async16(win + k * (CL_WIN * 8), src);
                if (l16 + 512 < bytes) cp_async16(win + k * (CL_WIN * 8) + 512, src + 512);
            }
            const unsigned wbytes = min((pw >> 24) & 0x7fu, (unsigned)CL_NWS) * 128u;
            const char* src = Lbytes + (size_t)u * (CL_UNITWORDS * 4) + l16;
#pragma unroll
            for (int c = 0; c < CL_SWBYTES; c += 512)
                if (l16 + c < wbytes) cp_async16(sw + c, src + c);
        }
        cp_async_commit();
    };
#else
    auto issue = [&](int u, const int4& p, int buf) {
        if (u < u_hi && p.w < 0) {
            const unsigned pw = (unsigned)p.w;
            const unsigned nws = min((pw >> 24) & 0x7fu, (unsigned)CL_NWS);
            const unsigned bar = wp.bar + buf * 8;
            if (lane == 0)
                mbar_expect_tx(bar, ((pw & 0xffu) + ((pw >> 8) & 0xffu) + ((pw >> 16) & 0xffu)) * 8u + nws * 128u);
            __syncwarp();
            if (lane < 4) {
                int ws = p.z;
                ws = lane == 1 ? p.y : ws;
                ws = lane == 0 ? p.x : ws;
                unsigned bytes = ((pw >> (8 * lane)) & 0xffu) * 8u;
                long long off = (long long)ws * 8;
                const char* base = Rbytes;
                if (lane == 3) { bytes = nws * 128u; off = (long long)u * (CL_UNITWORDS * 4); base = Lbytes; }
                CL_ASSERT(lane == 3 ? (off >= 0 && off + bytes <= (long long)a.Nalloc * CL_NW * 4)
                                    : (off >= 0 && off + bytes <= (long long)a.Nalloc * 8 && bytes <= CL_WIN * 8));
                CL_ASSERT((off & 15) == 0 && (bytes & 15) == 0);
                if (bytes) bulk_g2s(my_dst + buf * my_stride, base + off, bytes, bar);
            }
        }
    };
#endif
    // Schedule: the first ~60 % of the units statically interleaved (no traffic), the rest drawn one by
    // one from a per-step counter: warps that met several slow (edge) units take fewer of the tail.
    const int rounds0 = (int)(a.static_frac * (float)((u_hi - u_lo) / W));
    const int dyn_lo = u_lo + rounds0 * W;
    // (the dynamic draw returns the RAW counter value of lane 0; `fix` adds the base after the broadcast,
    //  a whole unit later, so that no instruction waits for the atomic's round trip to L2)
    auto grab = [&](int j) -> int {                       // j-th unit of this warp, relative to base(j)
        if (j < rounds0) return gw + j * W;
        int t = 0;
        if (lane == 0) t = atomicAdd(&a.sched[fl.par * CL_QMAX + ctx.q], 1);
        return t;
    };
    // dynamic units are dealt round-robin to the SM queues: the CTAs that share an SM (and its issue
    // slots, which the warp arbiter does not hand out evenly) draw from the same counter.  (Measured and
    // dropped: a warp whose queue has run dry trying 3 / 8 other SMs' queues - 144.3 / 147.4 against
    // 143.3 us/step: the failed attempts of the last warps cost more than the stolen units save; keeping the
    // last 3 - 20 % of the units in one global overflow queue - 142.1 ... 144.5 vs 142.9 us/step: no effect.)
    auto fix = [&](int raw, int j) -> int { return j < rounds0 ? raw + u_lo : dyn_lo + ctx.q + ctx.nq * raw; };
    const int4 z4 = make_int4(0, 0, 0, 0);
    int u = fix(__shfl_sync(0xffffffffu, grab(0), 0), 0), un = fix(__shfl_sync(0xffffffffu, grab(1), 0), 1);
    int4 p = z4, q = z4;
    if (u < u_hi) p = a.wplan[u];
    if (un < u_hi) q = a.wplan[un];
    issue(u, p, 0);
#if CL_DEPTH3
    int g3 = grab(2);
#endif

    for (int k = 0; u < u_hi; ++k) {
        const int buf = k & 1;
        issue(un, q, buf ^ 1);                            // next unit's windows + words
#if CL_DEPTH3
        // (older schedule: a warp holds three units - the draw is made a whole unit before its plan is read)
        const int unn = fix(__shfl_sync(0xffffffffu, g3, 0), k + 2);
        g3 = grab(k + 3);
        int4 r = z4;
        if (unn < u_hi) r = a.wplan[unn];                 // consumed next iteration
#else
        // the unit after next is drawn now; its number is broadcast and its plan requested after the pair
        // loop (the atomic's round trip hides behind it, the plan's behind the epilogue), so a warp holds
        // TWO units when the queue runs dry: a shorter tail at the step barrier
        const int g = grab(k + 2);
#endif
        const int  i    = u * 32 + lane;
        const bool live = (i >= ctx.own_s) & (i < ctx.own_e);
        // epilogue operands requested now, consumed after the pair loop
        float2 v = make_float2(0.0f, 0.0f), rb = make_float2(0.0f, 0.0f);
        if (live && (PLAIN || rc.nsteps > 0)) { v = V[i]; rb = a.Rb[i]; }
        float2 ri = make_float2(0.0f, 0.0f);
        float Fx = 0.0f, Fy = 0.0f, pe = 0.0f, ke = 0.0f, vir = 0.0f;
#if CL_COPY == 1
        cp_async_wait<1>();                               // this unit's copy group has landed
        __syncwarp();
#endif
        if (p.w < 0) {
#if CL_COPY == 0
            // this unit's copies have landed when the buffer's mbarrier completes its phase
            const unsigned bar = wp.bar + buf * 8, par = (wp.phase >> buf) & 1u;
            if (!mbar_try_wait(bar, par)) mbar_wait_slow(a, bar, par);
            wp.phase ^= 1u << buf;
#endif
            const unsigned win = wp.base + buf * CL_WINBYTES;
            CL_ASSERT(!live || (i - p.y >= 0 && i - p.y < (int)(((unsigned)p.w >> 8) & 0xffu)));
#ifdef LJMD_DEBUG_CHECKS
            if (live) {   // every listed index names a staged slot of its window or the sentinel
                const unsigned pw = (unsigned)p.w;
                const int nwd = (int)((pw >> 24) & 0x7fu);
                for (int w = 0; w < nwd; ++w) {
                    const unsigned word = a.nb4[(size_t)u * CL_UNITWORDS + w * 32 + lane];
                    for (int b = 0; b < 4; ++b) {
                        const int idx = (int)((word >> (8 * b)) & 0xffu);
                        const int k = idx / CL_WIN;
                        CL_ASSERT(idx == CL_DUMMY || (k < 3 && idx - k * CL_WIN < (int)((pw >> (8 * k)) & 0xffu)));
                    }
                }
            }
#endif
            if (live) ri = lds64(win + (CL_WIN + (i - p.y)) * 8);      // own row window holds the own slot
            bytes_force_staged<PE, VIR>(a, win, wp.base + 2 * CL_WINBYTES + buf * CL_SWBYTES, u,
                                        (int)(((unsigned)p.w >> 24) & 0x7fu), ri, Fx, Fy, pe, vir);
        } else {
            unsigned meta = 0u;
            const int ii = live ? i : ctx.own_s;
            if (live) { ri = R[i]; meta = a.meta[i]; }
            const int n = meta & 0xff;
            const bool wedge = __any_sync(0xffffffffu, (meta & 0x100u) != 0u);
            if (wedge) list_force<PE, true,  VIR>(a, R, ii, n, ri, Fx, Fy, pe, vir);
            else       list_force<PE, false, VIR>(a, R, ii, n, ri, Fx, Fy, pe, vir);
        }
#if !CL_DEPTH3
        const int unn = fix(__shfl_sync(0xffffffffu, g, 0), k + 2);
        int4 r = z4;
        if (unn < u_hi) r = a.wplan[unn];                 // consumed at the top of the next iteration
#endif
        if (live) {
            if (kick1) { v.x = kick(v.x, Fx, a.dt); v.y = kick(v.y, Fy, a.dt); }               // MD:74
            if (want_ke) ke = v.x * v.x + v.y * v.y;
            int o = 0;
            if (!PLAIN) o = (sample || (final && !thermo)) ? og[i] : 0;
            if (sample) rc.traj[(size_t)(fl.s / rc.sample_every) * a.N + o] = ri;              // MD:93-100
            if (thermo) {
                V[i] = v;
                a.Fs[i] = make_float2(Fx, Fy);
            } else if (final) {
                if (a.blk > 0) {
                    const int qd = o / a.blk, oo = o - qd * a.blk;
                    a.peer_stageR[qd][oo] = ri;
                    a.peer_stageV[qd][oo] = v;
                } else {
                    if (a.R_out) a.R_out[o] = ri;
                    if (a.V_out) a.V_out[o] = v;
                    if (a.F_out) a.F_out[o] = make_float2(Fx, Fy);
                }
            } else {
                v.x = kick(v.x, Fx, a.dt); v.y = kick(v.y, Fy, a.dt);                           // MD:70
                V[i] = v;
                const float2 rn = make_float2(drift(ri.x, v.x, a.dt, a.pc.box),                 // MD:71-72
                                              drift(ri.y, v.y, a.dt, a.pc.box));
                Rnext[i] = rn;
                if (a.P > 1) {
                    // halo exchange: the new position and velocity of a boundary-row particle go
                    // straight into the neighbour's halo slot (NVLink peer store)
                    if (i < first_e) {
                        const int j = peer_hi_start + (i - ctx.own_s);
                        a.peerR[ctx.pr ^ 1][dn][j] = rn; a.peerV[ctx.pv][dn][j] = v;
                    }
                    if (i >= last_s) {
                        const int j = i - last_s;
                        a.peerR[ctx.pr ^ 1][up][j] = rn; a.peerV[ctx.pv][up][j] = v;
                    }
                }
                const float ddx = min_image(__fsub_rn(rn.x, rb.x), a.pc.box, a.pc.timg);
                const float ddy = min_image(__fsub_rn(rn.y, rb.y), a.pc.box, a.pc.timg);
                moved |= (ddx * ddx + ddy * ddy > a.half_skin2);
            }
        }
        // the warps that pushed halo particles order those peer stores at system scope now (hidden behind
        // the other warps' work) instead of every thread of the grid fencing at the end of the step
        if (a.P > 1 && !thermo && !final) {
            const bool pushed = live && (i < first_e || i >= last_s);
            if (__any_sync(0xffffffffu, pushed)) __threadfence_system();
        }
        // per-unit energy partials (fixed shuffle tree), summed in unit order after the barrier
        if (PE) {
            const float t = warp_sum(live ? pe : 0.0f);       // (idle lanes of a boundary unit evaluate a dummy)
            if (lane == 0) __stcg(&a.pe_part[fl.par * a.nchunks + (u - u_lo)], t);
        }
        if (VIR) {
            const float t = warp_sum(live ? vir : 0.0f);
            if (lane == 0) __stcg(&a.vir_part[fl.par * a.nchunks + (u - u_lo)], t);
        }
        if (want_ke) {
            const float t = warp_sum(ke);
            if (lane == 0) __stcg(&a.ke_part[fl.par * a.nchunks + (u - u_lo)], t);
        }
        __syncwarp();                                     // all lanes are done with `buf`
        u = un; un = unn; p = q; q = r;
    }
#if CL_COPY == 1
    cp_async_wait<0>();
#endif
}

extern __shared__ __align__(16) unsigned char cells_smem[];

// VIR: the energy steps also accumulate the pair virial (own instantiation, launched only on request)
template <bool VIR>
__global__ void __launch_bounds__(CL_THREADS, 1024 / CL_THREADS)
cells_persistent_kernel(const CellsArgs a) {
    __shared__ int    sscan[CL_THREADS / 32 + 1];
    __shared__ double sdbl[CL_THREADS / 32];
    __shared__ float  s_lambda;
    __shared__ long long s_pt[12];
    __shared__ __align__(8) unsigned long long s_mbar[CL_WARPS][2];
    const int tid = threadIdx.x, gtid = blockIdx.x * CL_THREADS + tid, gsz = a.G * CL_THREADS;
    const RunCtl rc = a.rc;
    Ctx ctx;
    ctx.epoch = 0;
    ctx.pt = a.prof ? s_pt : nullptr;
    if (ctx.pt && tid == 0) { for (int k = 0; k < 11; ++k) s_pt[k] = 0; s_pt[11] = clock64(); }
    ctx.pr = a.state[ST_PR];
    ctx.pv = a.state[ST_PV];
    ctx.nheld = a.state[ST_NHELD];
    ctx.own_s = a.state[ST_OWN_S];
    ctx.own_e = a.state[ST_OWN_E];
    ctx.xepoch = (unsigned)a.state[ST_XEPOCH];
    // per warp: two window buffers (+ sentinel slots) and two word buffers, filled by bulk copies; the
    // list build uses window buffer 0 and lays its byte rows over everything behind it
    float2* my_win = reinterpret_cast<float2*>(cells_smem + (size_t)(tid >> 5) * CL_WARP_SMEM);
    unsigned char* my_bytes = cells_smem + (size_t)(tid >> 5) * CL_WARP_SMEM + CL_WINBYTES;
    WarpPipe wp;
    // (the two addresses pass through an opaque move: ptxas otherwise rebuilds them from the CTA's
    //  shared window and the warp index at every use instead of keeping two registers)
    asm volatile("mov.u32 %0, %1;" : "=r"(wp.base) : "r"(smem_u32(my_win)));
    asm volatile("mov.u32 %0, %1;" : "=r"(wp.bar) : "r"(smem_u32(&s_mbar[tid >> 5][0])));
    wp.phase = 0u;
    if ((tid & 31) == 0) {
        mbar_init(wp.bar, 1);
        mbar_init(wp.bar + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // unit queues: the CTAs resident on one SM share a queue.  The first CTA of an SM to get here takes
    // the next queue number and publishes it in the SM's table entry (the launch is cooperative, so the
    // CTA being waited for is resident).  Table and count are zeroed by the host before every launch.
    {
        __shared__ int s_q;
        if (tid == 0) {
            unsigned smid;
            asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
            int* tab = a.sched + 2 * CL_QMAX;
            int* qcount = tab + CL_QMAX;
            const int slot = (int)(smid % CL_QMAX);
            int v = atomicCAS(&tab[slot], 0, -1);
            if (v == 0) {
                v = atomicAdd(qcount, 1) + 1;
                atomicExch(&tab[slot], v);
            } else {
                const long long t0 = clock64();
                while ((v = atomicAdd(&tab[slot], 0)) <= 0) {
                    if (a.spin_limit > 0 && clock64() - t0 > a.spin_limit) { atomicExch(a.state + ST_ABORT, 1); v = 1; break; }
                }
            }
            s_q = v - 1;
        }
        __syncthreads();
        ctx.q = s_q;
    }
    CL_BARRIER();
    ctx.nq = max(1, __ldcg(a.sched + 3 * CL_QMAX));

    if (a.s_begin < 0) {
        // load the caller's state (original order) and sort it.  Slabs: every rank reads the whole
        // (replicated) input and keeps the particles of its owned rows, in arrival order (the sort
        // orders them); the halo rows are filled by the neighbours during the rebuild.
        if (a.P == 1) {
            for (int i = gtid; i < a.N; i += gsz) {
                a.R[ctx.pr][i] = load_wrap(a.R_in[i], a.pc.box);
                a.V[ctx.pv][i] = a.V_in ? a.V_in[i] : make_float2(0.0f, 0.0f);
                a.orig[ctx.pv][i] = i;
            }
            ctx.nheld = a.N;
        } else {
            for (int i = gtid; i < a.N; i += gsz) {
                const float2 r = load_wrap(a.R_in[i], a.pc.box);
                if (owned_row(a, local_row(a, r.y))) {
                    const int k = atomicAdd(a.state + ST_LOADCNT, 1);
                    if (k < a.Nalloc) {
                        a.R[ctx.pr][k] = r;
                        a.V[ctx.pv][k] = a.V_in ? a.V_in[i] : make_float2(0.0f, 0.0f);
                        a.orig[ctx.pv][k] = i;
                    } else {
                        atomicOr(a.state + ST_ERR, CERR_CAPACITY);
                    }
                }
            }
            CL_BARRIER();
            ctx.nheld = min(__ldcg(a.state + ST_LOADCNT), a.Nalloc);
        }
        CL_BARRIER();
        cells_rebuild(a, ctx, sscan, my_win, my_bytes, (a.mode == 1) ? a.count_r2 : a.rlist2);
        if (a.mode == 1) {
            const int* og = a.orig[ctx.pv];
            for (int i = gtid; i < a.N; i += gsz) a.count_out[og[i]] = a.key[i];
            if (gtid == 0) { a.state[ST_PR] = ctx.pr; a.state[ST_PV] = ctx.pv; }
            return;
        }
    }

    for (long long s = a.s_begin; s < a.s_end; ++s) {
        const int  par     = (int)((s + 1) & 1);
        const bool kick1   = (s >= 0);
        const bool final   = (s == rc.nsteps - 1);
        const bool want_e  = kick1 && rc.energy_every > 0 && (s % rc.energy_every == 0);
        bool       want_pe = want_e || (rc.nsteps == 0 && a.pe_out != nullptr);
        if constexpr (VIR) want_pe = want_pe || (rc.nsteps == 0 && a.vir_out != nullptr);   // ljmd_virial
        const bool thermo  = kick1 && rc.thermo_every > 0 && rc.thermo_kT > 0.0f &&
                             ((s + 1) % rc.thermo_every == 0);
        const bool sample  = kick1 && rc.sample_every > 0 && (s % rc.sample_every == 0) &&
                             (s / rc.sample_every < rc.S);
        const bool want_ke = want_e || thermo;
        // rebuild requested by the previous step's displacement test?
        if (s > a.s_begin || a.s_begin >= 0) {
            if (__ldcg(a.state + ST_FLAG) == (int)(s + 1)) cells_rebuild(a, ctx, sscan, my_win, my_bytes, a.rlist2);
        }
        // (slabs: ST_FLAG holds the decision of ALL ranks, see the end of the step)
        const float2* __restrict__ R = a.R[ctx.pr];
        float2*       Rnext = a.R[ctx.pr ^ 1];
        float2*       V     = a.V[ctx.pv];
        const int*    og    = a.orig[ctx.pv];
        StepFlags fl;
        fl.s = s; fl.par = par; fl.kick1 = kick1; fl.final = final; fl.want_e = want_e; fl.want_pe = want_pe;
        fl.want_ke = want_ke; fl.thermo = thermo; fl.sample = sample;
        const int u_lo = ctx.own_s >> 5, u_hi = (ctx.own_e + 31) >> 5;      // 32-slot units
        for (int k = gtid; k < CL_QMAX; k += gsz) __stcg(&a.sched[(par ^ 1) * CL_QMAX + k], 0);   // the other parity's unit counters: idle this step
        int moved = 0;
        if (want_pe)
            warp_pass<true, false, VIR>(a, ctx, fl, wp, moved);
        else if (kick1 && !final && !thermo && !sample && !want_ke)
            warp_pass<false, true, false>(a, ctx, fl, wp, moved);
        else
            warp_pass<false, false, false>(a, ctx, fl, wp, moved);
        if (thermo) {
            CL_BARRIER();
            const double ke2 = block_sum_array(a.ke_part + par * a.nchunks, u_hi - u_lo, sdbl);
            if (tid == 0) s_lambda = ke2 > 0.0 ? sqrtf(rc.thermo_kT / ((float)(0.5 * ke2) / (float)a.N)) : 1.0f;
            __syncthreads();
            const float lam = s_lambda;
            for (int i = ctx.own_s + gtid; i < ctx.own_e; i += gsz) {
                const float2 ri = R[i];
                const float2 F = a.Fs[i];
                float2 v = V[i];
                v.x *= lam; v.y *= lam;
                if (final) {
                    const int o = og[i];
                    if (a.R_out) a.R_out[o] = ri;
                    if (a.V_out) a.V_out[o] = v;
                    if (a.F_out) a.F_out[o] = F;
                } else {
                    v.x = kick(v.x, F.x, a.dt); v.y = kick(v.y, F.y, a.dt);
                    V[i] = v;
                    const float2 rn = make_float2(drift(ri.x, v.x, a.dt, a.pc.box),
                                                  drift(ri.y, v.y, a.dt, a.pc.box));
                    Rnext[i] = rn;
                    const float2 rb = a.Rb[i];
                    const float ddx = min_image(__fsub_rn(rn.x, rb.x), a.pc.box, a.pc.timg);
                    const float ddy = min_image(__fsub_rn(rn.y, rb.y), a.pc.box, a.pc.timg);
                    moved |= (ddx * ddx + ddy * ddy > a.half_skin2);
                }
            }
        }
        // a particle left the skin/2 ball: ask for a rebuild before the next force evaluation.
        // The flag carries the step stamp, so it never needs clearing (no reset race).
        if (__syncthreads_or(moved) && tid == 0) __stcg(a.state + (a.P > 1 ? ST_LMOVED : ST_FLAG), (int)(s + 2));
        if (!final) ctx.pr ^= 1;
        CL_PROF(0);
        if (final && a.blk > 0) __threadfence_system();      // the staged outputs live on peer GPUs
        unsigned long long gt0 = 0;
        if (ctx.pt && tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt0));
        CL_BARRIER();
        if (ctx.pt && tid == 0) {                            // (debug) wall-clock ns of this CTA's arrival / exit
            unsigned long long gt1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt1));
            ctx.pt[9] = (long long)gt0; ctx.pt[10] = (long long)gt1;
        }
        CL_PROF(1);
        if (a.P > 1 && final && a.blk > 0) (void)peer_sync(a, ctx, false);   // every rank's outputs have landed
        if (a.P > 1 && !final) {
            // one NVLink round trip per step: every rank's halo pushes have landed once all arrival
            // words carry this epoch; the words also carry "one of my particles left its skin/2 ball",
            // so that all ranks rebuild at the same step
            const bool mine = (__ldcg(a.state + ST_LMOVED) == (int)(s + 2));
            const bool any = peer_sync(a, ctx, mine);
            if (any && gtid == 0) __stcg(a.state + ST_FLAG, (int)(s + 2));
            if (any) CL_BARRIER();                           // (rare) the flag is read at the next step
        }
        CL_PROF(8);

        if (blockIdx.x == 0 && want_pe) {
            const double pe2 = block_sum_array(a.pe_part + par * a.nchunks, u_hi - u_lo, sdbl);
            double ke2 = 0.0, w2 = 0.0;
            if (want_e) ke2 = block_sum_array(a.ke_part + par * a.nchunks, u_hi - u_lo, sdbl);
            if (VIR) w2 = block_sum_array(a.vir_part + par * a.nchunks, u_hi - u_lo, sdbl);
            if (tid == 0) {
                if (want_e) {
                    float* o = rc.ke_pe + 2 * (s / rc.energy_every);
                    o[0] = (float)(0.5 * ke2);
                    o[1] = (float)(0.5 * pe2);
                    if (VIR) a.vir_out[s / rc.energy_every] = (float)(0.5 * w2);
                } else {
                    if (!VIR || a.pe_out) a.pe_out[0] = (float)(0.5 * pe2);
                    if (VIR) a.vir_out[0] = (float)(0.5 * w2);
                }
            }
        }
    }
    if (gtid == 0) {
        a.state[ST_PR] = ctx.pr; a.state[ST_PV] = ctx.pv;
        a.state[ST_NHELD] = ctx.nheld; a.state[ST_OWN_S] = ctx.own_s; a.state[ST_OWN_E] = ctx.own_e;
        a.state[ST_XEPOCH] = (int)ctx.xepoch;
    }
    if (ctx.pt && tid == 0)
        for (int k = 0; k < 11; ++k) a.prof[blockIdx.x * 12 + k] = s_pt[k];
}

// ---- stand-alone binning for ljmd_cell_assign (original order) ------------------------------------
__global__ void cell_assign_kernel(const float2* __restrict__ R, int N, int nrows, int nbx, float inv_hy,
                                   float inv_wx, int* __restrict__ cell_id, int* __restrict__ cell_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const float2 r = R[i];
    const int c = strip_coord(r.y, inv_hy, nrows) * nbx + strip_coord(r.x, inv_wx, nbx);
    if (cell_id) cell_id[i] = c;
    if (cell_count) atomicAdd(&cell_count[c], 1);
}

}  // namespace

// ----------------------------------------------------------------------------------------------------
struct Cells {
    int G = 0, nrows = 0, nbx = 0, ncells = 0, Nalloc = 0, nchunks = 0;
    int P = 1, g0 = 0, nloc = 0, nlr = 0, own_lo = 0, ncells_max = 0;
    int nloc_of[LJMD_MAX_RANKS] = {};
    float inv_hy = 0, inv_wx = 0, hy = 0, wx = 0, rlist = 0;
    // one allocation (IPC-shared with the peers when P > 1): R[2], V[2], orig[2], cell_count, arrival
    // words, mailbox -- at the same offsets on every rank
    void* shared = nullptr;
    size_t off_R[2] = {}, off_V[2] = {}, off_O[2] = {}, off_cc = 0, off_flags = 0, off_mail = 0;
    size_t off_stage[2] = {};       // block-distributed output staging (R, V), P > 1 only
    float2 *Rfull = nullptr, *Vfull = nullptr;   // all-gathered input of ljmd_run_blocked (allocated on first use)
    char* peer_base[LJMD_MAX_RANKS] = {};
    float2 *Rb = nullptr, *Fs = nullptr;
    int *key = nullptr, *rank = nullptr, *tmpk = nullptr, *tmpo = nullptr, *tmpc = nullptr,
        *cell_start = nullptr, *row_tot = nullptr;
    unsigned* meta = nullptr;
    uint2* ent = nullptr;
    unsigned* nb4 = nullptr;
    int4* wplan = nullptr;
    float *pe_part = nullptr, *ke_part = nullptr, *vir_part = nullptr;
    bool vir_fits = false;          // the virial kernel is co-resident on the grid G of the force kernel
    int* state = nullptr;
    int* sched = nullptr;
    unsigned* bar = nullptr;
    long long* prof = nullptr;
};

int cells_create(ljmd_handle* h) {
    Cells* cl = new Cells();
    h->cells = cl;
    const long long N = h->p.N;
    const int P = h->nranks;
    cl->P = P;
    if (N > (1ll << 30)) { set_error("N too large for 32-bit particle indices"); return LJMD_E_INVALID; }
    const float rc = h->p.rc, skin = h->p.skin;
    cl->rlist = rc + skin;
    // rows at least rc + skin high, bins at least (rc + skin) / K wide, each with a few ulp(box) of
    // margin for the fp32 binning (one multiply + truncation)
    const double ulp = (double)(nextafterf(h->p.box, 2.0f * h->p.box) - h->p.box);
    cl->nrows = (int)floor((double)h->p.box / ((double)cl->rlist + 8.0 * ulp));
    cl->nbx   = (int)floor((double)h->p.box / ((double)cl->rlist / CL_K + 4.0 * ulp));
    if (cl->nrows < 3 || cl->nbx < 2 * CL_K + 1) {
        set_error("box %.3f is smaller than 3 rows of height rc+skin=%.3f: use the all-pairs path",
                  h->p.box, cl->rlist);
        return LJMD_E_INVALID;
    }
    if ((long long)cl->nrows * cl->nbx > (1ll << 30)) { set_error("cell index too large"); return LJMD_E_INVALID; }
    cl->hy = h->p.box / (float)cl->nrows;
    cl->wx = h->p.box / (float)cl->nbx;
    cl->inv_hy = (float)cl->nrows / h->p.box;
    cl->inv_wx = (float)cl->nbx / h->p.box;
    // slab decomposition: contiguous blocks of rows, as even as possible; one halo row per side
    if (P > 1 && cl->nrows < 2 * P) {
        set_error("cell list: %d rows cannot be split over %d GPUs (need 2 rows per GPU)", cl->nrows, P);
        return LJMD_E_INVALID;
    }
    int g = 0, maxloc = 0;
    for (int q = 0; q < P; ++q) {
        cl->nloc_of[q] = cl->nrows / P + (q < cl->nrows % P ? 1 : 0);
        if (q == h->rank) cl->g0 = g;
        g += cl->nloc_of[q];
        maxloc = std::max(maxloc, cl->nloc_of[q]);
    }
    cl->nloc = cl->nloc_of[h->rank];
    cl->own_lo = (P > 1) ? 1 : 0;
    cl->nlr = cl->nloc + 2 * cl->own_lo;
    cl->ncells = cl->nlr * cl->nbx;
    cl->ncells_max = (maxloc + 2 * cl->own_lo) * cl->nbx;
    if (P == 1) {
        cl->Nalloc = (int)(((N + 2 + 63) / 64) * 64);    // (+2: a bulk copy may read one slot past a window)
    } else {
        // owned rows + two halo rows, with room for density fluctuations between slabs
        const double per = (double)N / P;
        const double row = (double)N / cl->nrows;
        cl->Nalloc = (int)((((long long)(1.35 * per + 6.0 * row) + 4096 + 63) / 64) * 64);
    }
    cl->nchunks = cl->Nalloc / 32 + 2;              // capacity in 32-slot units (energy partials)

    const size_t smem = (size_t)CL_WARPS * CL_WARP_SMEM;
    LJ_CUDA(cudaFuncSetAttribute(cells_persistent_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    LJ_CUDA(cudaFuncSetAttribute(cells_persistent_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0, per_sm_vir = 0;
    LJ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cells_persistent_kernel<false>, CL_THREADS, smem));
    LJ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_vir, cells_persistent_kernel<true>, CL_THREADS, smem));
    if (per_sm < 1) { set_error("cell-list kernel does not fit on an SM"); return LJMD_E_STATE; }
    if (const char* e = getenv("LJMD_CELLS_CTAS_PER_SM")) per_sm = std::min(per_sm, std::max(1, atoi(e)));
    long long gg = (long long)per_sm * h->num_sms;
    gg = std::min<long long>(gg, std::max<long long>(1, (N / P + CL_THREADS - 1) / CL_THREADS));
    cl->G = (int)gg;
    cl->vir_fits = (long long)per_sm_vir * h->num_sms >= gg;

    const size_t na = (size_t)cl->Nalloc;
    {   // the shared allocation
        auto up = [](size_t x) { return (x + 255) / 256 * 256; };
        size_t off = 0;
        for (int k = 0; k < 2; ++k) { cl->off_R[k] = off; off += up(sizeof(float2) * na); }
        for (int k = 0; k < 2; ++k) { cl->off_V[k] = off; off += up(sizeof(float2) * na); }
        for (int k = 0; k < 2; ++k) { cl->off_O[k] = off; off += up(sizeof(int) * na); }
        cl->off_cc = off;    off += up(sizeof(int) * (size_t)cl->ncells_max);
        cl->off_flags = off; off += up(sizeof(unsigned) * 2 * LJMD_MAX_RANKS);
        cl->off_mail = off;  off += up(sizeof(int) * MB_WORDS);
        if (P > 1 && N % P == 0)
            for (int k = 0; k < 2; ++k) { cl->off_stage[k] = off; off += up(sizeof(float2) * (size_t)(N / P)); }
        const size_t bytes = std::max<size_t>((off + (2u << 20) - 1) / (2u << 20) * (2u << 20), 4u << 20);
        LJ_CUDA(cudaMalloc(&cl->shared, bytes));
        LJ_CUDA(cudaMemset(cl->shared, 0, bytes));
        cl->peer_base[h->rank] = reinterpret_cast<char*>(cl->shared);
        if (P > 1) {
            void* peers[LJMD_MAX_RANKS];
            int r = dist_share(h, cl->shared, peers);
            if (r) return r;
            for (int q = 0; q < P; ++q) cl->peer_base[q] = reinterpret_cast<char*>(peers[q]);
        }
    }
    LJ_CUDA(cudaMalloc(&cl->Rb, sizeof(float2) * na));
    LJ_CUDA(cudaMalloc(&cl->Fs, sizeof(float2) * na));
    LJ_CUDA(cudaMalloc(&cl->key, sizeof(int) * na));
    LJ_CUDA(cudaMalloc(&cl->rank, sizeof(int) * na));
    LJ_CUDA(cudaMalloc(&cl->tmpk, sizeof(int) * na));
    LJ_CUDA(cudaMalloc(&cl->tmpo, sizeof(int) * na));
    LJ_CUDA(cudaMalloc(&cl->tmpc, sizeof(int) * na));
    LJ_CUDA(cudaMalloc(&cl->meta, sizeof(unsigned) * na));
    LJ_CUDA(cudaMalloc(&cl->ent, sizeof(uint2) * na * CL_E));
    LJ_CUDA(cudaMalloc(&cl->wplan, sizeof(int4) * (na / 32 + 1)));
    LJ_CUDA(cudaMalloc(&cl->nb4, sizeof(unsigned) * na * CL_NW));
    LJ_CUDA(cudaMalloc(&cl->cell_start, sizeof(int) * ((size_t)cl->ncells + 1)));
    LJ_CUDA(cudaMalloc(&cl->row_tot, sizeof(int) * (size_t)cl->nlr));
    LJ_CUDA(cudaMalloc(&cl->pe_part, sizeof(float) * 2 * cl->nchunks));
    LJ_CUDA(cudaMalloc(&cl->ke_part, sizeof(float) * 2 * cl->nchunks));
    LJ_CUDA(cudaMalloc(&cl->state, sizeof(int) * ST_WORDS));
    LJ_CUDA(cudaMemset(cl->state, 0, sizeof(int) * ST_WORDS));
    LJ_CUDA(cudaMalloc(&cl->bar, sizeof(unsigned)));
    LJ_CUDA(cudaMalloc(&cl->sched, sizeof(int) * (3 * CL_QMAX + 1)));
    if (getenv("LJMD_CELLS_PROF")) LJ_CUDA(cudaMalloc(&cl->prof, sizeof(long long) * 12 * cl->G));
    return 0;
}

void cells_destroy(ljmd_handle* h) {
    Cells* cl = h->cells;
    if (!cl) return;
    cudaFree(cl->shared);
    cudaFree(cl->Rfull); cudaFree(cl->Vfull);
    cudaFree(cl->Rb); cudaFree(cl->Fs); cudaFree(cl->key); cudaFree(cl->rank);
    cudaFree(cl->tmpk); cudaFree(cl->tmpo); cudaFree(cl->tmpc); cudaFree(cl->meta);
    cudaFree(cl->ent); cudaFree(cl->wplan); cudaFree(cl->nb4);
    cudaFree(cl->cell_start); cudaFree(cl->row_tot);
    cudaFree(cl->pe_part); cudaFree(cl->ke_part); cudaFree(cl->vir_part);
    cudaFree(cl->state); cudaFree(cl->bar); cudaFree(cl->prof); cudaFree(cl->sched);
    delete cl;
    h->cells = nullptr;
}

static void fill_args(ljmd_handle* h, CellsArgs& a) {
    Cells* cl = h->cells;
    a.pc = h->pc;
    a.N = (int)h->p.N; a.Nalloc = cl->Nalloc; a.G = cl->G; a.nchunks = cl->nchunks;
    a.nrows = cl->nrows; a.nbx = cl->nbx; a.ncells = cl->ncells;
    a.P = cl->P; a.me = h->rank; a.g0 = cl->g0; a.nloc = cl->nloc; a.nlr = cl->nlr; a.own_lo = cl->own_lo;
    for (int q = 0; q < LJMD_MAX_RANKS; ++q) a.nloc_of[q] = cl->nloc_of[q];
    a.inv_hy = cl->inv_hy; a.inv_wx = cl->inv_wx;
    a.rlist2 = cl->rlist * cl->rlist;
    a.half_skin2 = (0.5f * h->p.skin) * (0.5f * h->p.skin);
    a.static_frac = 0.5f;      // measured at N = 4M (liquid, 300-step calls, per-SM queues): 0.0 -> 145.8, 0.2 -> 143.4,
                               // 0.4 -> 142.8, 0.6 -> 142.6, 0.8 -> 144.2 us/step (one global queue: 0.4 -> 154.2, 0.8 -> 143.9)
    if (const char* e = getenv("LJMD_CELLS_STATIC")) a.static_frac = fminf(1.0f, fmaxf(0.0f, (float)atof(e)));
    a.dt = h->p.dt;
    a.spin_limit = h->spin_limit;
    for (int q = 0; q < cl->P; ++q) {
        char* base = cl->peer_base[q];
        for (int k = 0; k < 2; ++k) {
            a.peerR[k][q] = reinterpret_cast<float2*>(base + cl->off_R[k]);
            a.peerV[k][q] = reinterpret_cast<float2*>(base + cl->off_V[k]);
            a.peerO[k][q] = reinterpret_cast<int*>(base + cl->off_O[k]);
        }
        a.peer_cc[q] = reinterpret_cast<int*>(base + cl->off_cc);
        a.peer_flags[q] = reinterpret_cast<unsigned*>(base + cl->off_flags);
        a.peer_mail[q] = reinterpret_cast<int*>(base + cl->off_mail);
        a.peer_stageR[q] = reinterpret_cast<float2*>(base + cl->off_stage[0]);
        a.peer_stageV[q] = reinterpret_cast<float2*>(base + cl->off_stage[1]);
    }
    for (int k = 0; k < 2; ++k) { a.R[k] = a.peerR[k][h->rank]; a.V[k] = a.peerV[k][h->rank]; a.orig[k] = a.peerO[k][h->rank]; }
    a.cell_count = a.peer_cc[h->rank];
    a.mail = a.peer_mail[h->rank];
    a.Rb = cl->Rb; a.Fs = cl->Fs;
    a.key = cl->key; a.rank = cl->rank; a.tmpk = cl->tmpk; a.tmpo = cl->tmpo; a.tmpc = cl->tmpc;
    a.cell_start = cl->cell_start; a.row_tot = cl->row_tot;
    a.meta = cl->meta; a.ent = cl->ent; a.wplan = cl->wplan; a.nb4 = cl->nb4;
    a.pe_part = cl->pe_part; a.ke_part = cl->ke_part;
    a.state = cl->state; a.bar = cl->bar; a.prof = cl->prof; a.sched = cl->sched;
}

static int launch(ljmd_handle* h, CellsArgs& a) {
    Cells* cl = h->cells;
    LJ_CUDA(cudaMemsetAsync(cl->bar, 0, sizeof(unsigned), h->stream));
    LJ_CUDA(cudaMemsetAsync(cl->sched, 0, sizeof(int) * (3 * CL_QMAX + 1), h->stream));
    void* args[] = {(void*)&a};
    void* kern = a.vir_out ? (void*)cells_persistent_kernel<true> : (void*)cells_persistent_kernel<false>;
    LJ_CUDA(cudaLaunchCooperativeKernel(kern, dim3(cl->G), dim3(CL_THREADS), args, (size_t)CL_WARPS * CL_WARP_SMEM,
                                        h->stream));
    h->launches++;
    return 0;
}

int cells_run(ljmd_handle* h, const float2* R_in, const float2* V_in, float2* R_out, float2* V_out,
              float2* F_out, float* pe_out, const RunCtl& rc, float* vir_out) {
    Cells* cl = h->cells;
    if (vir_out && (cl->P > 1 || !cl->vir_fits)) {
        set_error("the cell-list virial is single-GPU only and needs its kernel to fit this handle's grid");
        return LJMD_E_UNSUPPORTED;
    }
    if (vir_out && !cl->vir_part) LJ_CUDA(cudaMalloc(&cl->vir_part, sizeof(float) * 2 * cl->nchunks));   // see ap_run
    const long long N = h->p.N;
    const int P = cl->P;
    cudaStream_t st = h->stream;
    const bool blocked = P > 1 && rc.blocked != 0;
    if (blocked) {
        if (N % P != 0 || cl->off_stage[1] == 0) { set_error("block-distributed I/O needs N divisible by the GPU count"); return LJMD_E_INVALID; }
        if (rc.nsteps <= 0 || rc.sample_every > 0 || F_out || !R_out || !V_out) {
            set_error("block-distributed I/O: a run of >= 1 step without trajectory sampling");
            return LJMD_E_UNSUPPORTED;
        }
        // the caller's index blocks -> the full arrays the slab filter of the load phase reads
        if (!cl->Rfull) {
            LJ_CUDA(cudaMalloc(&cl->Rfull, sizeof(float2) * N));
            LJ_CUDA(cudaMalloc(&cl->Vfull, sizeof(float2) * N));
        }
        int r = dist_allgather_from(h, R_in, cl->Rfull, sizeof(float2) * (size_t)(N / P));
        if (!r) r = dist_allgather_from(h, V_in, cl->Vfull, sizeof(float2) * (size_t)(N / P));
        if (r) return r;
        R_in = cl->Rfull; V_in = cl->Vfull;
    }
    if (P > 1) {
        if (rc.thermo_every > 0 && rc.thermo_kT > 0.0f) {
            set_error("the thermostat is not available on the multi-GPU cell-list path");
            return LJMD_E_UNSUPPORTED;
        }
        if (!blocked && ((R_out && R_out == R_in) || (V_out && V_out == V_in))) {
            set_error("multi-GPU cell-list path: outputs must not alias the inputs");
            return LJMD_E_UNSUPPORTED;
        }
        // every rank writes only the particles it owns; the replicated result is the sum
        if (!blocked) {
            if (R_out) LJ_CUDA(cudaMemsetAsync(R_out, 0, sizeof(float2) * N, st));
            if (V_out) LJ_CUDA(cudaMemsetAsync(V_out, 0, sizeof(float2) * N, st));
            if (F_out) LJ_CUDA(cudaMemsetAsync(F_out, 0, sizeof(float2) * N, st));
        }
    }
    if (rc.nsteps > 0 && rc.traj && rc.S > 0)
        LJ_CUDA(cudaMemsetAsync(rc.traj, 0, sizeof(float2) * N * rc.S, st));      // MD:89
    // fresh call: parities 0, rebuild counter 0, flags and status words 0 (the cross-GPU epoch persists)
    LJ_CUDA(cudaMemsetAsync(cl->state, 0, sizeof(int) * ST_XEPOCH, st));
    LJ_CUDA(cudaMemsetAsync(cl->state + ST_LMOVED, 0, sizeof(int) * (ST_WORDS - ST_LMOVED), st));
    CellsArgs a{};
    fill_args(h, a);
    a.R_in = R_in; a.V_in = V_in;
    a.rc = rc;
    a.R_out = R_out; a.V_out = V_out; a.F_out = F_out; a.pe_out = pe_out;
    a.vir_part = cl->vir_part; a.vir_out = vir_out;
    a.blk = blocked ? (int)(N / P) : 0;
    a.mode = 0;
    // bound one launch to roughly half a second (conservative 2e10 particle-steps/s)
    long long chunk = std::max<long long>(1, (long long)(1.0e10 / (double)N));
    if (const char* e = getenv("LJMD_CELLS_CHUNK")) chunk = std::max(1, atoi(e));
    if (h->timed) LJ_CUDA(cudaEventRecord(h->ev0, st));
    long long s = -1;
    while (s < rc.nsteps) {
        const long long e = std::min(rc.nsteps, s + chunk);
        a.s_begin = s; a.s_end = std::max<long long>(e, 0);
        if (P > 1) { int rb = dist_barrier(h); if (rb) return rb; }   // the ranks enter the kernel together
        int r = launch(h, a);
        if (r) return r;
        s = a.s_end;
        if (rc.nsteps == 0) break;
    }
    if (P > 1) {
        // replicated out (NCCL over NVLink, once per call): owner-written entries + zeros elsewhere
        int r = 0;
        if (blocked) {
            // the kernel's last cross-GPU sync guarantees that every owner's stores into this rank's staging
            // block have landed; the next call's entry barrier keeps the peers from overwriting it early
            char* base = reinterpret_cast<char*>(cl->shared);
            LJ_CUDA(cudaMemcpyAsync(R_out, base + cl->off_stage[0], sizeof(float2) * (size_t)(N / P), cudaMemcpyDeviceToDevice, st));
            LJ_CUDA(cudaMemcpyAsync(V_out, base + cl->off_stage[1], sizeof(float2) * (size_t)(N / P), cudaMemcpyDeviceToDevice, st));
        }
        if (!blocked && R_out && (r = dist_allreduce_f32(h, reinterpret_cast<float*>(R_out), (size_t)2 * N))) return r;
        if (!blocked && V_out && (r = dist_allreduce_f32(h, reinterpret_cast<float*>(V_out), (size_t)2 * N))) return r;
        if (F_out && (r = dist_allreduce_f32(h, reinterpret_cast<float*>(F_out), (size_t)2 * N))) return r;
        if (rc.traj && rc.S > 0 && (r = dist_allreduce_f32(h, reinterpret_cast<float*>(rc.traj), (size_t)2 * N * rc.S))) return r;
        if (pe_out && (r = dist_allreduce_f32(h, pe_out, 1))) return r;
        if (rc.ke_pe && rc.energy_every > 0) {       // "energies use one NCCL all-reduce"
            const long long ne = (rc.nsteps + rc.energy_every - 1) / rc.energy_every;
            if ((r = dist_allreduce_f32(h, rc.ke_pe, (size_t)(2 * ne)))) return r;
        }
    }
    if (h->timed) LJ_CUDA(cudaEventRecord(h->ev1, st));
    if (cl->prof) {   // debug: mean clocks per phase of the LAST launch, summed over its steps
        LJ_CUDA(cudaStreamSynchronize(st));
        std::vector<long long> pv(12 * cl->G);
        LJ_CUDA(cudaMemcpy(pv.data(), cl->prof, sizeof(long long) * pv.size(), cudaMemcpyDeviceToHost));
        const char* nm[9] = {"force+integrate", "step barrier", "B1 bin+hist", "B2 row totals",
                             "B3 scan", "B4 scatter", "B5 order+gather", "B6 list build", "cross-GPU sync"};
        for (int k = 0; k < 9; ++k) {
            double mean = 0, mx = 0;
            for (int c = 0; c < cl->G; ++c) { mean += pv[c * 12 + k]; mx = std::max<double>(mx, (double)pv[c * 12 + k]); }
            fprintf(stderr, "[ljmd cells prof] %-16s mean %12.0f  max %12.0f clocks (launch total)\n", nm[k], mean / cl->G, mx);
        }
        {   // the last step barrier of the launch in wall-clock time: how long after the LAST arrival a CTA leaves
            unsigned long long last_arr = 0, first_arr = ~0ull;
            for (int c = 0; c < cl->G; ++c) {
                last_arr = std::max<unsigned long long>(last_arr, (unsigned long long)pv[c * 12 + 9]);
                first_arr = std::min<unsigned long long>(first_arr, (unsigned long long)pv[c * 12 + 9]);
            }
            double mean_exit = 0, max_exit = 0, mean_arr = 0;
            for (int c = 0; c < cl->G; ++c) {
                const double e = (double)((unsigned long long)pv[c * 12 + 10] - last_arr);
                mean_exit += e; max_exit = std::max(max_exit, e);
                mean_arr += (double)(last_arr - (unsigned long long)pv[c * 12 + 9]);
            }
            fprintf(stderr, "[ljmd cells prof] last step barrier: arrivals spread %.2f us (mean CTA waits %.2f us for the last one), "
                            "exit %.2f us (mean) / %.2f us (max) after the last arrival\n",
                    1e-3 * (double)(last_arr - first_arr), 1e-3 * mean_arr / cl->G, 1e-3 * mean_exit / cl->G, 1e-3 * max_exit);
        }
        if (getenv("LJMD_CELLS_PROF_CTAS")) {
            fprintf(stderr, "[ljmd cells prof] force+integrate clocks by CTA (launch total, /1000):");
            for (int c = 0; c < cl->G; ++c) fprintf(stderr, "%s%lld", (c % 16) ? " " : "\n  ", pv[c * 12] / 1000);
            fprintf(stderr, "\n");
        }
    }
    return 0;
}

int cells_geometry(ljmd_handle* h, int* nrows, int* nbx, int* kbins, float* inv_hy, float* inv_wx) {
    Cells* cl = h->cells;
    if (nrows) *nrows = cl->nrows;
    if (nbx) *nbx = cl->nbx;
    if (kbins) *kbins = CL_K;
    if (inv_hy) *inv_hy = cl->inv_hy;
    if (inv_wx) *inv_wx = cl->inv_wx;
    return 0;
}

int cells_assign(ljmd_handle* h, const float2* R, int* cell_id, int* cell_count) {
    Cells* cl = h->cells;
    const int N = (int)h->p.N;
    if (cell_count) LJ_CUDA(cudaMemsetAsync(cell_count, 0, sizeof(int) * (size_t)cl->nrows * cl->nbx, h->stream));
    cell_assign_kernel<<<(N + 255) / 256, 256, 0, h->stream>>>(R, N, cl->nrows, cl->nbx, cl->inv_hy,
                                                               cl->inv_wx, cell_id, cell_count);
    LJ_CUDA(cudaGetLastError());
    h->launches++;
    return 0;
}

int cells_neighbor_count(ljmd_handle* h, const float2* R, float radius, int* nbr_count) {
    Cells* cl = h->cells;
    if (!(radius > 0.0f) || radius > cl->rlist) {
        set_error("neighbor_count radius %.4f must be in (0, rc + skin = %.4f]", radius, cl->rlist);
        return LJMD_E_INVALID;
    }
    if (cl->P > 1) { set_error("neighbor_count is single-GPU only"); return LJMD_E_UNSUPPORTED; }
    LJ_CUDA(cudaMemsetAsync(cl->state, 0, sizeof(int) * ST_XEPOCH, h->stream));
    LJ_CUDA(cudaMemsetAsync(cl->state + ST_LMOVED, 0, sizeof(int) * (ST_WORDS - ST_LMOVED), h->stream));
    CellsArgs a{};
    fill_args(h, a);
    a.R_in = R; a.V_in = nullptr;
    a.mode = 1;
    a.count_r2 = radius * radius;
    a.count_out = nbr_count;
    a.s_begin = -1; a.s_end = 0;
    return launch(h, a);
}

long long cells_last_rebuilds(ljmd_handle* h) {
    Cells* cl = h->cells;
    int v = 0;
    cudaStreamSynchronize(h->stream);
    cudaMemcpy(&v, cl->state + ST_REBUILDS, sizeof(int), cudaMemcpyDeviceToHost);
    return v;
}

int cells_check_error(ljmd_handle* h) {
    Cells* cl = h->cells;
    if (!cl) return 0;
    int e[ST_WORDS] = {};
    LJ_CUDA(cudaMemcpy(e, cl->state, sizeof(e), cudaMemcpyDeviceToHost));
    if (e[ST_ABORT]) {
        set_error("cell-list persistent kernel: %s timed out (LJMD_SPIN_TIMEOUT_S)",
                  e[ST_ABORT] == 2 ? "a peer GPU's arrival word" : "a grid barrier");
        return LJMD_E_TIMEOUT;
    }
    if (e[ST_ERR] & CERR_LIST_OVERFLOW) {
        set_error("cell-list: a particle has more neighbours within rc + skin than its Verlet list holds "
                  "(%d; %d (slot, mask) entries for warps at the box edge): too dense for this rc + skin",
                  4 * CL_NW, CL_E);
        return LJMD_E_OVERFLOW;
    }
    if (e[ST_ERR] & CERR_CAPACITY) {
        set_error("cell-list: a slab holds more particles than its buffers (density too uneven over the GPUs)");
        return LJMD_E_OVERFLOW;
    }
    if (e[ST_ERR] & CERR_DEBUG) {
        set_error("cell-list: a debug bounds assertion failed (LJMD_DEBUG_CHECKS build)");
        return LJMD_E_STATE;
    }
    return 0;
}

}  // namespace ljmd
