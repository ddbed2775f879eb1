// allpairs.cu — dense O(N^2) path: the reference's own formulation (MD:50-75) on B200.
//
// Every kernel here is PERSISTENT: one launch runs a whole equilibrate_fn / production_fn call
// (MD:77-106) without returning to the host.  Three kernels, chosen at create (ljmd_allpairs_mode):
//
//   ap_cluster_kernel            N <= 640, one GPU: one thread-block cluster, positions in distributed
//                                shared memory, velocities in registers, one cluster barrier per step.
//   ap_persistent_kernel<3>      N >= 2048: Newton's-third-law tiles (64 i x 32 j, the j particle and its
//                                force travel around the warp by shuffle), patch partial vectors, dynamic
//                                patch queue; on several GPUs the patches are dealt to the ranks and the
//                                partial forces are reduce-scattered with NVLink peer stores.
//   ap_persistent_kernel<1|2>    everything else: ordered pairs, the flattened
//                                (i-block x j) work cut into equal-cost contiguous ranges (stream-K style),
//                                j positions staged through shared memory.
//
// The grid kernels run, per step:  [b] partial forces -> grid barrier -> [d] reduce the partials in a
// fixed order (deterministic, atomic-free), finish the velocity-Verlet step, write the sample / energies,
// drift into the other position buffer (ping-pong) -> grid barrier.
//
// F(R_new) of step n is carried to step n+1 (the reference recomputes it, bit-identically:
// SURVEY.md §0), so there is one O(N^2) evaluation per step.  Each particle's state is read
// and written once per step.
#include "ljmd_device.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdio>
#include <type_traits>

namespace cg = cooperative_groups;

namespace ljmd {

namespace {

constexpr int AP_THREADS = 128;   // 4 warps: one per SM sub-partition
constexpr int AP_MINBLOCKS = 4;   // CTAs per SM the grid kernel's register budget is sized for
constexpr int AP_UNROLL  = 8;     // j particles per unrolled inner-loop body (ordered pairs)
constexpr int AP_TB_UNROLL = 4;   // rotation steps per unrolled body of tile_both
constexpr int J_UNIT     = 8;     // granularity of the j split (particles)
constexpr int TILE_J     = 512;   // j particles staged per shared-memory tile (8 KB)
constexpr int RED_LANES  = 8;     // lanes that cooperate on one particle's partial sum
constexpr int RED_BATCH  = 6;     // partial vectors a lane keeps in flight (tile mode)
constexpr float SENT_I   = -1.0e18f;   // padding i particles, far from every SENT_J (ljmd_device.cuh)

struct ApArgs {
    PairConsts pc;
    int   N, G, NJu, nI, maxseg, ppc;   // ppc = particles owned per CTA in phase [d]
    int   i_lo, Nloc;                   // this rank owns particles [i_lo, i_lo + Nloc) (atom decomposition)
    int   rank, P;                      // P > 1: positions are pushed to every peer over NVLink
    unsigned xepoch0;                   // cross-GPU barrier epochs already consumed by earlier launches
    float2*   peerR0[LJMD_MAX_RANKS];   // every rank's ping-pong position buffers (peer-mapped)
    float2*   peerR1[LJMD_MAX_RANKS];
    unsigned* peer_flags[LJMD_MAX_RANKS];   // every rank's arrival words [P]; [rank] is the local one
    float dt;
    const long long* cta_start;   // [G+1] flat (i-block * NJu + j-unit) range owned by each CTA
    const int*       cta_ib0;     // [G]   first i-block a CTA touches
    const int2*      iblk_ctas;   // [nI]  first / last CTA contributing to an i-block
    const float2*    R_in;        // positions of the state the call starts from
    float2*          Rbuf0;       // ping-pong position buffers
    float2*          Rbuf1;
    float2*          Vh;          // velocities (half-step between kernels' phases)
    float2*          Ftmp;        // forces held across the thermostat barrier
    float2*          part;        // [G*maxseg*BLOCK_I] partial forces
    // Newton's-third-law tile mode (IPT == 3): upper-triangular patches of Pt x Pt tiles of 64 x 64
    int              Pt, q, npr;  // patch edge in tiles, tiles per warp edge (Pt = 2q), patch rows
    int              npatch, npe; // number of patches; number of energy partials per parity
    int*             sched;       // [2] patch counters (by step parity)
    const int2*      patches;     // (pa, pb) patch coordinates, pa <= pb
    // tile mode on several GPUs: the patches are dealt to the ranks; a rank sums ITS partial vectors into one
    // partial force per particle of the WHOLE system and stores it into the owner's receive buffer
    // (a reduce-scatter made of NVLink peer stores), the owner adds the P contributions in rank order
    const int*       blk_off;     // [npr+1] CSR over blocks of Pt*64 particles ...
    const int*       blk_ent;     // ... of (local patch index * 2 + side), side 0 = row, 1 = column
    float2*          peerF[LJMD_MAX_RANKS];   // every rank's receive buffer [P][Nloc]
    float2*          rowpart;     // [npatch][Pt*64] partial force on the patch's row (i) side
    float2*          colpart;     // [npatch][Pt*64] partial force on the patch's column (j) side
    float*           pe_part;     // [2*G] per-CTA partial potential energy (by step parity)
    float*           ke_part;     // [2*G]
    unsigned*        bar;
    int*             err;
    long long*       prof;        // optional [G][4] phase clocks (debug: LJMD_AP_PROF=1)
    long long        s_begin, s_end;   // steps [s_begin, s_end); s = -1 is the prologue force
    long long        spin_limit;       // clocks a spin wait may last (0 = unlimited)
    RunCtl           rc;
    float2*          R_out;
    float2*          V_out;
    float2*          F_out;
    float*           pe_out;
    // virial kernels (VIR): per-CTA / per-patch partial virial like pe_part, and the output: W of R_in
    // when nsteps == 0, else one float per ke_pe row
    float*           vir_part;    // [2*npe]
    float*           vir_out;
};

// ---- phase [b]: one segment = (i-block ib) x (j units [ju0, ju0+julen)) ---------------------
// Shared-memory tile layout: one float4 per j particle = (-xj, -xj, -yj, -yj): a single
// broadcast LDS.128 feeds the packed (two i per thread) pair evaluation.
template <int IPT, bool CUTOFF, bool PE, bool VIR>
__device__ __forceinline__ void ap_segment(const ApArgs& a, const float2* __restrict__ Rcur,
                                           int ib, int ju0, int julen, float4* sj,
                                           float (&fx)[IPT], float (&fy)[IPT], float& pe_acc,
                                           float& vir_acc) {
    constexpr int BI = AP_THREADS * IPT;
    const int tid = threadIdx.x;
    const PairConsts pc = a.pc;
    const PairConsts2 pc2 = make_pair_consts2(pc);
    float xi[IPT], yi[IPT];
    int   ii[IPT];
#pragma unroll
    for (int k = 0; k < IPT; ++k) {
        ii[k] = a.i_lo + ib * BI + k * AP_THREADS + tid;
        if (ii[k] < a.i_lo + a.Nloc) {
            const float* rp = reinterpret_cast<const float*>(Rcur + ii[k]);
            xi[k] = ldcg_f32(rp); yi[k] = ldcg_f32(rp + 1);
        } else { xi[k] = SENT_I; yi[k] = SENT_I; }
        fx[k] = 0.0f; fy[k] = 0.0f;
    }
    const int j0 = ju0 * J_UNIT, jend = (ju0 + julen) * J_UNIT;
    const int i_lo = a.i_lo + ib * BI, i_hi = i_lo + BI;

    for (int jt = j0; jt < jend; jt += TILE_J) {
        const int cnt = min(TILE_J, jend - jt);           // multiple of J_UNIT
        __syncthreads();                                   // previous tile fully consumed
        for (int q = tid; q < cnt; q += AP_THREADS) {
            const int j = jt + q;
            float2 r = (j < a.N) ? __ldcg(&Rcur[j]) : make_float2(SENT_J, SENT_J);
            sj[q] = make_float4(-r.x, -r.x, -r.y, -r.y);
        }
        __syncthreads();
        // the only j that can equal one of this CTA's i lie in [i_lo, i_hi): split the tile into
        // (before | diagonal | after) so the index test is paid on the overlap only
        const int qd0 = min(max(i_lo - jt, 0), cnt), qd1 = min(max(i_hi - jt, 0), cnt);
        if constexpr (IPT == 2) {
            const float2 xi2 = make_float2(xi[0], xi[1]), yi2 = make_float2(yi[0], yi[1]);
            float2 tfx = make_float2(0.0f, 0.0f), tfy = tfx, tpe = tfx, tvir = tfx;   // per-tile sums
#pragma unroll 1
            for (int part = 0; part < 3; ++part) {
                const int qa = (part == 0) ? 0 : (part == 1 ? qd0 : qd1);
                const int qb = (part == 0) ? qd0 : (part == 1 ? qd1 : cnt);
                if (part != 1) {
#pragma unroll AP_UNROLL
                    for (int q = qa; q < qb; ++q) {
                        const float4 v = sj[q];            // one j particle, warp broadcast
                        pair2_accum<CUTOFF, PE, false, VIR>(xi2, yi2, make_float2(v.x, v.y), make_float2(v.z, v.w),
                                                            true, true, pc, pc2, tfx, tfy, tpe, tvir);
                    }
                } else {
#pragma unroll AP_UNROLL
                    for (int q = qa; q < qb; ++q) {
                        const float4 v = sj[q];
                        const int j = jt + q;
                        pair2_accum<CUTOFF, PE, true, VIR>(xi2, yi2, make_float2(v.x, v.y), make_float2(v.z, v.w),
                                                           j != ii[0], j != ii[1], pc, pc2, tfx, tfy, tpe, tvir);
                    }
                }
            }
            fx[0] += tfx.x; fx[1] += tfx.y; fy[0] += tfy.x; fy[1] += tfy.y;
            if (PE) pe_acc += tpe.x + tpe.y;
            if (VIR) vir_acc += tvir.x + tvir.y;
        } else {
            float tfx = 0.0f, tfy = 0.0f, tpe = 0.0f, tvir = 0.0f;
#pragma unroll 1
            for (int part = 0; part < 3; ++part) {
                const int qa = (part == 0) ? 0 : (part == 1 ? qd0 : qd1);
                const int qb = (part == 0) ? qd0 : (part == 1 ? qd1 : cnt);
                if (part != 1) {
#pragma unroll AP_UNROLL
                    for (int q = qa; q < qb; ++q) {
                        const float4 v = sj[q];
                        pair_accum<CUTOFF, PE, false, VIR>(xi[0], yi[0], -v.x, -v.z, true, pc, tfx, tfy, tpe, tvir);
                    }
                } else {
#pragma unroll AP_UNROLL
                    for (int q = qa; q < qb; ++q) {
                        const float4 v = sj[q];
                        pair_accum<CUTOFF, PE, true, VIR>(xi[0], yi[0], -v.x, -v.z, (jt + q) != ii[0], pc, tfx, tfy, tpe,
                                                          tvir);
                    }
                }
            }
            fx[0] += tfx; fy[0] += tfy;
            if (PE) pe_acc += tpe;
            if (VIR) vir_acc += tvir;
        }
    }
}

// ---- Newton's-third-law tiles -------------------------------------------------------------------
// A tile is 64 i-particles (two per lane, packed) x 32 j-particles (one per lane).  The j particle
// and the force accumulated ON it travel around the warp by shuffle: after 32 steps every j has met
// every lane's two i and is back in its home lane, so each unordered pair is evaluated once and
// applied to both sides with no atomics and a fixed summation order.
constexpr int T3_BLK = 64;

__device__ __forceinline__ int tri_base(int pa, int npr) { return pa * npr - (pa * (pa - 1)) / 2; }

// Both halves of a 64 x 64 tile in ONE rotation loop: the two travelling j sets (h = 0: lanes' j, h = 1:
// j + 32) are independent dependency chains (evaluate -> accumulate the reaction -> four shuffles), so
// interleaving them doubles the instruction-level parallelism of a warp that shares its scheduler with
// only three others (107 registers: 4 CTAs of 4 warps per SM).  The reaction on a travelling j is
// accumulated as ONE scalar per component (the two i of this lane added in a fixed order); after 32
// rotations the travelling j and its accumulator are home again.
template <bool CUTOFF, bool PE, bool N3L, bool VIR>
__device__ __forceinline__ void tile_both(const PairConsts& pc, const PairConsts2& pc2, float2 xi2, float2 yi2,
                                          float xja, float yja, float xjb, float yjb,
                                          float2& fx2, float2& fy2, float2& pe2, float2& vir2,
                                          float& fjxa, float& fjya, float& fjxb, float& fjyb) {
    const int src = (threadIdx.x + 1) & 31;
    float aax = 0.0f, aay = 0.0f, abx = 0.0f, aby = 0.0f;
    float2 gx2 = make_float2(0.0f, 0.0f), gy2 = gx2;       // second accumulator pair (half b)
    {   // step 0 peeled: the only step at which j can be one of this lane's own i (diagonal tiles):
        // half a meets i0 (self0), half b meets i1 (self1)
        float2 fa, dxa, dya, fb, dxb, dyb;
        if (N3L) {
            pair2_eval<CUTOFF, PE, false, VIR>(xi2, yi2, make_float2(-xja, -xja), make_float2(-yja, -yja),
                                               true, true, pc, pc2, fa, dxa, dya, pe2, vir2);
            pair2_eval<CUTOFF, PE, false, VIR>(xi2, yi2, make_float2(-xjb, -xjb), make_float2(-yjb, -yjb),
                                               true, true, pc, pc2, fb, dxb, dyb, pe2, vir2);
        } else {
            pair2_eval<CUTOFF, PE, true, VIR>(xi2, yi2, make_float2(-xja, -xja), make_float2(-yja, -yja),
                                              false, true, pc, pc2, fa, dxa, dya, pe2, vir2);
            pair2_eval<CUTOFF, PE, true, VIR>(xi2, yi2, make_float2(-xjb, -xjb), make_float2(-yjb, -yjb),
                                              true, false, pc, pc2, fb, dxb, dyb, pe2, vir2);
        }
        fx2 = __ffma2_rn(fa, dxa, fx2); fy2 = __ffma2_rn(fa, dya, fy2);
        gx2 = __ffma2_rn(fb, dxb, gx2); gy2 = __ffma2_rn(fb, dyb, gy2);
        if (N3L) {
            aax = fmaf(fa.y, dxa.y, __fmul_rn(fa.x, dxa.x)); aay = fmaf(fa.y, dya.y, __fmul_rn(fa.x, dya.x));
            abx = fmaf(fb.y, dxb.y, __fmul_rn(fb.x, dxb.x)); aby = fmaf(fb.y, dyb.y, __fmul_rn(fb.x, dyb.x));
        }
        xja = __shfl_sync(0xffffffffu, xja, src); yja = __shfl_sync(0xffffffffu, yja, src);
        xjb = __shfl_sync(0xffffffffu, xjb, src); yjb = __shfl_sync(0xffffffffu, yjb, src);
        if (N3L) {
            aax = __shfl_sync(0xffffffffu, aax, src); aay = __shfl_sync(0xffffffffu, aay, src);
            abx = __shfl_sync(0xffffffffu, abx, src); aby = __shfl_sync(0xffffffffu, aby, src);
        }
    }
#pragma unroll AP_TB_UNROLL
    for (int s = 1; s < 32; ++s) {
        float2 fa, dxa, dya, fb, dxb, dyb;
        pair2_eval<CUTOFF, PE, false, VIR>(xi2, yi2, make_float2(-xja, -xja), make_float2(-yja, -yja),
                                           true, true, pc, pc2, fa, dxa, dya, pe2, vir2);
        pair2_eval<CUTOFF, PE, false, VIR>(xi2, yi2, make_float2(-xjb, -xjb), make_float2(-yjb, -yjb),
                                           true, true, pc, pc2, fb, dxb, dyb, pe2, vir2);
        fx2 = __ffma2_rn(fa, dxa, fx2); fy2 = __ffma2_rn(fa, dya, fy2);
        gx2 = __ffma2_rn(fb, dxb, gx2); gy2 = __ffma2_rn(fb, dyb, gy2);
        if (N3L) {
            aax = fmaf(fa.y, dxa.y, fmaf(fa.x, dxa.x, aax)); aay = fmaf(fa.y, dya.y, fmaf(fa.x, dya.x, aay));
            abx = fmaf(fb.y, dxb.y, fmaf(fb.x, dxb.x, abx)); aby = fmaf(fb.y, dyb.y, fmaf(fb.x, dyb.x, aby));
        }
        xja = __shfl_sync(0xffffffffu, xja, src); yja = __shfl_sync(0xffffffffu, yja, src);
        xjb = __shfl_sync(0xffffffffu, xjb, src); yjb = __shfl_sync(0xffffffffu, yjb, src);
        if (N3L) {
            aax = __shfl_sync(0xffffffffu, aax, src); aay = __shfl_sync(0xffffffffu, aay, src);
            abx = __shfl_sync(0xffffffffu, abx, src); aby = __shfl_sync(0xffffffffu, aby, src);
        }
    }
    fx2.x += gx2.x; fx2.y += gx2.y; fy2.x += gy2.x; fy2.y += gy2.y;
    fjxa = -aax; fjya = -aay; fjxb = -abx; fjyb = -aby;
}

__device__ __forceinline__ float2 ld_pos(const float2* __restrict__ R, int j, int N, float sent) {
    return (j < N) ? __ldcg(&R[j]) : make_float2(sent, sent);
}

template <bool CUTOFF, bool PE, bool VIR>
__device__ __forceinline__ void ap3_phase_forces(const ApArgs& a, const float2* __restrict__ Rcur,
                                                 float2* sacc /* 4 warps x 2 x q x 64 */, float* sred,
                                                 int par) {
    const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int wr = w >> 1, wc = w & 1, q = a.q, Pt = a.Pt;
    const PairConsts pc = a.pc;
    const PairConsts2 pc2 = make_pair_consts2(pc);
    float2* rowacc = sacc + (size_t)w * 2 * q * T3_BLK;        // this warp's [q][64] row-side sums
    float2* colacc = rowacc + (size_t)q * T3_BLK;              //             [q][64] column-side sums
    // CTA c takes patch c, then draws further patches from a per-step counter: rows of the triangle
    // differ in cost (diagonal patches, padding) and so do the SMs' shares of the L2; results and
    // partial sums are indexed by patch, so nothing depends on which CTA ran it.
    __shared__ int s_pi;
    for (int it = 0;; ++it) {
        if (tid == 0) s_pi = (it == 0) ? c : a.G + atomicAdd(&a.sched[par], 1);
        __syncthreads();
        const int pi = s_pi;
        if (pi >= a.npatch) break;
        float pe_thread = 0.0f, vir_thread = 0.0f;
        const int2 pp = a.patches[pi];
        // the partial vectors are indexed by position in the patch list (on one GPU the list is the whole
        // triangle in (pa, pb) order: that index is tri_base(pa) + pb - pa, which the reduction relies on)
        const int pid = pi;
        for (int k = lane; k < q * T3_BLK; k += 32) colacc[k] = make_float2(0.0f, 0.0f);
        __syncwarp();
        for (int r = 0; r < q; ++r) {
            const int ba = pp.x * Pt + wr * q + r;              // i block
            const int i0 = ba * T3_BLK + lane, i1 = i0 + 32;
            const float2 p0 = ld_pos(Rcur, i0, a.N, SENT_I), p1 = ld_pos(Rcur, i1, a.N, SENT_I);
            const float2 xi2 = make_float2(p0.x, p1.x), yi2 = make_float2(p0.y, p1.y);
            float2 fx2 = make_float2(0.0f, 0.0f), fy2 = fx2;
            for (int cc = 0; cc < q; ++cc) {
                const int bb = pp.y * Pt + wc * q + cc;         // j block
                if (ba > bb) continue;                          // lower triangle (diagonal patches only)
                float2 pe2 = make_float2(0.0f, 0.0f), vir2 = pe2;
                float2 tfx = make_float2(0.0f, 0.0f), tfy = tfx;   // per-tile sums (bounded chains)
                const int ja = bb * T3_BLK + lane, jb = ja + 32;
                const float2 pa = ld_pos(Rcur, ja, a.N, SENT_J), pb = ld_pos(Rcur, jb, a.N, SENT_J);
                float fjxa, fjya, fjxb, fjyb;
                if (ba < bb) {
                    tile_both<CUTOFF, PE, true, VIR>(pc, pc2, xi2, yi2, pa.x, pa.y, pb.x, pb.y, tfx, tfy, pe2, vir2,
                                                     fjxa, fjya, fjxb, fjyb);
                    float2 acc = colacc[cc * T3_BLK + lane];
                    acc.x += fjxa; acc.y += fjya;
                    colacc[cc * T3_BLK + lane] = acc;
                    acc = colacc[cc * T3_BLK + 32 + lane];
                    acc.x += fjxb; acc.y += fjyb;
                    colacc[cc * T3_BLK + 32 + lane] = acc;
                } else {
                    tile_both<CUTOFF, PE, false, VIR>(pc, pc2, xi2, yi2, pa.x, pa.y, pb.x, pb.y, tfx, tfy, pe2, vir2,
                                                      fjxa, fjya, fjxb, fjyb);
                }
                fx2.x += tfx.x; fx2.y += tfx.y; fy2.x += tfy.x; fy2.y += tfy.y;
                // energy bookkeeping in the ORDERED-pair convention of the caller (0.5 * sum):
                // an unordered pair of an off-diagonal tile counts twice, a diagonal tile is ordered
                if (PE) pe_thread += (ba < bb ? 2.0f : 1.0f) * (pe2.x + pe2.y);
                if (VIR) vir_thread += (ba < bb ? 2.0f : 1.0f) * (vir2.x + vir2.y);   // same weights
            }
            rowacc[r * T3_BLK + lane]      = make_float2(fx2.x, fy2.x);
            rowacc[r * T3_BLK + 32 + lane] = make_float2(fx2.y, fy2.y);
        }
        __syncthreads();
        // combine the two warps that share a patch row / column (fixed order) -> global partials
        float2* rp = a.rowpart + (size_t)pid * Pt * T3_BLK;
        float2* cp = a.colpart + (size_t)pid * Pt * T3_BLK;
        for (int k = tid; k < Pt * T3_BLK; k += AP_THREADS) {
            const int blk = k / T3_BLK, off = k - blk * T3_BLK;
            const int g2 = blk / q, rr = blk - g2 * q;          // warp-grid coordinate, tile within warp
            const float2* ra0 = sacc + (size_t)(g2 * 2 + 0) * 2 * q * T3_BLK + rr * T3_BLK + off;          // wr=g2, wc=0
            const float2* ra1 = sacc + (size_t)(g2 * 2 + 1) * 2 * q * T3_BLK + rr * T3_BLK + off;          // wr=g2, wc=1
            const float2* ca0 = sacc + (size_t)(0 * 2 + g2) * 2 * q * T3_BLK + (q + rr) * T3_BLK + off;    // wr=0, wc=g2
            const float2* ca1 = sacc + (size_t)(1 * 2 + g2) * 2 * q * T3_BLK + (q + rr) * T3_BLK + off;    // wr=1, wc=g2
            __stcg(&rp[k], make_float2(ra0->x + ra1->x, ra0->y + ra1->y));
            __stcg(&cp[k], make_float2(ca0->x + ca1->x, ca0->y + ca1->y));
        }
        if (PE) {                                    // per-patch energy partial (fixed reduction tree)
            float t = block_sum<AP_THREADS>(pe_thread, sred);
            if (tid == 0) __stcg(&a.pe_part[par * a.npe + pid], t);
        }
        if (VIR) {
            float t = block_sum<AP_THREADS>(vir_thread, sred);
            if (tid == 0) __stcg(&a.vir_part[par * a.npe + pid], t);
        }
        __syncthreads();
    }
}

template <int IPT, bool CUTOFF, bool PE, bool VIR>
__device__ __forceinline__ void ap_phase_forces(const ApArgs& a, const float2* __restrict__ Rcur,
                                                float4* sj, float* sred, int par) {
    constexpr int BI = AP_THREADS * IPT;
    const int c = blockIdx.x, tid = threadIdx.x;
    long long w = a.cta_start[c];
    const long long w1 = a.cta_start[c + 1];
    int seg = 0;
    float pe_thread = 0.0f, vir_thread = 0.0f;
    while (w < w1) {
        const int ib = (int)(w / a.NJu);
        const int ju0 = (int)(w - (long long)ib * a.NJu);
        const int len = (int)min((long long)(a.NJu - ju0), w1 - w);
        float fx[IPT], fy[IPT];
        ap_segment<IPT, CUTOFF, PE, VIR>(a, Rcur, ib, ju0, len, sj, fx, fy, pe_thread, vir_thread);
        float2* dst = a.part + ((size_t)c * a.maxseg + seg) * BI;
#pragma unroll
        for (int k = 0; k < IPT; ++k) __stcg(&dst[k * AP_THREADS + tid], make_float2(fx[k], fy[k]));
        w += len;
        ++seg;
    }
    if (PE) {
        float t = block_sum<AP_THREADS>(pe_thread, sred);
        if (tid == 0) __stcg(&a.pe_part[par * a.npe + c], t);
    }
    if (VIR) {
        float t = block_sum<AP_THREADS>(vir_thread, sred);
        if (tid == 0) __stcg(&a.vir_part[par * a.npe + c], t);
    }
}

// fixed-order sum of a per-CTA partial array by one warp, in double
__device__ __forceinline__ double warp_sum_array(const float* p, int n) {
    double s = 0.0;
    for (int k = threadIdx.x & 31; k < n; k += 32) s += (double)__ldcg(&p[k]);
    return warp_sum(s);
}

// VIR: the energy steps also accumulate the pair virial (a separate instantiation, launched only when the
// caller asked for it, so that the force-only kernels stay exactly as they are)
template <int IPT, bool CUTOFF, bool VIR>
__global__ void __launch_bounds__(AP_THREADS, AP_MINBLOCKS)
ap_persistent_kernel(const ApArgs a) {
    constexpr int BI = AP_THREADS * (IPT == 3 ? 1 : IPT);
    constexpr bool V3 = (IPT == 3);
    __shared__ float4 smem_buf[V3 ? 2048 : TILE_J];          // v2: j tile; v3: per-warp tile sums (32 KB)
    float4* sj = smem_buf;
    __shared__ float  sred[AP_THREADS / 32];
    __shared__ float  s_lambda;
    const int c = blockIdx.x, tid = threadIdx.x;
    const RunCtl rc = a.rc;
    unsigned epoch = 0;
    __shared__ long long pt[5];                              // debug phase clocks (thread 0 only)
    const bool prof = (a.prof != nullptr) && tid == 0;
    if (prof) { pt[0] = pt[1] = pt[2] = pt[3] = 0; }

    for (long long s = a.s_begin; s < a.s_end; ++s) {
        // (s = -1: the caller's positions, wrapped into the box by ap_load_kernel, are in Rbuf1)
        const float2* Rcur  = (s & 1) ? a.Rbuf1 : a.Rbuf0;
        float2*       Rnext = ((s + 1) & 1) ? a.Rbuf1 : a.Rbuf0;
        const StepFlags fl = step_flags<VIR>(rc, s, a.pe_out, a.vir_out);

        if (prof) pt[4] = clock64();
        // ---- [b] partial forces of R_cur ------------------------------------------------------
        if constexpr (V3) {
            if (c == 0 && tid == 0) __stcg(&a.sched[fl.par ^ 1], 0);   // the other parity's patch counter
            if (fl.want_pe) ap3_phase_forces<CUTOFF, true,  VIR  >(a, Rcur, reinterpret_cast<float2*>(smem_buf), sred, fl.par);
            else            ap3_phase_forces<CUTOFF, false, false>(a, Rcur, reinterpret_cast<float2*>(smem_buf), sred, fl.par);
        } else {
            if (fl.want_pe) ap_phase_forces<IPT, CUTOFF, true,  VIR  >(a, Rcur, sj, sred, fl.par);
            else            ap_phase_forces<IPT, CUTOFF, false, false>(a, Rcur, sj, sred, fl.par);
        }
        if (prof) { long long t = clock64(); pt[0] += t - pt[4]; pt[4] = t; }
        grid_barrier(a.bar, (++epoch) * (unsigned)a.G, a.err, a.spin_limit);
        if (prof) { long long t = clock64(); pt[1] += t - pt[4]; pt[4] = t; }
        // cross-GPU epochs of this step (tile mode on several GPUs uses two: partial forces, positions)
        const unsigned xper = (V3 && a.P > 1) ? 2u : 1u;
        const unsigned xe0 = a.xepoch0 + xper * (unsigned)(s - a.s_begin);
        auto peer_wait = [&](unsigned xe) {
            // every rank's peer stores of this phase have landed once all P arrival words carry the epoch
            if (c == 0 && tid < a.P && tid != a.rank) {
                __threadfence_system();
                volatile unsigned* f = a.peer_flags[tid] + a.rank;
                *f = xe;
            }
            if (tid < 32) {
                // lane q polls the word of rank q: the P - 1 words are in flight together (one round trip
                // to L2 when they have already landed, instead of P - 1 dependent ones)
                const bool other = (tid < a.P) && (tid != a.rank);
                const unsigned* word = a.peer_flags[a.rank] + (other ? tid : 0);
                const long long t0 = clock64();
                for (;;) {
                    bool done = true;
                    if (other) {
                        unsigned w;
                        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(w) : "l"(word) : "memory");
                        done = (int)(w - xe) >= 0;
                    }
                    if (__all_sync(0xffffffffu, done)) break;
                    const bool giveup = a.spin_limit > 0 && clock64() - t0 > 2 * a.spin_limit;
                    if (__any_sync(0xffffffffu, giveup)) { if (tid == 0) atomicExch(a.err, 2); break; }
                }
            }
            __syncthreads();
        };
        if constexpr (V3) {
            if (a.P > 1) {
                // ---- [c] this rank's partial force on EVERY particle -> the owner's receive buffer --------
                const int bsz = a.Pt * T3_BLK;
                const int grp_c = tid / RED_LANES, gl_c = tid % RED_LANES;
                for (int gb = c * (AP_THREADS / RED_LANES); gb < a.N; gb += a.G * (AP_THREADS / RED_LANES)) {
                    const int g = gb + grp_c;
                    const bool live = g < a.N;
                    float Fx = 0.0f, Fy = 0.0f;
                    if (live) {
                        const int blk = g / bsz;
                        const size_t off = (size_t)(g - blk * bsz);
                        const int e1 = a.blk_off[blk + 1];
                        // RED_BATCH entries of a lane are in flight together (entry -> partial vector is two
                        // dependent L2 round trips; one at a time this phase was 2/3 of the sharded step's
                        // overhead), added in the fixed entry order
                        for (int e0 = a.blk_off[blk] + gl_c; e0 < e1; e0 += RED_BATCH * RED_LANES) {
                            int ent[RED_BATCH];
                            float2 pv[RED_BATCH];
#pragma unroll
                            for (int u = 0; u < RED_BATCH; ++u) {
                                const int e = e0 + u * RED_LANES;
                                ent[u] = (e < e1) ? a.blk_ent[e] : -1;
                            }
#pragma unroll
                            for (int u = 0; u < RED_BATCH; ++u) {
                                const float2* base = (ent[u] & 1) ? a.colpart : a.rowpart;
                                pv[u] = (ent[u] >= 0) ? __ldcg(base + (size_t)(ent[u] >> 1) * bsz + off)
                                                      : make_float2(0.0f, 0.0f);
                            }
#pragma unroll
                            for (int u = 0; u < RED_BATCH; ++u) { Fx += pv[u].x; Fy += pv[u].y; }
                        }
                    }
#pragma unroll
                    for (int o = RED_LANES / 2; o > 0; o >>= 1) {
                        Fx += __shfl_xor_sync(0xffffffffu, Fx, o);
                        Fy += __shfl_xor_sync(0xffffffffu, Fy, o);
                    }
                    if (live && gl_c == 0) {
                        const int owner = g / a.Nloc;
                        a.peerF[owner][(size_t)a.rank * a.Nloc + (g - owner * a.Nloc)] = make_float2(Fx, Fy);
                    }
                }
                __threadfence_system();
                grid_barrier(a.bar, (++epoch) * (unsigned)a.G, a.err, a.spin_limit);
                peer_wait(xe0 + 1u);
            }
        }

        // ---- [d] reduce partials, finish the velocity-Verlet step -----------------------------
        // CTA c owns particles [c*ppc, (c+1)*ppc); a group of RED_LANES lanes sums the partials of
        // one particle (strided over the contributing CTAs, then a fixed xor-shuffle tree), and
        // lane 0 of the group integrates it.  Fixed order => bit-reproducible, no atomics.
        float ke_thread = 0.0f;
        const int grp = tid / RED_LANES, gl = tid % RED_LANES;
        const int g_end = min(a.Nloc, (c + 1) * a.ppc);                          // slab-local indices
        for (int gb = c * a.ppc; gb < g_end; gb += AP_THREADS / RED_LANES) {   // block-uniform trip count
            const int gloc = gb + grp;
            const int g = a.i_lo + gloc;                                       // global particle index
            const bool live = gloc < g_end;
            float Fx = 0.0f, Fy = 0.0f;
            float2 r = make_float2(0.0f, 0.0f), v = make_float2(0.0f, 0.0f);
            if (live && gl == 0) {                          // issued early: overlaps the partial loads
                r = __ldcg(&Rcur[g]);
                if (rc.nsteps > 0) v = a.Vh[g];
            }
            if (live) {
                if (V3 && a.P > 1) {
                    // the P ranks' partial forces on my particle (rank order, then the fixed shuffle tree)
                    for (int t = gl; t < a.P; t += RED_LANES) {
                        const float2 pv = __ldcg(&a.peerF[a.rank][(size_t)t * a.Nloc + gloc]);
                        Fx += pv.x; Fy += pv.y;
                    }
                } else if constexpr (V3) {
                    // row-side partials of patches (pr, pb >= pr), then column-side of (pa <= pr, pr)
                    const int blk = g / T3_BLK, pr = blk / a.Pt;
                    const size_t off = (size_t)(blk - pr * a.Pt) * T3_BLK + (g - blk * T3_BLK);
                    const size_t pstride = (size_t)a.Pt * T3_BLK;
                    const int n1 = a.npr - pr, ntot = n1 + pr + 1;
                    // all of a lane's partial vectors of a batch are in flight together (N = 4096: 33 vectors
                    // over 8 lanes = one L2 round trip instead of two), added in the fixed patch order
                    for (int t0 = gl; t0 < ntot; t0 += RED_BATCH * RED_LANES) {
                        float2 pb[RED_BATCH];
#pragma unroll
                        for (int u = 0; u < RED_BATCH; ++u) {
                            const int t = t0 + u * RED_LANES, pa = t - n1;
                            const float2* src = (t < n1) ? a.rowpart + (size_t)(tri_base(pr, a.npr) + t) * pstride
                                                         : a.colpart + (size_t)(tri_base(pa, a.npr) + (pr - pa)) * pstride;
                            pb[u] = (t < ntot) ? __ldcg(src + off) : make_float2(0.0f, 0.0f);
                        }
#pragma unroll
                        for (int u = 0; u < RED_BATCH; ++u) { Fx += pb[u].x; Fy += pb[u].y; }
                    }
                } else {
                    const int ib = gloc / BI, il = gloc - ib * BI;
                    const int2 cc = a.iblk_ctas[ib];
#pragma unroll 4
                    for (int c2 = cc.x + gl; c2 <= cc.y; c2 += RED_LANES) {
                        const int seg = ib - a.cta_ib0[c2];
                        const float2 p = __ldcg(&a.part[((size_t)c2 * a.maxseg + seg) * BI + il]);
                        Fx += p.x; Fy += p.y;
                    }
                }
            }
#pragma unroll
            for (int o = RED_LANES / 2; o > 0; o >>= 1) {
                Fx += __shfl_xor_sync(0xffffffffu, Fx, o);
                Fy += __shfl_xor_sync(0xffffffffu, Fy, o);
            }
            if (!live || gl != 0) continue;
            if (fl.kick1) { v.x = kick(v.x, Fx, a.dt); v.y = kick(v.y, Fy, a.dt); }   // MD:74
            if (fl.want_e || fl.thermo) ke_thread += v.x * v.x + v.y * v.y;
            if (fl.sample) rc.traj[(size_t)(s / rc.sample_every) * a.N + g] = r;
            if (fl.thermo) {                                // finish after the KE barrier
                a.Vh[g] = v;
                a.Ftmp[g] = make_float2(Fx, Fy);
                continue;
            }
            if (fl.final) {
                if (a.R_out) a.R_out[g] = r;
                if (a.V_out) a.V_out[g] = v;
                if (a.F_out) a.F_out[g] = make_float2(Fx, Fy);
            } else {
                v.x = kick(v.x, Fx, a.dt); v.y = kick(v.y, Fy, a.dt);                // MD:70
                a.Vh[g] = v;
                const float2 rn = make_float2(drift(r.x, v.x, a.dt, a.pc.box),      // MD:71-72
                                              drift(r.y, v.y, a.dt, a.pc.box));
                __stcg(&Rnext[g], rn);
                if (a.P > 1) {                               // position "all-gather": direct NVLink stores
                    const int nb = (int)((s + 1) & 1);
                    for (int q = 0; q < a.P; ++q)
                        if (q != a.rank) (nb ? a.peerR1[q] : a.peerR0[q])[g] = rn;
                }
            }
        }
        if (a.P > 1) __threadfence_system();                 // peer stores visible before the arrival
        if (fl.want_e || fl.thermo) {
            float t = block_sum<AP_THREADS>(ke_thread, sred);
            if (tid == 0) __stcg(&a.ke_part[fl.par * a.G + c], t);
        }
        if (fl.thermo) {
            // velocity rescale (single-GPU only)
            grid_barrier(a.bar, (++epoch) * (unsigned)a.G, a.err, a.spin_limit);
            if (tid < 32) {
                double ke2 = warp_sum_array(a.ke_part + fl.par * a.G, a.G);
                if (tid == 0) s_lambda = rescale_lambda(ke2, rc.thermo_kT, a.N);
            }
            __syncthreads();
            const float lam = s_lambda;
            for (int gloc = c * a.ppc + tid; gloc < g_end; gloc += AP_THREADS) {
                const int g = a.i_lo + gloc;
                const float2 r = __ldcg(&Rcur[g]);
                const float2 F = a.Ftmp[g];
                float2 v = a.Vh[g];
                v.x *= lam; v.y *= lam;
                if (fl.final) {
                    if (a.R_out) a.R_out[g] = r;
                    if (a.V_out) a.V_out[g] = v;
                    if (a.F_out) a.F_out[g] = F;
                } else {
                    v.x = kick(v.x, F.x, a.dt); v.y = kick(v.y, F.y, a.dt);
                    a.Vh[g] = v;
                    __stcg(&Rnext[g], make_float2(drift(r.x, v.x, a.dt, a.pc.box),
                                                  drift(r.y, v.y, a.dt, a.pc.box)));
                }
            }
        }
        if (prof) { long long t = clock64(); pt[2] += t - pt[4]; pt[4] = t; }
        grid_barrier(a.bar, (++epoch) * (unsigned)a.G, a.err, a.spin_limit);
        if (a.P > 1 && !fl.final) {
            // every rank has pushed its slab into our next-position buffer: one NVLink round trip per step,
            // no NCCL on the step path
            peer_wait(xe0 + xper);
        }
        if (prof) { long long t = clock64(); pt[3] += t - pt[4]; pt[4] = t; }

        // ---- energies of the post-step state (one warp, fixed order, double combine) ----------
        if (c == 0 && tid < 32 && fl.want_pe) {
            double pe2 = warp_sum_array(a.pe_part + fl.par * a.npe, a.npe);
            double ke2 = fl.want_e ? warp_sum_array(a.ke_part + fl.par * a.G, a.G) : 0.0;
            double w2 = VIR ? warp_sum_array(a.vir_part + fl.par * a.npe, a.npe) : 0.0;
            if (tid == 0) store_energy_row<VIR>(rc, fl, pe2, ke2, w2, a.pe_out, a.vir_out);
        }
    }
    if (prof) {
#pragma unroll
        for (int k = 0; k < 4; ++k) a.prof[c * 4 + k] = pt[k];
    }
}

// ---- small systems: ONE thread-block cluster, state resident in distributed shared memory --------
// At N <= ~1000 (config 1 is N = 400) a step holds so little work that the grid kernel above spends
// its time in two grid barriers and ~6 L2 round trips.  Here the whole system lives on chip:
//   * every CTA of the cluster keeps ALL positions in shared memory (ping-pong, as (-x,-x,-y,-y) so one
//     LDS.128 feeds the packed pair evaluation);
//   * CTA k owns particles [k*n_i, (k+1)*n_i).  A group of S lanes (S <= 32, one warp or part of one)
//     shares a PAIR of them: lane sl evaluates the pair against the j slice sl, an xor-butterfly of
//     shuffles leaves the bit-identical total force in all S lanes, and every lane finishes the
//     velocity-Verlet step of the pair redundantly with the velocities in REGISTERS for the whole call;
//   * lane sl then stores the new positions straight into the next-position buffer of CTA sl, sl+S, ...
//     of the cluster (st.shared::cluster: one warp instruction reaches up to 32 CTAs' worth of
//     destinations; a single thread pushing to 16 CTAs in turn measured ~190 clocks per store), and
//     ONE hardware cluster barrier (barrier.cluster arrive.release / wait.acquire) ends the step.
// No global memory traffic between samples, no L2 round trip, no __syncthreads on the step path.
constexpr int CLU_THREADS = 512;
constexpr int CLU_MAXC    = 16;

struct CluArgs {
    PairConsts pc;
    int   N, C, n_i, half, S, jl;       // half: particle pairs per CTA; S lanes per pair, slices of jl (odd) particles
    float dt, r2min;                    // r2min: see clu_pair2_f
    const float2* R_in;
    float2 *Rbuf0, *Rbuf1, *Vh;
    long long s_begin, s_end;
    RunCtl rc;
    float2 *R_out, *V_out, *F_out;
    float*  pe_out;
    long long* prof;                    // optional [C][4] phase clocks (debug: LJMD_AP_PROF=1)
    float*  vir_out;                    // virial kernel: W of R_in (nsteps == 0) or one float per ke_pe row
};

// The force-only slice loop is PREDICATE-FREE.  Inside the kernel the seven predicate registers are held
// by loop-invariant step flags; with the usual compare+select forms the compiler funnelled every compare
// of the four unrolled pair evaluations through the one or two registers left (measured: IPC 0.5).
//   * minimum image: d - m * copysign(box, d) with m = (|d| >= timg) as 1.0f / 0.0f (FSET.BF + FFMA, one
//     rounding: bit-identical to min_image());
//   * cutoff: ir2 *= (r2 < rc2) as 1.0f / 0.0f (FSET.BF + one packed FMUL2);
//   * the i == j term: r2 is clamped from below (FMNMX) at r2min, chosen on the host so that the force
//     scalar stays finite there; dx = dy = 0 then makes the term exactly 0, as the reference's
//     diagonal mask does (MD:54-55).  Distinct particles closer than sqrt(r2min) ~ 0.003 sigma overflow
//     fp32 in the reference itself.  The energy variant (rare steps) keeps the exact index test.
struct SliceSum { float2 fx, fy, pe; };
struct SliceSumVir { float2 fx, fy, pe, vir; };     // energy steps of the virial kernel

__device__ __forceinline__ float min_image_bf(float d, float box, float timg) {
    return fmaf(-set_ge_f32(fabsf(d), timg), copysignf(box, d), d);
}

template <bool CUTOFF>
__device__ __forceinline__ void clu_pair2_f(float2 xi2, float2 yi2, float4 q, float r2min, const PairConsts& c,
                                            const PairConsts2& c2, float2& fx2, float2& fy2) {
    float2 dx = __fadd2_rn(xi2, make_float2(q.x, q.y));
    float2 dy = __fadd2_rn(yi2, make_float2(q.z, q.w));
    dx.x = min_image_bf(dx.x, c.box, c.timg); dx.y = min_image_bf(dx.y, c.box, c.timg);
    dy.x = min_image_bf(dy.x, c.box, c.timg); dy.y = min_image_bf(dy.y, c.box, c.timg);
    float2 r2 = __ffma2_rn(__fmul2_rn(dx, dx), c2.one, __fmul2_rn(dy, dy));         // unfused sum
    r2.x = fmaxf(r2.x, r2min); r2.y = fmaxf(r2.y, r2min);
    float2 ir2 = make_float2(rcp_approx(r2.x), rcp_approx(r2.y));
    if (CUTOFF) {
        const float2 m = make_float2(set_lt_f32(r2.x, c.rc2), set_lt_f32(r2.y, c.rc2));
        ir2 = __fmul2_rn(ir2, m);
    }
    const float2 ir6 = __fmul2_rn(__fmul2_rn(ir2, ir2), ir2);
    const float2 f = __fmul2_rn(__ffma2_rn(ir6, c2.c12, c2.nc6), __fmul2_rn(ir6, ir2));
    fx2 = __ffma2_rn(f, dx, fx2);
    fy2 = __ffma2_rn(f, dy, fy2);
}

template <bool CUTOFF>
__device__ __forceinline__ SliceSum clu_slice_f(const float4* cur, int j0, int j1, float2 xi2, float2 yi2,
                                                float r2min, const PairConsts& pc) {
    const PairConsts2 pc2 = make_pair_consts2(pc);
    SliceSum r;
    r.fx = make_float2(0.0f, 0.0f); r.fy = r.fx; r.pe = r.fx;
#pragma unroll 4
    for (int j = j0; j < j1; ++j) clu_pair2_f<CUTOFF>(xi2, yi2, cur[j], r2min, pc, pc2, r.fx, r.fy);
    return r;
}

template <bool CUTOFF, bool VIR>
__device__ __noinline__ std::conditional_t<VIR, SliceSumVir, SliceSum>
clu_slice_pe(const float4* cur, int j0, int j1, int i0, int i1, float2 xi2, float2 yi2, PairConsts pc) {
    const PairConsts2 pc2 = make_pair_consts2(pc);
    std::conditional_t<VIR, SliceSumVir, SliceSum> r;
    r.fx = make_float2(0.0f, 0.0f); r.fy = r.fx; r.pe = r.fx;
    float2 vir = r.fx;
#pragma unroll 2
    for (int j = j0; j < j1; ++j) {
        const float4 q = cur[j];
        pair2_accum<CUTOFF, true, true, VIR>(xi2, yi2, make_float2(q.x, q.y), make_float2(q.z, q.w), j != i0,
                                             j != i1, pc, pc2, r.fx, r.fy, r.pe, vir);
    }
    if constexpr (VIR) r.vir = vir;
    return r;
}

// VIR: energy steps also sum the pair virial (own instantiation; its per-CTA partials follow sred)
template <bool CUTOFF, bool VIR>
__global__ void __launch_bounds__(CLU_THREADS, 1)
ap_cluster_kernel(const CluArgs a) {
    cg::cluster_group cluster = cg::this_cluster();
    const int k = (int)cluster.block_rank(), tid = threadIdx.x;
    extern __shared__ __align__(16) unsigned char clu_smem[];
    float4* spos = reinterpret_cast<float4*>(clu_smem);                // [2][N]
    float*  sE   = reinterpret_cast<float*>(spos + 2 * (size_t)a.N);   // [2 parity][pe, ke][CLU_MAXC] (CTA 0 sums)
    float*  sK   = sE + 4 * CLU_MAXC;                                  // [CLU_MAXC] thermostat kinetic partials
    float*  sred = sK + CLU_MAXC;                                      // [CLU_THREADS / 32]
    float*  sW   = sred + CLU_THREADS / 32;                            // VIR: [2 parity][CLU_MAXC] (CTA 0 sums)
    __shared__ float s_lambda;
    const RunCtl rc = a.rc;
    const PairConsts pc = a.pc;
    const int i_lo = min(a.N, k * a.n_i), i_hi = min(a.N, i_lo + a.n_i);
    const int sl = tid & (a.S - 1), p = tid / a.S;                     // j slice, pair of particles
    const int i0 = i_lo + p, i1 = i_lo + a.half + p;
    const bool has0 = (p < a.half) && i0 < i_hi, has1 = (p < a.half) && i1 < i_hi;
    const int j0 = min(a.N, sl * a.jl), j1 = min(a.N, j0 + a.jl);
    const bool lead = (sl == 0);                                       // writes the pair's global outputs
    float2 v0 = make_float2(0.0f, 0.0f), v1 = v0;                      // replicated in the S lanes of the pair
    if (rc.nsteps > 0) {
        if (has0) v0 = a.Vh[i0];
        if (has1) v1 = a.Vh[i1];
    }
    {
        const float2* Rsrc = (a.s_begin < 0) ? a.R_in : ((a.s_begin & 1) ? a.Rbuf1 : a.Rbuf0);
        for (int j = tid; j < a.N; j += CLU_THREADS) {
            float2 r = Rsrc[j];
            if (a.s_begin < 0) r = load_wrap(r, pc.box);
            spos[j] = make_float4(-r.x, -r.x, -r.y, -r.y);
        }
    }
    int b = 0;
    long long pt[4] = {0, 0, 0, 0}, tl = 0;
    const bool prof = a.prof != nullptr && tid == 0;
    cluster.sync();                       // every CTA of the cluster is resident before remote stores start

    for (long long s = a.s_begin; s < a.s_end; ++s) {
        const StepFlags fl = step_flags<VIR>(rc, s, a.pe_out, a.vir_out);
        const float4* cur = spos + (size_t)b * a.N;
        float4*       nxt = spos + (size_t)(b ^ 1) * a.N;
        if (prof) tl = clock64();

        // ---- forces on the pair from this lane's j slice, then the butterfly over the S lanes -------
        float4 c0 = make_float4(-SENT_I, -SENT_I, -SENT_I, -SENT_I), c1 = c0;
        if (has0) c0 = cur[i0];
        if (has1) c1 = cur[i1];
        const float2 xi2 = make_float2(-c0.x, -c1.x), yi2 = make_float2(-c0.z, -c1.z);
        SliceSum ss;
        float2 tvir = make_float2(0.0f, 0.0f);
        if constexpr (VIR) {
            if (fl.want_pe) {
                const SliceSumVir sv = clu_slice_pe<CUTOFF, true>(cur, j0, j1, i0, i1, xi2, yi2, pc);
                ss.fx = sv.fx; ss.fy = sv.fy; ss.pe = sv.pe; tvir = sv.vir;
            } else {
                ss = clu_slice_f<CUTOFF>(cur, j0, j1, xi2, yi2, a.r2min, pc);
            }
        } else {
            ss = fl.want_pe ? clu_slice_pe<CUTOFF, false>(cur, j0, j1, i0, i1, xi2, yi2, pc)
                         : clu_slice_f<CUTOFF>(cur, j0, j1, xi2, yi2, a.r2min, pc);
        }
        float2 tfx = ss.fx, tfy = ss.fy;
        const float2 tpe = ss.pe;
        for (int o = a.S >> 1; o > 0; o >>= 1) {          // commutative adds: all lanes end bit-identical
            tfx.x += __shfl_xor_sync(0xffffffffu, tfx.x, o);
            tfx.y += __shfl_xor_sync(0xffffffffu, tfx.y, o);
            tfy.x += __shfl_xor_sync(0xffffffffu, tfy.x, o);
            tfy.y += __shfl_xor_sync(0xffffffffu, tfy.y, o);
        }
        if (fl.want_pe) {                  // fixed tree: per-CTA potential energy -> CTA 0
            const float t = block_sum<CLU_THREADS>((has0 ? tpe.x : 0.0f) + (has1 ? tpe.y : 0.0f), sred);
            if (tid == 0) *cluster.map_shared_rank(&sE[(fl.par * 2 + 0) * CLU_MAXC + k], 0) = t;
        }
        if (VIR && fl.want_pe) {           // the virial partial takes the same route
            const float t = block_sum<CLU_THREADS>((has0 ? tvir.x : 0.0f) + (has1 ? tvir.y : 0.0f), sred);
            if (tid == 0) *cluster.map_shared_rank(&sW[fl.par * CLU_MAXC + k], 0) = t;
        }
        if (prof) { const long long t = clock64(); pt[0] += t - tl; tl = t; }

        // ---- finish the velocity-Verlet step of the pair (every lane of the group, redundantly) -------
        const float2 r0 = make_float2(-c0.x, -c0.z), r1 = make_float2(-c1.x, -c1.z);
        if (fl.kick1) {                                                                           // MD:74
            v0.x = kick(v0.x, tfx.x, a.dt); v0.y = kick(v0.y, tfy.x, a.dt);
            v1.x = kick(v1.x, tfx.y, a.dt); v1.y = kick(v1.y, tfy.y, a.dt);
        }
        if (fl.sample && lead) {                                                                  // MD:93-100
            float2* row = rc.traj + (size_t)(s / rc.sample_every) * a.N;
            if (has0) row[i0] = r0;
            if (has1) row[i1] = r1;
        }
        if (fl.want_e || fl.thermo) {
            float ke_thread = 0.0f;
            if (lead && has0) ke_thread += v0.x * v0.x + v0.y * v0.y;
            if (lead && has1) ke_thread += v1.x * v1.x + v1.y * v1.y;
            const float t = block_sum<CLU_THREADS>(ke_thread, sred);
            if (tid == 0) {
                if (fl.want_e) *cluster.map_shared_rank(&sE[(fl.par * 2 + 1) * CLU_MAXC + k], 0) = t;
                if (fl.thermo)
                    for (int q = 0; q < a.C; ++q) *cluster.map_shared_rank(&sK[k], q) = t;
            }
        }
        if (fl.thermo) {
            // velocity rescale; every CTA sums the same C partials
            cluster.sync();
            if (tid == 0) {
                double ke2 = 0.0;
                for (int q = 0; q < a.C; ++q) ke2 += (double)sK[q];
                s_lambda = rescale_lambda(ke2, rc.thermo_kT, a.N);
            }
            __syncthreads();
            const float lam = s_lambda;
            v0.x *= lam; v0.y *= lam; v1.x *= lam; v1.y *= lam;
        }
        if (fl.final) {
            if (lead && has0) {
                if (a.R_out) a.R_out[i0] = r0;
                if (a.V_out) a.V_out[i0] = v0;
                if (a.F_out) a.F_out[i0] = make_float2(tfx.x, tfy.x);
            }
            if (lead && has1) {
                if (a.R_out) a.R_out[i1] = r1;
                if (a.V_out) a.V_out[i1] = v1;
                if (a.F_out) a.F_out[i1] = make_float2(tfx.y, tfy.y);
            }
        } else {
            v0.x = kick(v0.x, tfx.x, a.dt); v0.y = kick(v0.y, tfy.x, a.dt);                       // MD:70
            v1.x = kick(v1.x, tfx.y, a.dt); v1.y = kick(v1.y, tfy.y, a.dt);
            const float2 n0 = make_float2(drift(r0.x, v0.x, a.dt, pc.box), drift(r0.y, v0.y, a.dt, pc.box));   // MD:71-72
            const float2 n1 = make_float2(drift(r1.x, v1.x, a.dt, pc.box), drift(r1.y, v1.y, a.dt, pc.box));
            const float4 q0 = make_float4(-n0.x, -n0.x, -n0.y, -n0.y), q1 = make_float4(-n1.x, -n1.x, -n1.y, -n1.y);
            for (int q = sl; q < a.C; q += a.S) {
                if (has0) *cluster.map_shared_rank(&nxt[i0], q) = q0;
                if (has1) *cluster.map_shared_rank(&nxt[i1], q) = q1;
            }
            if (s == a.s_end - 1 && lead) {      // the next launch of a long call resumes from global memory
                float2* Rg = ((s + 1) & 1) ? a.Rbuf1 : a.Rbuf0;
                if (has0) { Rg[i0] = n0; a.Vh[i0] = v0; }
                if (has1) { Rg[i1] = n1; a.Vh[i1] = v1; }
            }
        }
        if (prof) { const long long t = clock64(); pt[1] += t - tl; tl = t; }
        cluster.sync();                          // all next positions have landed in every CTA
        if (prof) { const long long t = clock64(); pt[2] += t - tl; tl = t; }
        b ^= 1;

        if (k == 0 && tid == 0 && fl.want_pe) {  // energies of the post-step state (fixed order, double)
            double pe2 = 0.0, ke2 = 0.0, w2 = 0.0;
            for (int q = 0; q < a.C; ++q) pe2 += (double)sE[(fl.par * 2 + 0) * CLU_MAXC + q];
            if (VIR)
                for (int q = 0; q < a.C; ++q) w2 += (double)sW[fl.par * CLU_MAXC + q];
            if (fl.want_e)
                for (int q = 0; q < a.C; ++q) ke2 += (double)sE[(fl.par * 2 + 1) * CLU_MAXC + q];
            store_energy_row<VIR>(rc, fl, pe2, ke2, w2, a.pe_out, a.vir_out);
        }
    }
    if (prof) {
#pragma unroll
        for (int q = 0; q < 4; ++q) a.prof[k * 4 + q] = pt[q];
    }
}

// the caller's positions -> Rbuf1 (the buffer step s = -1 reads), wrapped into [0, box] (ljmd.h)
__global__ void ap_load_kernel(const float2* __restrict__ R_in, float2* __restrict__ dst, int N, float box) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) dst[i] = load_wrap(R_in[i], box);
}

using CluKernel = void (*)(const CluArgs);

using ApKernel = void (*)(const ApArgs);

template <bool VIR>
ApKernel pick_kernel(int ipt, bool cutoff) {
    if (ipt == 3) return cutoff ? ap_persistent_kernel<3, true, VIR> : ap_persistent_kernel<3, false, VIR>;
    if (ipt == 1) return cutoff ? ap_persistent_kernel<1, true, VIR> : ap_persistent_kernel<1, false, VIR>;
    return cutoff ? ap_persistent_kernel<2, true, VIR> : ap_persistent_kernel<2, false, VIR>;
}

}  // namespace

// ----------------------------------------------------------------------------------------------
struct AllPairs {
    int ipt = 1, G = 0, NJu = 0, nI = 0, maxseg = 0;
    int Pt = 0, q = 0, npr = 0, npatch = 0, npe = 0;   // Newton's-third-law tile mode (ipt == 3)
    int* sched = nullptr;
    int2* d_patches = nullptr;
    int *d_blk_off = nullptr, *d_blk_ent = nullptr;     // tile mode on several GPUs: per-block partial lists
    float2* peerF[LJMD_MAX_RANKS] = {};                 //   and every rank's receive buffer
    float2 *rowpart = nullptr, *colpart = nullptr;
    long long* d_cta_start = nullptr;
    int*       d_cta_ib0 = nullptr;
    int2*      d_iblk = nullptr;
    float2 *Rbuf0 = nullptr, *Rbuf1 = nullptr, *Vh = nullptr, *Ftmp = nullptr, *part = nullptr;
    float *pe_part = nullptr, *ke_part = nullptr, *vir_part = nullptr;
    int i_lo = 0, Nloc = 0;
    void* shared = nullptr;             // one allocation (IPC-shareable): Rbuf0 | Rbuf1 | arrival words
    unsigned* xflags = nullptr;
    unsigned  xepoch = 0;
    float2*   peerR0[LJMD_MAX_RANKS] = {};
    float2*   peerR1[LJMD_MAX_RANKS] = {};
    unsigned* peer_flags[LJMD_MAX_RANKS] = {};
    unsigned* bar = nullptr;
    int* err = nullptr;
    long long* prof = nullptr;
    ApKernel kernel = nullptr;
    ApKernel kernel_vir = nullptr;      // the same kernel with the virial on energy steps (nullptr: it does not
                                        // fit the grid of `kernel`)
    // single-cluster kernel for small systems (nullptr: not used)
    CluKernel clu_kernel = nullptr;
    CluKernel clu_kernel_vir = nullptr;
    int cluC = 0, clu_n_i = 0, clu_half = 0, clu_S = 0, clu_jl = 0;
    size_t clu_smem = 0, clu_smem_vir = 0;
};

int ap_mode(ljmd_handle* h) { return h->ap ? (h->ap->clu_kernel ? 4 : h->ap->ipt) : 0; }

// Can the whole system run inside one thread-block cluster?  (16 CTAs needs the non-portable opt-in.)
static int clu_setup(ljmd_handle* h, AllPairs* ap) {
    const long long N = h->p.N;
    // measured crossover with the grid kernel (which can use all 148 SMs): N = 400: 3.7 vs 6.9 us/step,
    // N = 1024: 9.0 vs 6.6 us/step
    long long nmax = 640;
    if (const char* e = getenv("LJMD_AP_CLUSTER_NMAX")) nmax = atoll(e);
    if (std::max(1, h->nranks) != 1 || N > nmax || N > 4096) return 0;
    CluKernel kern = h->pc.cutoff != 0 ? ap_cluster_kernel<true, false> : ap_cluster_kernel<false, false>;
    CluKernel kern_vir = h->pc.cutoff != 0 ? ap_cluster_kernel<true, true> : ap_cluster_kernel<false, true>;
    const size_t smem = 32 * (size_t)N + sizeof(float) * (5 * CLU_MAXC + CLU_THREADS / 32);
    const size_t smem_vir = smem + sizeof(float) * 2 * CLU_MAXC;         // + the virial partials
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) { cudaGetLastError(); return 0; }
    int want = CLU_MAXC;
    if (const char* e = getenv("LJMD_AP_CLUSTER_SIZE")) want = std::max(1, std::min(CLU_MAXC, atoi(e)));
    for (int C = want; C >= 1; C >>= 1) {
        if (C > 8 && cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) { cudaGetLastError(); continue; }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(C); cfg.blockDim = dim3(CLU_THREADS); cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int nclusters = 0;
        if (cudaOccupancyMaxActiveClusters(&nclusters, kern, &cfg) != cudaSuccess || nclusters < 1) { cudaGetLastError(); continue; }
        ap->clu_kernel = kern; ap->cluC = C; ap->clu_smem = smem;
        {   // the virial variant runs with the same cluster (or not at all: ljmd_virial then reports it)
            cfg.dynamicSmemBytes = smem_vir;
            if (cudaFuncSetAttribute(kern_vir, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_vir) == cudaSuccess &&
                (C <= 8 || cudaFuncSetAttribute(kern_vir, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) &&
                cudaOccupancyMaxActiveClusters(&nclusters, kern_vir, &cfg) == cudaSuccess && nclusters >= 1) {
                ap->clu_kernel_vir = kern_vir; ap->clu_smem_vir = smem_vir;
            }
            cudaGetLastError();
        }
        ap->clu_n_i = (int)((N + C - 1) / C);
        ap->clu_half = (ap->clu_n_i + 1) / 2;
        if (ap->clu_half > CLU_THREADS) { ap->clu_kernel = ap->clu_kernel_vir = nullptr; return 0; }
        int S = 32;                                        // lanes per particle pair (one warp at most)
        while (S > 1 && ap->clu_half * S > CLU_THREADS) S >>= 1;
        while (S > 1 && (long long)S > N) S >>= 1;
        ap->clu_S = S;
        ap->clu_jl = (int)((N + S - 1) / S) | 1;           // odd slice length: conflict-free LDS.128 across lanes
        return 0;
    }
    return 0;
}

int ap_create(ljmd_handle* h) {
    AllPairs* ap = new AllPairs();
    h->ap = ap;
    const long long N = h->p.N;
    const int P = std::max(1, h->nranks);
    // ipt 1 / 2: ordered pairs, one / two i per thread (stream-K split, any rank count);
    // ipt 3: Newton's-third-law tiles (each unordered pair once); on several GPUs the patches are dealt to
    //        the ranks and the partial forces are reduce-scattered over NVLink
    ap->ipt = (N >= 2048) ? 3 : 1;
    if (P > 1 && N / P < 2048) ap->ipt = (N >= 2048) ? 2 : 1;     // too few patches per rank for the tile mode
    if (const char* e = getenv("LJMD_AP_IPT")) { const int v = atoi(e); if (v >= 1 && v <= 3 && (v != 3 || P == 1 || ap->ipt == 3)) ap->ipt = v; }
    const int BI = AP_THREADS * (ap->ipt == 3 ? 1 : ap->ipt);
    if (N % P != 0) { set_error("all-pairs atom decomposition needs N divisible by the rank count"); return LJMD_E_INVALID; }
    ap->Nloc = (int)(N / P);
    ap->i_lo = h->rank * ap->Nloc;
    ap->nI  = (ap->Nloc + BI - 1) / BI;             // i-blocks of THIS rank's slab
    ap->NJu = (int)((N + J_UNIT - 1) / J_UNIT);
    ap->kernel = pick_kernel<false>(ap->ipt, h->pc.cutoff != 0);
    if (!getenv("LJMD_AP_IPT")) clu_setup(h, ap);      // (forcing a grid-kernel variant disables the cluster path)

    int per_sm = 0;
    LJ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ap->kernel, AP_THREADS, 0));
    int want = 4;
    if (const char* e = getenv("LJMD_AP_CTAS_PER_SM")) want = std::max(1, atoi(e));
    per_sm = std::min(per_sm, want);
    if (per_sm < 1) { set_error("all-pairs kernel does not fit on an SM"); return LJMD_E_STATE; }
    {   // the virial variant must be co-resident on the same grid (its launch bounds make it so)
        ApKernel kv = pick_kernel<true>(ap->ipt, h->pc.cutoff != 0);
        int per_sm_vir = 0;
        LJ_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_vir, kv, AP_THREADS, 0));
        if (per_sm_vir >= per_sm) ap->kernel_vir = kv;
    }
    const long long W = (long long)ap->nI * ap->NJu;
    // at least ~64 j per thread per CTA so tiny systems do not pay for a wide barrier
    long long g_work = std::max<long long>(1, W / (64 / J_UNIT));
    ap->G = (int)std::min<long long>((long long)per_sm * h->num_sms, std::min(g_work, W));
    if (const char* e = getenv("LJMD_AP_GRID")) ap->G = std::max(1, std::min(atoi(e), ap->G));
    std::vector<int2> patches;
    std::vector<int> blk_off, blk_ent;
    if (ap->ipt == 3) {
        // upper-triangular patches of Pt x Pt tiles (tile = 64 x 64 particles); a CTA's 2 x 2 warps take
        // q x q tiles each (Pt = 2q).  A diagonal patch does half the work of an off-diagonal one but
        // takes the same time (its busiest warp has q*q tiles), so patches are dealt out evenly.
        const int blocks = (int)((N + T3_BLK - 1) / T3_BLK);
        const long long slots = (long long)per_sm * h->num_sms;
        int q = 8;
        for (; q > 1; q >>= 1) {
            const long long npr = (blocks + 2 * q - 1) / (2 * q);
            if (npr * (npr + 1) / 2 / P >= 4 * slots) break;      // enough patches (per rank) to balance
        }
        if (const char* e = getenv("LJMD_AP_Q")) q = std::max(1, std::min(8, atoi(e)));
        ap->q = q; ap->Pt = 2 * q;
        ap->npr = (blocks + ap->Pt - 1) / ap->Pt;
        // several GPUs: the triangle's patches are dealt to the ranks round-robin (diagonal patches, which
        // cost half, are spread evenly that way); a rank's partial vectors are indexed by its own list
        {
            long long k = 0;
            for (int pa = 0; pa < ap->npr; ++pa)
                for (int pb = pa; pb < ap->npr; ++pb, ++k)
                    if (k % P == h->rank) patches.push_back(make_int2(pa, pb));
        }
        if (P > 1) {
            blk_off.assign(ap->npr + 1, 0);
            for (size_t lp = 0; lp < patches.size(); ++lp) { blk_off[patches[lp].x + 1]++; blk_off[patches[lp].y + 1]++; }
            for (int b = 0; b < ap->npr; ++b) blk_off[b + 1] += blk_off[b];
            blk_ent.resize(blk_off[ap->npr]);
            std::vector<int> fill(blk_off.begin(), blk_off.end() - 1);
            for (size_t lp = 0; lp < patches.size(); ++lp) blk_ent[fill[patches[lp].x]++] = (int)lp * 2;        // row side
            for (size_t lp = 0; lp < patches.size(); ++lp) blk_ent[fill[patches[lp].y]++] = (int)lp * 2 + 1;    // column side
        }
        const long long npatch = (long long)patches.size();
        ap->npatch = (int)npatch;
        ap->G = (int)std::min<long long>(slots, npatch);
        if (const char* e = getenv("LJMD_AP_GRID")) ap->G = std::max(1, std::min(atoi(e), ap->G));
    }

    // stream-K split of the flattened (i-block, j-unit) space, by COST: a j unit that overlaps
    // its own i-block runs the index-tested loop (~16% more instructions), so it weighs more.
    const long long W_PLAIN = 100, W_DIAG = (ap->ipt == 2) ? 116 : 110;
    const int du = BI / J_UNIT;                       // diagonal units per row
    auto row_cost = [&](int b, long long u) {         // cost of units [0, u) of row b
        const long long d0 = std::min<long long>((long long)ap->i_lo / J_UNIT + (long long)b * du, ap->NJu);
        const long long d1 = std::min<long long>(d0 + du, ap->NJu);
        const long long nd = std::max<long long>(0, std::min(u, d1) - d0);
        return u * W_PLAIN + nd * (W_DIAG - W_PLAIN);
    };
    std::vector<long long> rowsum(ap->nI + 1, 0);
    for (int b = 0; b < ap->nI; ++b) rowsum[b + 1] = rowsum[b] + row_cost(b, ap->NJu);
    const long long total_cost = rowsum[ap->nI];
    std::vector<long long> start(ap->G + 1);
    {
        int b = 0;
        for (int c = 0; c <= ap->G; ++c) {
            const long long target = (long long)(((__int128)total_cost * c) / ap->G);
            while (b + 1 < ap->nI && rowsum[b + 1] <= target) ++b;
            long long lo = 0, hi = ap->NJu;          // smallest u with rowsum[b] + row_cost(b,u) >= target
            while (lo < hi) {
                const long long mid = (lo + hi) / 2;
                if (rowsum[b] + row_cost(b, mid) >= target) hi = mid; else lo = mid + 1;
            }
            start[c] = (long long)b * ap->NJu + lo;
        }
        start[0] = 0;
        start[ap->G] = W;
        for (int c = 1; c <= ap->G; ++c) start[c] = std::max(start[c], start[c - 1]);
    }
    std::vector<int> ib0(ap->G);
    int maxseg = 1;
    for (int c = 0; c < ap->G; ++c) {
        ib0[c] = (int)(start[c] / ap->NJu);
        int ibl = (int)((start[c + 1] - 1) / ap->NJu);
        maxseg = std::max(maxseg, ibl - ib0[c] + 1);
    }
    ap->maxseg = maxseg;
    std::vector<int2> iblk(ap->nI);
    {
        int c = 0;
        for (int b = 0; b < ap->nI; ++b) {
            const long long lo = (long long)b * ap->NJu, hi = lo + ap->NJu;
            while (start[c + 1] <= lo) ++c;
            int cl = c;
            while (cl + 1 < ap->G && start[cl + 1] < hi) ++cl;
            iblk[b] = make_int2(c, cl);
        }
    }
    LJ_CUDA(cudaMalloc(&ap->d_cta_start, sizeof(long long) * (ap->G + 1)));
    LJ_CUDA(cudaMalloc(&ap->d_cta_ib0, sizeof(int) * ap->G));
    LJ_CUDA(cudaMalloc(&ap->d_iblk, sizeof(int2) * ap->nI));
    LJ_CUDA(cudaMemcpy(ap->d_cta_start, start.data(), sizeof(long long) * (ap->G + 1), cudaMemcpyHostToDevice));
    LJ_CUDA(cudaMemcpy(ap->d_cta_ib0, ib0.data(), sizeof(int) * ap->G, cudaMemcpyHostToDevice));
    LJ_CUDA(cudaMemcpy(ap->d_iblk, iblk.data(), sizeof(int2) * ap->nI, cudaMemcpyHostToDevice));
    {   // one >= 2 MiB allocation so that its IPC handle maps exactly this region on the peers
        const size_t rb = (sizeof(float2) * (size_t)N + 255) / 256 * 256;
        size_t bytes = 2 * rb + 256 + rb;          // Rbuf0 | Rbuf1 | arrival words | receive buffer [P][Nloc]
        bytes = std::max<size_t>((bytes + (2u << 20) - 1) / (2u << 20) * (2u << 20), 4u << 20);
        LJ_CUDA(cudaMalloc(&ap->shared, bytes));
        LJ_CUDA(cudaMemset(ap->shared, 0, bytes));
        ap->Rbuf0 = reinterpret_cast<float2*>(ap->shared);
        ap->Rbuf1 = reinterpret_cast<float2*>(reinterpret_cast<char*>(ap->shared) + rb);
        ap->xflags = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(ap->shared) + 2 * rb);
        ap->peerR0[h->rank] = ap->Rbuf0; ap->peerR1[h->rank] = ap->Rbuf1; ap->peer_flags[h->rank] = ap->xflags;
        ap->peerF[h->rank] = reinterpret_cast<float2*>(reinterpret_cast<char*>(ap->shared) + 2 * rb + 256);
        if (P > 1) {
            void* peers[LJMD_MAX_RANKS];
            int r = dist_share(h, ap->shared, peers);
            if (r) return r;
            for (int q = 0; q < P; ++q) {
                char* base = reinterpret_cast<char*>(peers[q]);
                ap->peerR0[q] = reinterpret_cast<float2*>(base);
                ap->peerR1[q] = reinterpret_cast<float2*>(base + rb);
                ap->peer_flags[q] = reinterpret_cast<unsigned*>(base + 2 * rb);
                ap->peerF[q] = reinterpret_cast<float2*>(base + 2 * rb + 256);
            }
        }
    }
    LJ_CUDA(cudaMalloc(&ap->Vh, sizeof(float2) * N));
    LJ_CUDA(cudaMalloc(&ap->Ftmp, sizeof(float2) * N));
    LJ_CUDA(cudaMalloc(&ap->part, sizeof(float2) * (size_t)ap->G * ap->maxseg * BI));
    if (ap->ipt == 3) {
        const size_t np = patches.size(), ps = (size_t)ap->Pt * T3_BLK;
        LJ_CUDA(cudaMalloc(&ap->d_patches, sizeof(int2) * np));
        LJ_CUDA(cudaMemcpy(ap->d_patches, patches.data(), sizeof(int2) * np, cudaMemcpyHostToDevice));
        if (!blk_ent.empty()) {
            LJ_CUDA(cudaMalloc(&ap->d_blk_off, sizeof(int) * blk_off.size()));
            LJ_CUDA(cudaMalloc(&ap->d_blk_ent, sizeof(int) * blk_ent.size()));
            LJ_CUDA(cudaMemcpy(ap->d_blk_off, blk_off.data(), sizeof(int) * blk_off.size(), cudaMemcpyHostToDevice));
            LJ_CUDA(cudaMemcpy(ap->d_blk_ent, blk_ent.data(), sizeof(int) * blk_ent.size(), cudaMemcpyHostToDevice));
        }
        LJ_CUDA(cudaMalloc(&ap->rowpart, sizeof(float2) * np * ps));
        LJ_CUDA(cudaMalloc(&ap->colpart, sizeof(float2) * np * ps));
    }
    ap->npe = (ap->ipt == 3) ? (int)patches.size() : ap->G;
    LJ_CUDA(cudaMalloc(&ap->pe_part, sizeof(float) * 2 * ap->npe));
    LJ_CUDA(cudaMalloc(&ap->sched, sizeof(int) * 2));
    LJ_CUDA(cudaMalloc(&ap->ke_part, sizeof(float) * 2 * ap->G));
    LJ_CUDA(cudaMalloc(&ap->bar, sizeof(unsigned)));
    LJ_CUDA(cudaMalloc(&ap->err, sizeof(int)));
    LJ_CUDA(cudaMemset(ap->err, 0, sizeof(int)));
    if (getenv("LJMD_AP_PROF")) LJ_CUDA(cudaMalloc(&ap->prof, sizeof(long long) * 4 * std::max(ap->G, CLU_MAXC)));
    return 0;
}

void ap_destroy(ljmd_handle* h) {
    AllPairs* ap = h->ap;
    if (!ap) return;
    cudaFree(ap->d_cta_start); cudaFree(ap->d_cta_ib0); cudaFree(ap->d_iblk);
    cudaFree(ap->shared); cudaFree(ap->Vh); cudaFree(ap->Ftmp);
    cudaFree(ap->part); cudaFree(ap->pe_part); cudaFree(ap->ke_part); cudaFree(ap->vir_part);
    cudaFree(ap->d_patches); cudaFree(ap->d_blk_off); cudaFree(ap->d_blk_ent); cudaFree(ap->rowpart); cudaFree(ap->colpart);
    cudaFree(ap->sched);
    cudaFree(ap->bar); cudaFree(ap->err);
    delete ap;
    h->ap = nullptr;
}

int ap_run(ljmd_handle* h, const float2* R_in, const float2* V_in, float2* R_out, float2* V_out,
           float2* F_out, float* pe_out, const RunCtl& rc, float* vir_out) {
    AllPairs* ap = h->ap;
    const long long N = h->p.N;
    cudaStream_t st = h->stream;
    const bool vir = vir_out != nullptr;
    if (vir && (ap->clu_kernel ? ap->clu_kernel_vir == nullptr : ap->kernel_vir == nullptr)) {
        set_error("the all-pairs virial kernel does not fit the launch configuration of this handle");
        return LJMD_E_UNSUPPORTED;
    }
    // allocated on first use: a process that never asks for the virial places every buffer (the grid-barrier
    // word among them, whose L2 home shows in the barrier-bound step time) where it was before the virial existed
    if (vir && !ap->vir_part) LJ_CUDA(cudaMalloc(&ap->vir_part, sizeof(float) * 2 * ap->npe));
    if (rc.nsteps > 0) {
        LJ_CUDA(cudaMemcpyAsync(ap->Vh, V_in, sizeof(float2) * N, cudaMemcpyDeviceToDevice, st));
        if (rc.traj && rc.S > 0)
            LJ_CUDA(cudaMemsetAsync(rc.traj, 0, sizeof(float2) * N * rc.S, st));   // MD:89
    }
    LJ_CUDA(cudaMemsetAsync(ap->err, 0, sizeof(int), st));     // status of THIS call (ljmd_check)
    ApArgs a{};
    a.pc = h->pc;
    a.spin_limit = h->spin_limit;
    a.ppc = (ap->Nloc + ap->G - 1) / ap->G;
    a.i_lo = ap->i_lo; a.Nloc = ap->Nloc; a.rank = h->rank; a.P = std::max(1, h->nranks);
    for (int q = 0; q < LJMD_MAX_RANKS; ++q) { a.peerR0[q] = ap->peerR0[q]; a.peerR1[q] = ap->peerR1[q]; a.peer_flags[q] = ap->peer_flags[q]; a.peerF[q] = ap->peerF[q]; }
    a.blk_off = ap->d_blk_off; a.blk_ent = ap->d_blk_ent;
    if (a.P > 1 && rc.thermo_every > 0) { set_error("the rescale thermostat is single-GPU only"); return LJMD_E_UNSUPPORTED; }
    a.N = (int)N; a.G = ap->G; a.NJu = ap->NJu; a.nI = ap->nI; a.maxseg = ap->maxseg;
    a.dt = h->p.dt;
    a.cta_start = ap->d_cta_start; a.cta_ib0 = ap->d_cta_ib0; a.iblk_ctas = ap->d_iblk;
    a.R_in = R_in; a.Rbuf0 = ap->Rbuf0; a.Rbuf1 = ap->Rbuf1; a.Vh = ap->Vh; a.Ftmp = ap->Ftmp;
    a.part = ap->part; a.pe_part = ap->pe_part; a.ke_part = ap->ke_part;
    a.Pt = ap->Pt; a.q = ap->q; a.npr = ap->npr; a.npatch = ap->npatch; a.npe = ap->npe; a.sched = ap->sched;
    a.patches = ap->d_patches; a.rowpart = ap->rowpart; a.colpart = ap->colpart;
    a.bar = ap->bar; a.err = ap->err; a.prof = ap->prof;
    a.rc = rc;
    a.R_out = R_out; a.V_out = V_out; a.F_out = F_out; a.pe_out = pe_out;
    a.vir_part = ap->vir_part; a.vir_out = vir_out;

    // bound the duration of a single launch (~0.5 s at a conservative 2e11 pairs/s)
    const double est_step_s = (double)N * (double)N / 2.0e11 + 3.0e-6;
    long long chunk = (long long)std::max(1.0, 0.5 / est_step_s);
    if (const char* e = getenv("LJMD_AP_CHUNK")) chunk = std::max(1, atoi(e));

    if (h->timed) LJ_CUDA(cudaEventRecord(h->ev0, st));
    long long s = -1;
    const long long s_last = rc.nsteps;     // exclusive
    if (ap->clu_kernel) {
        CluArgs c{};
        c.pc = h->pc; c.N = (int)N; c.C = ap->cluC; c.n_i = ap->clu_n_i; c.half = ap->clu_half;
        c.S = ap->clu_S; c.jl = ap->clu_jl; c.dt = h->p.dt;
        c.r2min = 2.0f * powf(fabsf(h->pc.c12) / 3.0e38f, 1.0f / 7.0f);      // c12 / r2min^7 stays finite
        c.R_in = R_in; c.Rbuf0 = ap->Rbuf0; c.Rbuf1 = ap->Rbuf1; c.Vh = ap->Vh;
        c.rc = rc; c.R_out = R_out; c.V_out = V_out; c.F_out = F_out; c.pe_out = pe_out;
        c.prof = ap->prof;
        c.vir_out = vir_out;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(ap->cluC); cfg.blockDim = dim3(CLU_THREADS); cfg.stream = st;
        cfg.dynamicSmemBytes = vir ? ap->clu_smem_vir : ap->clu_smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = ap->cluC; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        while (s < s_last) {
            const long long e = std::min(s_last, s + chunk);
            c.s_begin = s; c.s_end = e;
            LJ_CUDA(cudaLaunchKernelEx(&cfg, vir ? ap->clu_kernel_vir : ap->clu_kernel, c));
            h->launches++;
            s = e;
        }
        if (h->timed) LJ_CUDA(cudaEventRecord(h->ev1, st));
        if (ap->prof) {
            LJ_CUDA(cudaStreamSynchronize(st));
            std::vector<long long> pv(4 * ap->cluC);
            LJ_CUDA(cudaMemcpy(pv.data(), ap->prof, sizeof(long long) * pv.size(), cudaMemcpyDeviceToHost));
            const double nst = (double)std::max<long long>(1, c.s_end - c.s_begin);
            const char* nm[3] = {"forces", "integrate+push", "cluster sync"};
            for (int q = 0; q < 3; ++q) {
                double mean = 0, mx = 0;
                for (int j = 0; j < ap->cluC; ++j) { mean += pv[j * 4 + q]; mx = std::max<double>(mx, (double)pv[j * 4 + q]); }
                fprintf(stderr, "[ljmd prof] %-12s mean %8.0f  max %8.0f clocks/step (cluster of %d)\n", nm[q],
                        mean / ap->cluC / nst, mx / nst, ap->cluC);
            }
        }
        return 0;
    }
    ap_load_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(R_in, ap->Rbuf1, (int)N, h->pc.box);
    LJ_CUDA(cudaGetLastError());
    h->launches++;
    while (s < s_last) {
        const long long e = std::min(s_last, s + chunk);
        a.s_begin = s; a.s_end = e;
        a.xepoch0 = ap->xepoch;
        if (a.P > 1) { int rb = dist_barrier(h); if (rb) return rb; }   // the ranks enter the kernel together
        LJ_CUDA(cudaMemsetAsync(ap->bar, 0, sizeof(unsigned), st));
        LJ_CUDA(cudaMemsetAsync(ap->sched, 0, sizeof(int) * 2, st));
        void* args[] = {(void*)&a};
        LJ_CUDA(cudaLaunchCooperativeKernel((void*)(vir ? ap->kernel_vir : ap->kernel), dim3(ap->G), dim3(AP_THREADS),
                                            args, 0, st));
        h->launches++;
        ap->xepoch += (unsigned)(e - s) * ((ap->ipt == 3 && a.P > 1) ? 2u : 1u);   // cross-GPU epochs per step
        s = e;
    }
    if (a.P > 1) {
        // replicated out: slabs of the final state -> every rank (NCCL, once per call, not per step)
        const size_t slab = sizeof(float2) * (size_t)ap->Nloc;
        int r = 0;
        if (R_out && (r = dist_allgather(h, R_out, slab))) return r;
        if (V_out && (r = dist_allgather(h, V_out, slab))) return r;
        if (F_out && (r = dist_allgather(h, F_out, slab))) return r;
        for (long long k = 0; rc.traj && k < rc.S; ++k)
            if ((r = dist_allgather(h, rc.traj + (size_t)k * N, slab))) return r;
        if (pe_out && (r = dist_allreduce_f32(h, pe_out, 1))) return r;
        if (rc.ke_pe && rc.energy_every > 0) {       // "energies use one NCCL all-reduce"
            const long long ne = (rc.nsteps + rc.energy_every - 1) / rc.energy_every;
            if ((r = dist_allreduce_f32(h, rc.ke_pe, (size_t)(2 * ne)))) return r;
        }
    }
    if (h->timed) LJ_CUDA(cudaEventRecord(h->ev1, st));
    if (ap->prof) {   // debug: mean / max clocks per phase per step of the last launch
        LJ_CUDA(cudaStreamSynchronize(st));
        std::vector<long long> pv(4 * ap->G);
        LJ_CUDA(cudaMemcpy(pv.data(), ap->prof, sizeof(long long) * pv.size(), cudaMemcpyDeviceToHost));
        const double nst = (double)std::max<long long>(1, a.s_end - a.s_begin);
        const char* nm[4] = {"forces", "barrierA", "integrate", "barrierB"};
        for (int k = 0; k < 4; ++k) {
            double mean = 0, mx = 0;
            for (int c = 0; c < ap->G; ++c) { mean += pv[c * 4 + k]; mx = std::max<double>(mx, (double)pv[c * 4 + k]); }
            fprintf(stderr, "[ljmd prof] %-10s mean %9.0f  max %9.0f clocks/step (G=%d)\n", nm[k],
                    mean / ap->G / nst, mx / nst, ap->G);
        }
        if (getenv("LJMD_AP_PROF_CTAS")) {
            fprintf(stderr, "[ljmd prof] forces clocks/step by CTA:");
            for (int c = 0; c < ap->G; ++c) fprintf(stderr, "%s%d:%.0f", (c % 16) ? " " : "\n  ", c, pv[c * 4] / nst);
            fprintf(stderr, "\n");
        }
    }
    return 0;
}

int ap_check_error(ljmd_handle* h) {
    AllPairs* ap = h->ap;
    if (!ap) return 0;
    int e = 0;
    LJ_CUDA(cudaMemcpy(&e, ap->err, sizeof(int), cudaMemcpyDeviceToHost));
    if (e) {
        set_error("all-pairs persistent kernel: %s timed out (LJMD_SPIN_TIMEOUT_S)",
                  e == 2 ? "a peer GPU's arrival word" : "a grid barrier");
        return LJMD_E_TIMEOUT;
    }
    return 0;
}

}  // namespace ljmd
