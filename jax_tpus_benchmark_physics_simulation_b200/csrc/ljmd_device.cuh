// ljmd_device.cuh — device-side building blocks shared by the all-pairs and cell-list kernels.
#pragma once
#include "ljmd_internal.cuh"

namespace ljmd {

constexpr float SENT_J = 1.0e18f;   // padding particles: far away, contribute exactly 0

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));   // MUFU.RCP, <= 1 ulp
    return r;
}

// compare results as 1.0f / 0.0f in a register (FSET.BF): predicate-free masks
__device__ __forceinline__ float set_ge_f32(float a, float b) {       // 1.0f if a >= b else 0.0f, in a register
    float m;
    asm("set.ge.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
    return m;
}
__device__ __forceinline__ float set_lt_f32(float a, float b) {
    float m;
    asm("set.lt.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
    return m;
}

// minimum image, bit-identical to  d - box * round(d / box)  of MD:46-48 for |d| <= box
// (see PairConsts::timg).  FSETP + LOP3 + predicated FADD.
__device__ __forceinline__ float min_image(float d, float box, float timg) {
    return (fabsf(d) >= timg) ? __fsub_rn(d, copysignf(box, d)) : d;
}

// Histogram bin of the pair distance r with numpy.histogram's semantics (get_histogram, MD:117-124):
// bin k holds e[k] <= r < e[k+1], the last bin is right-closed, r outside [lo, hi] gives -1.
// e: the nbins+1 fp32 edges (ascending); lo = e[0]; hi = e[nbins], or less to drop longer pairs;
// scale = nbins / (e[nbins] - lo).  The uniform guess is corrected against the fp32 edges, so the
// result does not depend on how the edges were rounded.  Used by every g(r) kernel.
__device__ __forceinline__ int gr_bin(float r, const float* e, int nbins, float lo, float hi, float scale) {
    if (!(r >= lo && r <= hi)) return -1;
    int b = (int)((r - lo) * scale);
    b = max(0, min(b, nbins - 1));
    while (b > 0 && r < e[b]) --b;
    while (b < nbins - 1 && r >= e[b + 1]) ++b;
    return b;
}

// Cell of a position in [0, box] on the periodic nc x nc grid of g(r) and the bond order (gr.cu, bond.cu): one
// fp32 multiply and truncation per axis.  The clamps keep any other input (outside [0, box], non-finite)
// inside the grid; such pairs are then dropped by the binning or counted as gr_hist_kernel (gr.cu) would
// count them, as long as they are adjacent.
__device__ __forceinline__ int gr_cell(float2 p, float inv_cell, int nc) {
    const int cx = min(max((int)__fmul_rn(p.x, inv_cell), 0), nc - 1);
    const int cy = min(max((int)__fmul_rn(p.y, inv_cell), 0), nc - 1);
    return cy * nc + cx;
}

// The full 9-cell stencil of ri's cell on that grid (one cell, every particle, when nc < 3), for the bond order and
// the cluster hook (bond.cu, cluster.cu): f(j, dx, dy, r, acc...) for every j in those cells (i itself included),
// j in cell order, with d = min_image(fl(x_j - x_i)) and r = fl(sqrt(fl(fl(dx^2) + fl(dy^2)))), the r that g(r)
// bins.  Ps: the snapshot's positions in cell order; cs: its cell starts.  The caller's per-thread accumulators
// travel as the reference arguments acc rather than as captures of f: so bond_order_kernel compiles to the same
// instructions as its hand-written loop did.
template <class F, class... A>
__device__ __forceinline__ void gr_stencil_walk(const float2* Ps, const int* cs, float2 ri, float inv_cell, int nc,
                                                float box, float timg, F f, A&... acc) {
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
                f(j, dx, dy, r, acc...);
            }
        }
    }
}

// (d / |d|)^m of a bond vector d in double, every operation rounded once: r = sqrt(dx^2 + dy^2), u = d / r, then
// m - 1 sequential complex products w <- w u = (ac - bd, ad + bc).  The psi_m of bond.cu and voronoi.cu agree
// because both take u^m from here.
__device__ __forceinline__ double2 unit_pow(double dx, double dy, int m) {
    const double r = __dsqrt_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)));
    const double ux = __ddiv_rn(dx, r), uy = __ddiv_rn(dy, r);
    double wx = ux, wy = uy;
    for (int k = 1; k < m; ++k) {
        const double a = wx, b = wy;
        wx = __dsub_rn(__dmul_rn(a, ux), __dmul_rn(b, uy));
        wy = __dadd_rn(__dmul_rn(a, uy), __dmul_rn(b, ux));
    }
    return make_double2(wx, wy);
}

// Weight of a pair in the g_m(r) histogram (ljmd_bond_corr): w = Re psi_i Re psi_j + Im psi_i Im psi_j, each
// operation rounded once, added as the integer llrint(w 2^24) (exact and order-free).  false: w is not
// finite and the pair is skipped.
__device__ __forceinline__ bool bond_pair_weight(double2 pi, double2 pj, long long& q) {
    const double w = __dadd_rn(__dmul_rn(pi.x, pj.x), __dmul_rn(pi.y, pj.y));
    if (!isfinite(w)) return false;
    q = llrint(__dmul_rn(w, 16777216.0));
    return true;
}

// One ordered pair (i <- j) of total_energy_fn / force_fn (MD:50-64):
//   r2 = dx^2 + dy^2 with each operation rounded once (no FMA contraction), so the pair set
//   {r2 < rc2} is decided on the same fp32 r2 as the CPU restatement;
//   ir2 = 1/r2 (MUFU.RCP); force scalar and pair energy in the sigma/epsilon-folded form.
// KEEPTEST: an additional "j is not i" predicate is applied (diagonal mask MD:54-55,60).
// VIR: also accumulate the pair virial r.f = t * ir6 (t = c12*ir6 - c6, the force's own factor)
// into vir, with the same pair set and ir2 as the force (see ljmd_virial in include/ljmd.h).
template <bool CUTOFF, bool PE, bool KEEPTEST, bool VIR>
__device__ __forceinline__ void pair_accum(float xi, float yi, float xj, float yj, bool keep,
                                           const PairConsts& c, float& fx, float& fy, float& pe,
                                           float& vir) {
    float dx = min_image(__fsub_rn(xi, xj), c.box, c.timg);
    float dy = min_image(__fsub_rn(yi, yj), c.box, c.timg);
    float r2 = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    float ir2 = rcp_approx(r2);
    if (CUTOFF) {
        const bool in = KEEPTEST ? (keep & (r2 < c.rc2)) : (r2 < c.rc2);   // one FSETP(.AND)
        ir2 = in ? ir2 : 0.0f;
    } else if (KEEPTEST) {
        ir2 = keep ? ir2 : 0.0f;
    }
    float ir6 = ir2 * ir2 * ir2;
    const float t = fmaf(ir6, c.c12, -c.c6);
    float f = t * (ir6 * ir2);
    fx = fmaf(f, dx, fx);
    fy = fmaf(f, dy, fy);
    if (PE) pe = fmaf(ir6, fmaf(ir6, c.d12, -c.d6), pe);
    if (VIR) vir = fmaf(t, ir6, vir);
}

// Two ordered pairs at once, (i0 <- j) and (i1 <- j), on Blackwell's packed-FP32 pipe
// (FADD2 / FMUL2 / FFMA2 on aligned register pairs): the same arithmetic as pair_accum, one
// issue slot per two pairs for every FMA-pipe operation.  The minimum image stays scalar
// (compare + sign-merge + predicated add on each half) so it remains bit-identical to the
// reference's div+round; r2 is still the unfused dx*dx + dy*dy.
//   nxj2 / nyj2 hold (-xj, -xj) / (-yj, -yj): xi + (-xj) == xi - xj exactly.
struct PairConsts2 {
    float2 c12, nc6, d12, nd6, one;
};
__device__ __forceinline__ PairConsts2 make_pair_consts2(const PairConsts& c) {
    PairConsts2 p;
    p.c12 = make_float2(c.c12, c.c12);
    p.nc6 = make_float2(-c.c6, -c.c6);
    p.d12 = make_float2(c.d12, c.d12);
    p.nd6 = make_float2(-c.d6, -c.d6);
    p.one = make_float2(c.one, c.one);
    return p;
}

// 32-bit L2 load that the compiler may not merge with its neighbour into a 64-bit load: the
// packed path wants (x_i0, x_i1) in one aligned register pair, not (x_i0, y_i0).
__device__ __forceinline__ float ldcg_f32(const float* p) {
    float v;
    asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}

// Pack two floats into ONE 64-bit register that stays live (volatile: ptxas may not
// rematerialise it with two MOVs per use, which it otherwise does for loop-invariant pairs).
__device__ __forceinline__ float2 pack_pinned(float lo, float hi) {
    unsigned long long r;
    asm volatile("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return *reinterpret_cast<float2*>(&r);
}

// Packed evaluation of the two pairs (i0 <- j), (i1 <- j) against ONE j (broadcast): returns the
// force scalars f2 and the displacements so that the caller can apply the term to BOTH sides
// (Newton's third law: f_ji = -f_ij bit for bit, because the min-image and r2 are symmetric).
template <bool CUTOFF, bool PE, bool KEEPTEST, bool VIR>
__device__ __forceinline__ void pair2_eval(float2 xi2, float2 yi2, float2 nxj2, float2 nyj2, bool keep0,
                                           bool keep1, const PairConsts& c, const PairConsts2& c2,
                                           float2& f, float2& dx, float2& dy, float2& pe2,
                                           float2& vir2) {
    dx = __fadd2_rn(xi2, nxj2);
    dy = __fadd2_rn(yi2, nyj2);
    dx.x = min_image(dx.x, c.box, c.timg);
    dx.y = min_image(dx.y, c.box, c.timg);
    dy.x = min_image(dy.x, c.box, c.timg);
    dy.y = min_image(dy.y, c.box, c.timg);
    // unfused dx*dx + dy*dy: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2, so the add is
    // written as fma(t, 1, u) with a run-time 1.0f (exact product, one rounding of the sum).
    const float2 r2 = __ffma2_rn(__fmul2_rn(dx, dx), c2.one, __fmul2_rn(dy, dy));
    float2 ir2 = make_float2(rcp_approx(r2.x), rcp_approx(r2.y));
    if (CUTOFF) {
        const bool in0 = KEEPTEST ? (keep0 & (r2.x < c.rc2)) : (r2.x < c.rc2);
        const bool in1 = KEEPTEST ? (keep1 & (r2.y < c.rc2)) : (r2.y < c.rc2);
        ir2.x = in0 ? ir2.x : 0.0f;
        ir2.y = in1 ? ir2.y : 0.0f;
    } else if (KEEPTEST) {
        ir2.x = keep0 ? ir2.x : 0.0f;
        ir2.y = keep1 ? ir2.y : 0.0f;
    }
    const float2 ir6 = __fmul2_rn(__fmul2_rn(ir2, ir2), ir2);
    const float2 t = __ffma2_rn(ir6, c2.c12, c2.nc6);
    f = __fmul2_rn(t, __fmul2_rn(ir6, ir2));
    if (PE) pe2 = __ffma2_rn(ir6, __ffma2_rn(ir6, c2.d12, c2.nd6), pe2);
    if (VIR) vir2 = __ffma2_rn(t, ir6, vir2);
}

// pair2_eval with the force on the two i accumulated
template <bool CUTOFF, bool PE, bool KEEPTEST, bool VIR>
__device__ __forceinline__ void pair2_accum(float2 xi2, float2 yi2, float2 nxj2, float2 nyj2,
                                            bool keep0, bool keep1, const PairConsts& c,
                                            const PairConsts2& c2, float2& fx2, float2& fy2,
                                            float2& pe2, float2& vir2) {
    float2 f, dx, dy;
    pair2_eval<CUTOFF, PE, KEEPTEST, VIR>(xi2, yi2, nxj2, nyj2, keep0, keep1, c, c2, f, dx, dy, pe2, vir2);
    fx2 = __ffma2_rn(f, dx, fx2);
    fy2 = __ffma2_rn(f, dy, fy2);
}

// jnp.mod(x, box) of MD:72 (result has the divisor's sign; can return exactly `box` for tiny
// negative x).  Fast exact paths for the ranges a step can produce, generic fmodf otherwise.
__device__ __forceinline__ float wrap_box(float x, float box) {
    if (x >= 0.0f && x < box) return x + 0.0f;                 // (+0.0f maps -0 to +0 like copysign(0, box))
    if (x >= box && x < 2.0f * box) return __fsub_rn(x, box);  // exact (fmod is exact)
    if (x < 0.0f && x > -box) return __fadd_rn(x, box);        // fmod(x) = x, then + box (one rounding)
    float m = fmodf(x, box);
    if (m != 0.0f) { if (m < 0.0f) m = __fadd_rn(m, box); } else m = 0.0f;
    return m;
}

// velocity-Verlet pieces with the reference's rounding sequence (MD:70-74):
//   V_half = V + (0.5*F)*dt      R_new = mod(R + V_half*dt, box)
__device__ __forceinline__ float kick(float v, float f, float dt) {
    return __fadd_rn(v, __fmul_rn(__fmul_rn(0.5f, f), dt));
}
__device__ __forceinline__ float drift(float r, float vh, float dt, float box) {
    return wrap_box(__fadd_rn(r, __fmul_rn(vh, dt)), box);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum (deterministic: fixed shuffle tree + fixed warp order); result valid in thread 0.
template <int THREADS>
__device__ __forceinline__ float block_sum(float v, float* smem /* THREADS/32 floats */) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) smem[w] = v;
    __syncthreads();
    float t = 0.0f;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < THREADS / 32; ++k) t += smem[k];
    }
    return t;
}

__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Grid-wide barrier for a cooperative (co-resident) launch: monotone arrival counter in L2.
// `target` = number of arrivals that completes this barrier (epoch * gridDim.x).
// A spin that lasts longer than `limit` clocks (LJMD_SPIN_TIMEOUT_S; 0 = never) raises *abort_flag and
// falls through, so a lost rank can never hang the GPU.  *abort_flag holds ONLY such aborts (the
// list / capacity flags live in another word): once it is set the run is void and later barriers fall
// through at once.
__device__ __forceinline__ void grid_barrier(unsigned* counter, unsigned target, int* abort_flag,
                                             long long limit) {
    __syncthreads();                       // every thread's writes are ordered before thread 0's release
    if (threadIdx.x == 0) {
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(counter) : "memory");
        if (__ldcg(abort_flag) == 0) {
            const long long t0 = clock64();
            while (ld_acquire_gpu(counter) < target) {
                if (limit > 0 && clock64() - t0 > limit) { atomicExch(abort_flag, 1); break; }
            }
        }
    }
    __syncthreads();                       // ... and the acquire is ordered before every thread's reads
}

// What step s of a persistent step kernel does (MD:77-106); s = -1 is the prologue force evaluation.
struct StepFlags {
    long long s;
    int  par;        // parity of the partial-sum buffers this step writes
    bool kick1, final, want_e, want_pe, thermo, sample;
};

// VIR: the virial instantiations also evaluate the energy terms for a one-shot ljmd_virial (nsteps == 0)
template <bool VIR>
__device__ __forceinline__ StepFlags step_flags(const RunCtl& rc, long long s, const float* pe_out,
                                                const float* vir_out) {
    StepFlags fl;
    fl.s      = s;
    fl.par    = (int)((s + 1) & 1);
    fl.kick1  = (s >= 0);                              // the prologue only evaluates F(R_in)
    fl.final  = (s == rc.nsteps - 1);
    fl.want_e = fl.kick1 && rc.energy_every > 0 && (s % rc.energy_every == 0);
    fl.want_pe = fl.want_e || (rc.nsteps == 0 && pe_out != nullptr);
    // (under if constexpr: a short-circuit || here reshuffles the force-only kernels' prologue)
    if constexpr (VIR) fl.want_pe = fl.want_pe || (rc.nsteps == 0 && vir_out != nullptr);
    fl.thermo = fl.kick1 && rc.thermo_every > 0 && rc.thermo_kT > 0.0f && ((s + 1) % rc.thermo_every == 0);
    fl.sample = fl.kick1 && rc.sample_every > 0 && (s % rc.sample_every == 0) &&
                (s / rc.sample_every < rc.S);         // MD:93-100
    return fl;
}

// The energies of an energy step from the kernel's fixed-order double sums over ordered pairs (pe2, and
// w2 with the same weights) and over |v|^2 (ke2): a row of ke_pe (+ vir_out), or the one-shot results.
template <bool VIR>
__device__ __forceinline__ void store_energy_row(const RunCtl& rc, const StepFlags& fl, double pe2, double ke2,
                                                 double w2, float* pe_out, float* vir_out) {
    if (fl.want_e) {
        float* o = rc.ke_pe + 2 * (fl.s / rc.energy_every);
        o[0] = (float)(0.5 * ke2);
        o[1] = (float)(0.5 * pe2);                     // MD:61  0.5 * sum over ordered pairs
        if (VIR) vir_out[fl.s / rc.energy_every] = (float)(0.5 * w2);
    } else {
        if (!VIR || pe_out) pe_out[0] = (float)(0.5 * pe2);
        if (VIR) vir_out[0] = (float)(0.5 * w2);
    }
}

// Thermostat velocity rescale V *= lambda = sqrt(kT_target / (KE/N)), KE = 0.5 * ke2 (SURVEY App. A);
// 1 when KE is 0 in fp32.
__device__ __forceinline__ float rescale_lambda(double ke2, float kT, long long N) {
    const float ke = (float)(0.5 * ke2);
    return ke > 0.0f ? sqrtf(kT / (ke / (float)N)) : 1.0f;
}

// A caller's position on its way into the library: coordinates inside the closed interval [0, box]
// (all a step can produce, MD:72) pass bit for bit, anything else is wrapped like jnp.mod.
__device__ __forceinline__ float2 load_wrap(float2 r, float box) {
    if (!(r.x >= 0.0f && r.x <= box)) r.x = wrap_box(r.x, box);
    if (!(r.y >= 0.0f && r.y <= box)) r.y = wrap_box(r.y, box);
    return r;
}

}  // namespace ljmd
