// sk.cu — density modes rho_k(s) = sum_j exp(i 2 pi (n_x x_j + n_y y_j) / box) of S snapshots for K integer
// wave vectors (ljmd_density_modes), the input of the static structure factor S(k) = <|rho_k|^2> / N.
//
// Phase in fixed point.  Each coordinate becomes once a 32-bit phase word q = rint(x / box * 2^32) mod 2^32
// (sk_phase_word); the phase of (particle, vector) is then the uint32 word w = n_x q_x + n_y q_y, exact modulo one
// revolution for any integer n, and its angle is (int32)w * 2 pi / 2^32 in (-pi, pi].  Coordinates outside
// [0, box] are therefore periodic for free.  A naive fp32 k.r at |n| in the thousands and x ~ 2000 sigma is off by
// ~1e-3 rad; here the quantisation is at most (|n_x| + |n_y|) 2^-33 revolutions.
//
// Accuracy.  Per term and per component (cos or sin), with u = 2^-24:
//   phase words       (|n_x| + |n_y|) pi 2^-32 rad     (rint of each coordinate: half a unit of 2^-32 rev; the
//                                                      double quotient adds |x / box| 2^-53 rev per coordinate,
//                                                      below 2^-43 rev for |x| <= 1024 box)
//   I2FP of w         pi 2^-25 rad                     (|w| <= 2^31: half an fp32 ulp of 2^7 units of 2^-32 rev)
//   * fl(2 pi 2^-32)  pi 2^-24 + 2^-23 rad              (the constant's relative error times |angle| <= pi, and
//                                                      the product's rounding, half an ulp below 4)
//   sin / cos         2^-20.5 absolute                 (sin.approx / cos.approx.f32, PTX ISA: over |a| <= 100 pi)
// so eps_term = (|n_x| + |n_y|) pi 2^-32 + pi (2^-25 + 2^-24) + 2^-23 + 2^-20.5
//             = (|n_x| + |n_y|) * 7.32e-10 + 1.074e-6.
// Sums: terms are added in fp32 over chunks of SK_CHUNK = 32 consecutive particles (error <= u C (C + 1) / 2 per
// chunk of C terms of magnitude <= 1, i.e. u (C + 1) / 2 = 16.5 u per particle), and the chunk sums and then
// the segment sums in double (at most N / 32 + 1024 additions of partials <= N).  Hence for each of Re and Im
//   |rho_k(GPU) - rho_k(exact)| <= N (eps_term + 16.5 u) + (N / 32 + 1024) N 2^-53.
// For random rounding the observed error is ~sqrt(N) eps (tests/test_sk_gpu.py reports it).
//
// Layout.  One thread per wave vector, SK_THREADS vectors per CTA (blockIdx.x); blockIdx.y is a segment of
// sk_segment_len(N) consecutive particles, blockIdx.z a snapshot of the batch.  A CTA stages SK_TILE phase-word
// pairs (8 B per particle) in shared memory, so every load in the pair loop is a broadcast.  Each thread adds
// its chunk sums in double in particle order and writes one (Re, Im) per segment to scratch; sk_reduce_kernel
// adds the segments of a (snapshot, vector) in segment order.  The segment length depends on N only, so rho_k
// of a (snapshot, vector) is the same bits whichever other snapshots and vectors share the call and however
// the call is batched.  A segment that holds a non-finite coordinate writes NaN, which the segment sum carries
// into every rho_k of that snapshot; other snapshots are untouched.
#include "ljmd_device.cuh"

#include <algorithm>

namespace ljmd {

struct Sk {
    void*  buf = nullptr;   // (snapshot, segment, vector) partial (Re, Im) in double, for one batch
    size_t bytes = 0;
};

namespace {

constexpr size_t SK_BATCH_BYTES = size_t(512) << 20;
constexpr int    SK_THREADS     = 256;       // wave vectors per CTA
constexpr int    SK_TILE        = 1024;      // particles staged per pass (8 KiB of phase words)
constexpr int    SK_CHUNK       = 32;        // fp32 partial sums over this many particles
constexpr int    SK_MAX_SEGS    = 1024;      // particle segments per snapshot, at most
constexpr int    SKR_THREADS    = 256;
// fl(2 pi * 2^-32): angle in radians of one unit of the phase word
constexpr float  SK_RAD_PER_UNIT = 1.46291807926715968e-09f;

// rint(x / box * 2^32) mod 2^32 in double for any finite x: the quotient and the 2^32 scaling as in the
// definition (the scaling is exact), the reduction exact (r - 2^32 floor(r 2^-32) is an integer in [0, 2^32)).
__device__ __forceinline__ unsigned sk_phase_word(float x, double box) {
    const double r = rint(__ddiv_rn((double)x, box) * 4294967296.0);
    return (unsigned)(r - 4294967296.0 * floor(r * 2.3283064365386963e-10));
}

__device__ __forceinline__ void sk_term(unsigned nx, unsigned ny, unsigned qx, unsigned qy, float& re, float& im) {
    const unsigned w = nx * qx + ny * qy;
    const float a = __fmul_rn(__int2float_rn((int)w), SK_RAD_PER_UNIT);
    float s, c;
    __sincosf(a, &s, &c);
    re = __fadd_rn(re, c);
    im = __fadd_rn(im, s);
}

__global__ void __launch_bounds__(SK_THREADS)
sk_modes_kernel(const float2* __restrict__ R, long long N, long long seg_len, double box,
                const int2* __restrict__ nvec, int K, double2* __restrict__ part) {
    __shared__ __align__(16) uint2 sq[SK_TILE];
    const int k = blockIdx.x * SK_THREADS + threadIdx.x;
    const int2 n = (k < K) ? nvec[k] : make_int2(0, 0);
    const unsigned nx = (unsigned)n.x, ny = (unsigned)n.y;
    const float2* Rs = R + (size_t)blockIdx.z * N;
    const long long j0 = (long long)blockIdx.y * seg_len, j1 = min(N, j0 + seg_len);
    double re = 0.0, im = 0.0;
    bool bad = false;
    for (long long t0 = j0; t0 < j1 && !bad; t0 += SK_TILE) {
        const int nt = (int)min((long long)SK_TILE, j1 - t0);
        __syncthreads();                                   // the previous tile has been read
        int nonfinite = 0;
        for (int i = threadIdx.x; i < nt; i += SK_THREADS) {
            const float2 r = Rs[t0 + i];
            const bool ok = isfinite(r.x) && isfinite(r.y);
            nonfinite |= !ok;
            sq[i] = ok ? make_uint2(sk_phase_word(r.x, box), sk_phase_word(r.y, box)) : make_uint2(0u, 0u);
        }
        bad = __syncthreads_or(nonfinite) != 0;
        if (bad) break;
        const uint4* sq4 = reinterpret_cast<const uint4*>(sq);
        for (int c0 = 0; c0 < nt; c0 += SK_CHUNK) {
            float cr = 0.0f, ci = 0.0f;
            if (c0 + SK_CHUNK <= nt) {
#pragma unroll
                for (int i = 0; i < SK_CHUNK; i += 2) {
                    const uint4 q = sq4[(c0 + i) >> 1];
                    sk_term(nx, ny, q.x, q.y, cr, ci);
                    sk_term(nx, ny, q.z, q.w, cr, ci);
                }
            } else {
                for (int i = c0; i < nt; ++i) sk_term(nx, ny, sq[i].x, sq[i].y, cr, ci);
            }
            re += (double)cr;
            im += (double)ci;
        }
    }
    if (k >= K) return;
    if (bad) re = im = __longlong_as_double(0x7ff8000000000000ll);
    part[((size_t)blockIdx.z * gridDim.y + blockIdx.y) * K + k] = make_double2(re, im);
}

// rho[s, k] = sum over the segments, in segment order, of the partials of (s, k)
__global__ void __launch_bounds__(SKR_THREADS)
sk_reduce_kernel(const double2* __restrict__ part, int nseg, int Kb, double2* __restrict__ rho, long long K) {
    const int k = blockIdx.x * SKR_THREADS + threadIdx.x;
    if (k >= Kb) return;
    const size_t s = blockIdx.y;
    const double2* p = part + s * nseg * (size_t)Kb + k;
    double re = 0.0, im = 0.0;
    for (int g = 0; g < nseg; ++g) {
        const double2 v = p[(size_t)g * Kb];
        re += v.x;
        im += v.y;
    }
    rho[s * K + k] = make_double2(re, im);
}

// Particles per segment: whole tiles, and at most SK_MAX_SEGS segments.  A function of N only.
long long sk_segment_len(long long N) {
    const long long tiles = (N + SK_TILE - 1) / SK_TILE;
    return (long long)SK_TILE * ((tiles + SK_MAX_SEGS - 1) / SK_MAX_SEGS);
}

}  // namespace

int sk_density_modes(ljmd_handle* h, const float2* R_hist, long long S, const int2* nvec, long long K,
                     double2* rho) {
    const long long N = h->p.N;
    cudaStream_t st = h->stream;
    const long long seg_len = sk_segment_len(N);
    const long long nseg = (N + seg_len - 1) / seg_len;
    const size_t per = sizeof(double2) * (size_t)nseg;                    // scratch per (snapshot, vector)
    // vectors per batch: all of them, or a multiple of SK_THREADS that fits (nseg <= 1024: >= 32768 fit)
    long long kb = std::min<long long>(K, (long long)(SK_BATCH_BYTES / per));
    if (kb < K) kb = std::max<long long>(SK_THREADS, kb / SK_THREADS * SK_THREADS);
    const long long sb = std::max<long long>(1, std::min<long long>(std::min<long long>(S, 65535),
                                                                    (long long)(SK_BATCH_BYTES / (per * kb))));
    const size_t need = per * (size_t)(kb * sb);
    if (!h->sk) h->sk = new Sk();
    Sk* g = h->sk;
    if (g->bytes < need) {
        LJ_CUDA(cudaFree(g->buf));
        g->buf = nullptr;
        g->bytes = 0;
        LJ_CUDA(cudaMalloc(&g->buf, need));
        g->bytes = need;
    }
    double2* part = reinterpret_cast<double2*>(g->buf);
    const double box = (double)h->p.box;
    for (long long k0 = 0; k0 < K; k0 += kb) {
        const int nk = (int)std::min(kb, K - k0);
        for (long long s0 = 0; s0 < S; s0 += sb) {
            const unsigned ns = (unsigned)std::min(sb, S - s0);
            sk_modes_kernel<<<dim3((unsigned)((nk + SK_THREADS - 1) / SK_THREADS), (unsigned)nseg, ns), SK_THREADS, 0,
                              st>>>(R_hist + (size_t)s0 * N, N, seg_len, box, nvec + k0, nk, part);
            LJ_CUDA(cudaGetLastError());
            sk_reduce_kernel<<<dim3((unsigned)((nk + SKR_THREADS - 1) / SKR_THREADS), ns), SKR_THREADS, 0, st>>>(
                part, (int)nseg, nk, rho + (size_t)s0 * K + k0, K);
            LJ_CUDA(cudaGetLastError());
            h->launches += 2;
        }
    }
    return 0;
}

void sk_destroy(ljmd_handle* h) {
    if (!h->sk) return;
    cudaFree(h->sk->buf);
    delete h->sk;
    h->sk = nullptr;
}

}  // namespace ljmd
