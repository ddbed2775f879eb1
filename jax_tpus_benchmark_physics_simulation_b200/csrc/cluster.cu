// cluster.cu — connected components ("clusters") of the link graph of every snapshot of S (ljmd_clusters), through
// the periodic cell grid of g(r) (gr.cu).
//
// Links.  Two distinct active particles i != j are linked when r_ij <= r_link, r_ij exactly the fp32 r that g(r)
// bins (min_image of __fsub_rn, __fmul_rn / __fadd_rn, __fsqrt_rn; gr_stencil_walk); coincident particles (r = 0)
// are linked.  Active: both coordinates finite and, with a mask, mask[s N + i] != 0.  A non-finite coordinate gives
// r = NaN or inf to everyone, so such a particle is linked to nobody either way.
//
// Forest.  The caller's labels (S, N) hold a union-find forest per snapshot: parent[x] for an active x, -1 for an
// inactive one (a -1 is written by the init launch only and never changes).  Invariant: parent[x] <= x at all
// times.  It holds after the init (parent[x] = x) and every write keeps it:
//   hook     CAS(parent[hi], hi, lo) with lo < hi, and only while hi is still a root (the CAS fails otherwise);
//   halving  parent[x] <- parent[parent[x]], a value <= parent[x] <= x, written only if parent[x] is unchanged.
// Every chain x -> parent[x] -> ... therefore strictly decreases until it ends at a root, so there are no cycles
// and the root of every tree is the smallest index in it.  A write replaces a parent by one of its ancestors or
// links one root under another, so an ancestor of x stays an ancestor of x for the rest of the launch, and a
// stale relaxed load of parent[y] still returns an ancestor of y: find(x) always returns the root of a tree
// that holds x at the time of its last load.
//
// Union.  unite(a, b) repeats: ra = find(a), rb = find(b); equal -> done; else CAS the larger root under the
// smaller, done if it was still a root.  A failed CAS means that root was hooked by another thread in between,
// which only merges trees, so the loop retries on the merged trees; it ends because each failure is caused by a
// successful hook, of which there are fewer than N.  When it returns, a and b are in one tree; trees are only ever
// merged, and only along links.  After every link has been united (the end of the hook launch), the trees are
// exactly the connected components, whatever the interleaving of the CAS operations.
//
// Labels.  The flatten launch starts after the hook launch has finished, so no root changes any more: find(i)
// returns the root of i's component, its smallest index, and labels[i] = find(i) is canonical.  Its own path
// halving only writes ancestors, so concurrent finds still end at the true root.  The output does not depend on
// the order of any atomic operation: it is bit-identical run to run, across batching and across handles.  sizes
// get atomicAdd(&sizes[root], 1), integer counts, equally order-free.
//
// Launch boundaries: init -> hook (every forest entry is initialised before any thread reads one), hook ->
// flatten (every union is complete before labels are read out as roots).  The grid's own launches come first.
//
// Every read and write of the forest during the hook and the flatten is a relaxed device-scope atomic
// (cuda::atomic_ref), never a plain cached load: another thread's hooks must become visible to a retry, and a
// load through the non-coherent path could keep returning the stale value.
//
// Layout: one thread per particle p in cell order, grid.y = snapshot in the batch, as bond_order_kernel.  Each
// thread walks the full 9-cell stencil of its cell (cells of edge >= r_link + the gr_grid_side margin) and unites
// only with candidates q > p in cell order, so every unordered pair is united once.  With fewer than 3 cells per
// side (r_link > box / 3) the grid is one cell and every thread visits all N particles.
#include "ljmd_device.cuh"

#include <cuda/atomic>

#include <algorithm>

namespace ljmd {

namespace {

constexpr int CL_THREADS = 256;

using Ref = cuda::atomic_ref<int, cuda::thread_scope_device>;

// root of x (parent[x] >= 0), halving the path on the way
__device__ __forceinline__ int uf_find(int* parent, int x) {
    while (true) {
        const int p = Ref(parent[x]).load(cuda::memory_order_relaxed);
        if (p == x) return x;
        const int g = Ref(parent[p]).load(cuda::memory_order_relaxed);
        if (g != p) {
            int e = p;
            Ref(parent[x]).compare_exchange_strong(e, g, cuda::memory_order_relaxed);
        }
        x = g;
    }
}

__device__ __forceinline__ void uf_unite(int* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        int hi = max(a, b);
        const int lo = min(a, b);
        if (Ref(parent[hi]).compare_exchange_strong(hi, lo, cuda::memory_order_relaxed)) return;
    }
}

// labels[s N + i] = i for an active particle, -1 otherwise (original order)
__global__ void __launch_bounds__(CL_THREADS)
cluster_init_kernel(const float2* __restrict__ R, const unsigned char* __restrict__ mask, int N,
                    int* __restrict__ labels) {
    const int i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= N) return;
    const size_t o = (size_t)blockIdx.y * N + i;
    const float2 r = R[o];
    const bool active = isfinite(r.x) && isfinite(r.y) && (!mask || mask[o] != 0);
    labels[o] = active ? i : -1;
}

__global__ void __launch_bounds__(CL_THREADS)
cluster_hook_kernel(const float2* __restrict__ P, const int* __restrict__ idx, const int* __restrict__ cstart,
                    long long stride, int N, int nc, float inv_cell, float box, float timg, float r_link,
                    int* labels) {
    const int p = blockIdx.x * CL_THREADS + threadIdx.x;
    if (p >= N) return;
    const size_t s = blockIdx.y;
    const float2* Ps = P + s * N;
    const int* ids = idx + s * N;
    int* parent = labels + s * N;
    const int a = ids[p];
    if (Ref(parent[a]).load(cuda::memory_order_relaxed) < 0) return;     // inactive
    gr_stencil_walk(Ps, cstart + s * stride, Ps[p], inv_cell, nc, box, timg,
                    [=](int q, float, float, float r) {
                        if (q <= p || !(r <= r_link)) return;               // each pair once; NaN r: no link
                        const int b = ids[q];
                        if (Ref(parent[b]).load(cuda::memory_order_relaxed) < 0) return;   // inactive neighbour
                        uf_unite(parent, a, b);
                    });
}

// labels[i] = root of i (its cluster's smallest index), sizes[root] += 1 (sizes may be null)
__global__ void __launch_bounds__(CL_THREADS)
cluster_flatten_kernel(int N, int* labels, int* __restrict__ sizes) {
    const int i = blockIdx.x * CL_THREADS + threadIdx.x;
    if (i >= N) return;
    const size_t s = blockIdx.y;
    int* parent = labels + s * N;
    if (Ref(parent[i]).load(cuda::memory_order_relaxed) < 0) return;
    const int root = uf_find(parent, i);
    Ref(parent[i]).store(root, cuda::memory_order_relaxed);
    if (sizes) atomicAdd(&sizes[s * N + root], 1);
}

}  // namespace

int clusters(ljmd_handle* h, const float2* R_hist, long long S, float r_link, const unsigned char* mask,
             int* labels, int* sizes) {
    const long long N = h->p.N;
    if (S == 0) return 0;
    if (sizes) LJ_CUDA(cudaMemsetAsync(sizes, 0, sizeof(int) * (size_t)S * N, h->stream));
    int nc = gr_grid_side(N, h->p.box, r_link);
    if (nc < 3) nc = 1;                                   // the 9-cell stencil needs 3 distinct cells per side
    GrGrid g;
    if (int e = gr_grid_alloc(h, S, nc, true, false, &g)) return e;
    const unsigned pblocks = (unsigned)((N + CL_THREADS - 1) / CL_THREADS);
    for (long long s0 = 0; s0 < S; s0 += g.nb) {
        const unsigned ns = (unsigned)std::min(g.nb, S - s0);
        const size_t off = (size_t)s0 * N;
        if (int e = gr_grid_bin(h, g, R_hist + off, nullptr, ns)) return e;
        cluster_init_kernel<<<dim3(pblocks, ns), CL_THREADS, 0, h->stream>>>(
            R_hist + off, mask ? mask + off : nullptr, (int)N, labels + off);
        LJ_CUDA(cudaGetLastError());
        cluster_hook_kernel<<<dim3(pblocks, ns), CL_THREADS, 0, h->stream>>>(
            g.P, g.idx, g.cs, g.stride, (int)N, nc, g.inv_cell, h->pc.box, h->pc.timg, r_link, labels + off);
        LJ_CUDA(cudaGetLastError());
        cluster_flatten_kernel<<<dim3(pblocks, ns), CL_THREADS, 0, h->stream>>>(
            (int)N, labels + off, sizes ? sizes + off : nullptr);
        LJ_CUDA(cudaGetLastError());
        h->launches += 3;
    }
    return 0;
}

}  // namespace ljmd
