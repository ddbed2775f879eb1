// api.cu — the exported C ABI (include/ljmd.h) over the all-pairs and cell-list engines.
#include "ljmd_internal.cuh"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>

namespace ljmd {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

PairConsts make_pair_consts(float box, float sigma, float eps, float rc) {
    PairConsts c{};
    c.box = box;
    // smallest fp32 t with fl(t / box) > 0.5  (see PairConsts in ljmd_internal.cuh)
    volatile float t = 0.5f * box;
    while ((float)(t / box) > 0.5f) t = nextafterf(t, 0.0f);
    while (!((float)(t / box) > 0.5f)) t = nextafterf(t, std::numeric_limits<float>::infinity());
    c.timg = t;
    const bool cut = std::isfinite(rc) && rc > 0.0f;
    c.cutoff = cut ? 1 : 0;
    c.rc2 = cut ? rc * rc : std::numeric_limits<float>::infinity();
    const float s2 = sigma * sigma, s6 = s2 * s2 * s2, s12 = s6 * s6;
    c.c12 = 48.0f * eps * s12;
    c.c6  = 24.0f * eps * s6;
    c.d12 = 4.0f * eps * s12;
    c.d6  = 4.0f * eps * s6;
    c.one = 1.0f;
    return c;
}

int create_common(ljmd_t** out, const ljmd_params* p, int rank, int nranks, const void* nccl_uid) {
    if (!out || !p) { set_error("null argument"); return LJMD_E_INVALID; }
    *out = nullptr;
    if (nranks < 1 || nranks > LJMD_MAX_RANKS || rank < 0 || rank >= nranks) { set_error("bad rank %d / nranks %d (max %d)", rank, nranks, LJMD_MAX_RANKS); return LJMD_E_INVALID; }
    if (nranks > 1 && !nccl_uid) { set_error("missing NCCL unique id"); return LJMD_E_INVALID; }
    if (p->N < 2 || p->N > (1ll << 30)) { set_error("N out of range: %lld", (long long)p->N); return LJMD_E_INVALID; }
    if (!(p->box > 0.0f) || !std::isfinite(p->box)) { set_error("box must be positive and finite"); return LJMD_E_INVALID; }
    if (!(p->sigma > 0.0f) || !(p->epsilon > 0.0f)) { set_error("sigma and epsilon must be positive"); return LJMD_E_INVALID; }
    if (!std::isfinite(p->dt)) { set_error("dt must be finite"); return LJMD_E_INVALID; }
    int ndev = 0;
    LJ_CUDA(cudaGetDeviceCount(&ndev));
    if (p->device < 0 || p->device >= ndev) { set_error("no CUDA device %d (found %d)", p->device, ndev); return LJMD_E_INVALID; }
    LJ_CUDA(cudaSetDevice(p->device));
    cudaDeviceProp prop;
    LJ_CUDA(cudaGetDeviceProperties(&prop, p->device));
    if (prop.major != 10) {
        set_error("ljmd is built for sm_100a (B200) only; device %d is sm_%d%d", p->device, prop.major, prop.minor);
        return LJMD_E_UNSUPPORTED;
    }
    ljmd_handle* h = new ljmd_handle();
    memset(h, 0, sizeof(*h));
    h->p = *p;
    if (!(h->p.skin > 0.0f)) h->p.skin = 0.3f * p->sigma;
    h->pc = make_pair_consts(p->box, p->sigma, p->epsilon, p->rc);
    h->stream = (cudaStream_t)p->stream;
    h->num_sms = prop.multiProcessorCount;
    h->rank = rank;
    h->nranks = nranks;
    h->timed = true;
    {   // device-side spin waits (grid barrier, cross-GPU arrival words) give up after this long
        double sec = 4.0;
        if (const char* e = getenv("LJMD_SPIN_TIMEOUT_S")) sec = atof(e);
        h->spin_limit = sec > 0.0 ? (long long)(sec * 1.0e3 * (double)prop.clockRate) : 0;
    }
    int path = p->path;
    if (path == LJMD_PATH_AUTO) path = (p->N <= 131072 || !h->pc.cutoff) ? LJMD_PATH_ALLPAIRS : LJMD_PATH_CELLS;
    if (path == LJMD_PATH_CELLS && !h->pc.cutoff) {
        set_error("the cell-list path needs a finite cutoff rc");
        delete h;
        return LJMD_E_INVALID;
    }
    if (path != LJMD_PATH_ALLPAIRS && path != LJMD_PATH_CELLS) { set_error("bad path %d", path); delete h; return LJMD_E_INVALID; }
    h->path = path;
    int rcode = 0;
    if ((rcode = (int)cudaEventCreate(&h->ev0)) || (rcode = (int)cudaEventCreate(&h->ev1))) {
        set_error("cudaEventCreate failed");
        delete h;
        return rcode;
    }
    if (nranks > 1) {
        rcode = dist_init(h, nccl_uid);
        if (rcode) { ljmd_destroy(h); return rcode; }
    }
    rcode = (path == LJMD_PATH_ALLPAIRS) ? ap_create(h) : cells_create(h);
    if (rcode) { ljmd_destroy(h); return rcode; }
    *out = h;
    return 0;
}

}  // namespace ljmd

using namespace ljmd;

extern "C" {

int ljmd_abi_version(void) { return LJMD_ABI_VERSION; }
const char* ljmd_last_error(void) { return g_err; }

int ljmd_create(ljmd_t** out, const ljmd_params* p) { return create_common(out, p, 0, 1, nullptr); }

void ljmd_destroy(ljmd_t* h) {
    if (!h) return;
    cudaSetDevice(h->p.device);
    cudaStreamSynchronize(h->stream);
    ap_destroy(h);
    cells_destroy(h);
    dist_destroy(h);
    gr_destroy(h);
    sk_destroy(h);
    for (int k = 0; k < 4; ++k) cudaFree(h->blk_full[k]);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    delete h;
}

static int run_dispatch(ljmd_t* h, const float* R_in, const float* V_in, float* R_out, float* V_out,
                        float* F_out, float* pe_out, const RunCtl& rc, float* w_out = nullptr) {
    LJ_CUDA(cudaSetDevice(h->p.device));
    const float2* R = reinterpret_cast<const float2*>(R_in);
    const float2* V = reinterpret_cast<const float2*>(V_in);
    if (h->path == LJMD_PATH_ALLPAIRS)
        return ap_run(h, R, V, reinterpret_cast<float2*>(R_out), reinterpret_cast<float2*>(V_out),
                      reinterpret_cast<float2*>(F_out), pe_out, rc, w_out);
    return cells_run(h, R, V, reinterpret_cast<float2*>(R_out), reinterpret_cast<float2*>(V_out),
                     reinterpret_cast<float2*>(F_out), pe_out, rc, w_out);
}

int ljmd_energy(ljmd_t* h, const float* R, float* pe_dev) {
    if (!h || !R || !pe_dev) { set_error("null argument"); return LJMD_E_INVALID; }
    RunCtl rc{};
    return run_dispatch(h, R, nullptr, nullptr, nullptr, nullptr, pe_dev, rc);
}

int ljmd_forces(ljmd_t* h, const float* R, float* F, float* pe_dev) {
    if (!h || !R || !F) { set_error("null argument"); return LJMD_E_INVALID; }
    RunCtl rc{};
    return run_dispatch(h, R, nullptr, nullptr, nullptr, F, pe_dev, rc);
}

int ljmd_virial(ljmd_t* h, const float* R, float* w_dev) {
    if (!h || !R || !w_dev) { set_error("null argument"); return LJMD_E_INVALID; }
    if (h->nranks > 1) { set_error("ljmd_virial: single-GPU handles only"); return LJMD_E_UNSUPPORTED; }
    RunCtl rc{};
    return run_dispatch(h, R, nullptr, nullptr, nullptr, nullptr, nullptr, rc, w_dev);
}

int ljmd_run(ljmd_t* h, const float* R_in, const float* V_in, float* R_out, float* V_out,
             int64_t nsteps, int64_t sample_every, float* traj, int64_t energy_every, float* ke_pe,
             float thermostat_kT, int64_t thermostat_every) {
    return ljmd_run_virial(h, R_in, V_in, R_out, V_out, nsteps, sample_every, traj, energy_every, ke_pe,
                           thermostat_kT, thermostat_every, nullptr);
}

int ljmd_run_virial(ljmd_t* h, const float* R_in, const float* V_in, float* R_out, float* V_out,
                    int64_t nsteps, int64_t sample_every, float* traj, int64_t energy_every, float* ke_pe,
                    float thermostat_kT, int64_t thermostat_every, float* w) {
    if (!h || !R_in || !V_in || !R_out || !V_out) { set_error("null argument"); return LJMD_E_INVALID; }
    if (nsteps < 0 || sample_every < 0 || energy_every < 0 || thermostat_every < 0) {
        set_error("negative step count");
        return LJMD_E_INVALID;
    }
    if (w && !(ke_pe && energy_every > 0)) {
        set_error("ljmd_run_virial: the virial trace w needs ke_pe and energy_every > 0 (it has their rows)");
        return LJMD_E_INVALID;
    }
    if (w && h->nranks > 1) { set_error("ljmd_run_virial: single-GPU handles only"); return LJMD_E_UNSUPPORTED; }
    const size_t bytes = sizeof(float) * 2 * (size_t)h->p.N;
    if (nsteps == 0) {   // fori_loop(0, 0, ...) returns the initial state (MD:82)
        LJ_CUDA(cudaSetDevice(h->p.device));
        if (R_out != R_in) LJ_CUDA(cudaMemcpyAsync(R_out, R_in, bytes, cudaMemcpyDeviceToDevice, h->stream));
        if (V_out != V_in) LJ_CUDA(cudaMemcpyAsync(V_out, V_in, bytes, cudaMemcpyDeviceToDevice, h->stream));
        return 0;
    }
    RunCtl rc{};
    rc.nsteps = nsteps;
    rc.sample_every = (traj && sample_every > 0) ? sample_every : 0;
    rc.S = rc.sample_every ? nsteps / rc.sample_every : 0;
    if (rc.S == 0) rc.sample_every = 0;
    rc.traj = reinterpret_cast<float2*>(traj);
    rc.energy_every = (ke_pe && energy_every > 0) ? energy_every : 0;
    rc.ke_pe = ke_pe;
    rc.thermo_kT = (thermostat_kT > 0.0f && thermostat_every > 0) ? thermostat_kT : 0.0f;
    rc.thermo_every = rc.thermo_kT > 0.0f ? thermostat_every : 0;
    return run_dispatch(h, R_in, V_in, R_out, V_out, nullptr, nullptr, rc, w);
}

int ljmd_run_blocked(ljmd_t* h, const float* R_blk, const float* V_blk, float* R_blk_out, float* V_blk_out,
                     int64_t nsteps, int64_t energy_every, float* ke_pe) {
    if (!h || !R_blk || !V_blk || !R_blk_out || !V_blk_out) { set_error("null argument"); return LJMD_E_INVALID; }
    if (nsteps < 1 || energy_every < 0) { set_error("ljmd_run_blocked: nsteps >= 1"); return LJMD_E_INVALID; }
    if (h->nranks == 1)      // one rank: its block is everything
        return ljmd_run(h, R_blk, V_blk, R_blk_out, V_blk_out, nsteps, 0, nullptr, energy_every, ke_pe, 0.0f, 0);
    const long long N = h->p.N;
    if (N % h->nranks != 0) { set_error("block-distributed I/O needs N divisible by the GPU count"); return LJMD_E_INVALID; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    RunCtl rc{};
    rc.nsteps = nsteps;
    rc.energy_every = (ke_pe && energy_every > 0) ? energy_every : 0;
    rc.ke_pe = ke_pe;
    rc.blocked = 1;
    const float2* R = reinterpret_cast<const float2*>(R_blk);
    const float2* V = reinterpret_cast<const float2*>(V_blk);
    if (h->path != LJMD_PATH_ALLPAIRS)
        return cells_run(h, R, V, reinterpret_cast<float2*>(R_blk_out), reinterpret_cast<float2*>(V_blk_out),
                         nullptr, nullptr, rc, nullptr);
    // all-pairs: the state is at most 1 MiB, so the blocks are simply all-gathered (NCCL over NVLink), the
    // replicated run is used as it is, and the rank's block is sliced out of its result
    const size_t blk = sizeof(float2) * (size_t)(N / h->nranks);
    for (int k = 0; k < 4; ++k)
        if (!h->blk_full[k]) LJ_CUDA(cudaMalloc(&h->blk_full[k], sizeof(float2) * (size_t)N));
    int r = dist_allgather_from(h, R, h->blk_full[0], blk);
    if (!r) r = dist_allgather_from(h, V, h->blk_full[1], blk);
    if (r) return r;
    rc.blocked = 0;
    r = ap_run(h, h->blk_full[0], h->blk_full[1], h->blk_full[2], h->blk_full[3], nullptr, nullptr, rc, nullptr);
    if (r) return r;
    LJ_CUDA(cudaMemcpyAsync(R_blk_out, reinterpret_cast<char*>(h->blk_full[2]) + blk * h->rank, blk, cudaMemcpyDeviceToDevice, h->stream));
    LJ_CUDA(cudaMemcpyAsync(V_blk_out, reinterpret_cast<char*>(h->blk_full[3]) + blk * h->rank, blk, cudaMemcpyDeviceToDevice, h->stream));
    return 0;
}

int ljmd_gr_hist(ljmd_t* h, const float* R_hist, int64_t S, int32_t nbins, const float* edges,
                 int64_t* counts) {
    if (!h || !counts || !edges || (S > 0 && !R_hist) || S < 0) { set_error("bad argument"); return LJMD_E_INVALID; }
    if (nbins < 1 || nbins > LJMD_GR_MAXBINS) { set_error("g(r): nbins must be in [1,%d]", LJMD_GR_MAXBINS); return LJMD_E_INVALID; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return gr_allpairs_hist(h, reinterpret_cast<const float2*>(R_hist), S, nbins, edges,
                            std::numeric_limits<float>::infinity(), reinterpret_cast<long long*>(counts));
}

int ljmd_gr_hist_rmax(ljmd_t* h, const float* R_hist, int64_t S, int32_t nbins, const float* edges,
                      float r_max, int64_t* counts) {
    // with S == 0 there is nothing to read or write: R_hist and counts may then be NULL (empty arrays)
    if (!h || !edges || (S > 0 && (!R_hist || !counts))) { set_error("ljmd_gr_hist_rmax: null argument"); return LJMD_E_INVALID; }
    if (S < 0) { set_error("ljmd_gr_hist_rmax: S must be >= 0"); return LJMD_E_INVALID; }
    if (nbins < 1 || nbins > LJMD_GR_MAXBINS) { set_error("ljmd_gr_hist_rmax: nbins must be in [1,%d]", LJMD_GR_MAXBINS); return LJMD_E_INVALID; }
    if (!(r_max > 0.0f) || !std::isfinite(r_max)) { set_error("ljmd_gr_hist_rmax: r_max must be positive and finite"); return LJMD_E_INVALID; }
    if (S == 0) return 0;
    LJ_CUDA(cudaSetDevice(h->p.device));
    return gr_pair_hist(h, reinterpret_cast<const float2*>(R_hist), S, nbins, edges, r_max,
                        reinterpret_cast<long long*>(counts));
}

int ljmd_density_modes(ljmd_t* h, const float* R_hist, int64_t S, const int32_t* nvec, int64_t K, double* rho) {
    if (!h) { set_error("ljmd_density_modes: null handle"); return LJMD_E_INVALID; }
    if (S < 0 || K < 0) { set_error("ljmd_density_modes: S and K must be >= 0"); return LJMD_E_INVALID; }
    // with S == 0 or K == 0 there is nothing to read or write: the arrays may then be NULL (empty)
    if (S == 0 || K == 0) return 0;
    if (!R_hist || !nvec || !rho) { set_error("ljmd_density_modes: null argument"); return LJMD_E_INVALID; }
    if ((uintptr_t)R_hist % 8 || (uintptr_t)nvec % 8 || (uintptr_t)rho % 16) {
        set_error("ljmd_density_modes: R_hist and nvec must be 8-byte aligned, rho 16-byte aligned");
        return LJMD_E_INVALID;
    }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return sk_density_modes(h, reinterpret_cast<const float2*>(R_hist), S, reinterpret_cast<const int2*>(nvec), K,
                            reinterpret_cast<double2*>(rho));
}

int ljmd_bond_order(ljmd_t* h, const float* R_hist, int64_t S, int32_t m, float r_nb, double* psi, int32_t* nnb) {
    if (!h) { set_error("ljmd_bond_order: null handle"); return LJMD_E_INVALID; }
    if (S < 0) { set_error("ljmd_bond_order: S must be >= 0"); return LJMD_E_INVALID; }
    if (m < 1 || m > 12) { set_error("ljmd_bond_order: m must be in [1,12]"); return LJMD_E_INVALID; }
    if (!(r_nb > 0.0f) || !std::isfinite(r_nb)) { set_error("ljmd_bond_order: r_nb must be positive and finite"); return LJMD_E_INVALID; }
    // with S == 0 there is nothing to read or write: the arrays may then be NULL (empty)
    if (S == 0) return 0;
    if (!R_hist || !psi) { set_error("ljmd_bond_order: null argument"); return LJMD_E_INVALID; }
    if ((uintptr_t)R_hist % 8 || (uintptr_t)psi % 16 || (uintptr_t)nnb % 4) {
        set_error("ljmd_bond_order: R_hist must be 8-byte aligned, psi 16-byte aligned, nnb 4-byte aligned");
        return LJMD_E_INVALID;
    }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return bond_order(h, reinterpret_cast<const float2*>(R_hist), S, m, r_nb, reinterpret_cast<double2*>(psi), nnb);
}

int ljmd_bond_corr(ljmd_t* h, const float* R_hist, const double* psi, int64_t S, int32_t nbins,
                   const float* edges, float r_max, int64_t* counts, int64_t* wsum) {
    if (!h) { set_error("ljmd_bond_corr: null handle"); return LJMD_E_INVALID; }
    if (S < 0) { set_error("ljmd_bond_corr: S must be >= 0"); return LJMD_E_INVALID; }
    if (nbins < 1 || nbins > LJMD_GR_MAXBINS) { set_error("ljmd_bond_corr: nbins must be in [1,%d]", LJMD_GR_MAXBINS); return LJMD_E_INVALID; }
    if (!(r_max > 0.0f) || !std::isfinite(r_max)) { set_error("ljmd_bond_corr: r_max must be positive and finite"); return LJMD_E_INVALID; }
    if (S == 0) return 0;
    if (!R_hist || !psi || !edges || !counts || !wsum) { set_error("ljmd_bond_corr: null argument"); return LJMD_E_INVALID; }
    if ((uintptr_t)R_hist % 8 || (uintptr_t)psi % 16 || (uintptr_t)counts % 8 || (uintptr_t)wsum % 8) {
        set_error("ljmd_bond_corr: R_hist, counts and wsum must be 8-byte aligned, psi 16-byte aligned");
        return LJMD_E_INVALID;
    }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return gr_pair_hist(h, reinterpret_cast<const float2*>(R_hist), S, nbins, edges, r_max,
                        reinterpret_cast<long long*>(counts), reinterpret_cast<const double2*>(psi),
                        reinterpret_cast<long long*>(wsum));
}

int ljmd_clusters(ljmd_t* h, const float* R_hist, int64_t S, float r_link, const uint8_t* mask, int32_t* labels,
                  int32_t* sizes) {
    if (!h) { set_error("ljmd_clusters: null handle"); return LJMD_E_INVALID; }
    if (S < 0) { set_error("ljmd_clusters: S must be >= 0"); return LJMD_E_INVALID; }
    if (!(r_link > 0.0f) || !std::isfinite(r_link)) { set_error("ljmd_clusters: r_link must be positive and finite"); return LJMD_E_INVALID; }
    // with S == 0 there is nothing to read or write: the arrays may then be NULL (empty)
    if (S == 0) return 0;
    if (!R_hist || !labels) { set_error("ljmd_clusters: null argument"); return LJMD_E_INVALID; }
    if ((uintptr_t)R_hist % 8 || (uintptr_t)labels % 4 || (uintptr_t)sizes % 4) {
        set_error("ljmd_clusters: R_hist must be 8-byte aligned, labels and sizes 4-byte aligned");
        return LJMD_E_INVALID;
    }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return clusters(h, reinterpret_cast<const float2*>(R_hist), S, r_link, mask, labels, sizes);
}

int ljmd_voronoi(ljmd_t* h, const float* R_hist, int64_t S, int32_t* nvor, double* area, int32_t* adj,
                 int32_t adj_cap, int32_t m, double* psi) {
    if (!h) { set_error("ljmd_voronoi: null handle"); return LJMD_E_INVALID; }
    if (S < 0) { set_error("ljmd_voronoi: S must be >= 0"); return LJMD_E_INVALID; }
    if (adj && (adj_cap < 1 || adj_cap > 64)) { set_error("ljmd_voronoi: adj_cap must be in [1,64]"); return LJMD_E_INVALID; }
    if (psi && (m < 1 || m > 12)) { set_error("ljmd_voronoi: m must be in [1,12]"); return LJMD_E_INVALID; }
    // with S == 0 there is nothing to read or write: the arrays may then be NULL (empty)
    if (S == 0) return 0;
    if (!R_hist || !nvor) { set_error("ljmd_voronoi: null argument"); return LJMD_E_INVALID; }
    if ((uintptr_t)R_hist % 8 || (uintptr_t)nvor % 4 || (uintptr_t)area % 8 || (uintptr_t)adj % 4 ||
        (uintptr_t)psi % 16) {
        set_error("ljmd_voronoi: R_hist and area must be 8-byte aligned, psi 16-byte aligned, nvor and adj 4-byte aligned");
        return LJMD_E_INVALID;
    }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return voronoi(h, reinterpret_cast<const float2*>(R_hist), S, nvor, area, adj, adj_cap, m,
                   reinterpret_cast<double2*>(psi));
}

int ljmd_cell_geometry(ljmd_t* h, int32_t* nrows, int32_t* nbins_x, int32_t* kbins,
                       float* inv_row_height, float* inv_bin_width) {
    if (!h) { set_error("null handle"); return LJMD_E_INVALID; }
    if (h->path != LJMD_PATH_CELLS) { set_error("handle is not on the cell-list path"); return LJMD_E_STATE; }
    return cells_geometry(h, nrows, nbins_x, kbins, inv_row_height, inv_bin_width);
}

int ljmd_cell_assign(ljmd_t* h, const float* R, int32_t* cell_id, int32_t* cell_count) {
    if (!h || !R) { set_error("null argument"); return LJMD_E_INVALID; }
    if (h->path != LJMD_PATH_CELLS) { set_error("handle is not on the cell-list path"); return LJMD_E_STATE; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return cells_assign(h, reinterpret_cast<const float2*>(R), cell_id, cell_count);
}

int ljmd_neighbor_count(ljmd_t* h, const float* R, float radius, int32_t* nbr_count) {
    if (!h || !R || !nbr_count) { set_error("null argument"); return LJMD_E_INVALID; }
    if (h->path != LJMD_PATH_CELLS) { set_error("handle is not on the cell-list path"); return LJMD_E_STATE; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    return cells_neighbor_count(h, reinterpret_cast<const float2*>(R), radius, nbr_count);
}

int ljmd_last_rebuilds(ljmd_t* h, int64_t* rebuilds) {
    if (!h || !rebuilds) { set_error("null argument"); return LJMD_E_INVALID; }
    if (h->path != LJMD_PATH_CELLS) { *rebuilds = 0; return 0; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    *rebuilds = cells_last_rebuilds(h);
    return 0;
}

int ljmd_check(ljmd_t* h) {
    if (!h) { set_error("null handle"); return LJMD_E_INVALID; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    LJ_CUDA(cudaStreamSynchronize(h->stream));
    int e = ap_check_error(h);
    return e ? e : cells_check_error(h);
}

int ljmd_last_run_ms(ljmd_t* h, float* ms) {
    if (!h || !ms) { set_error("null argument"); return LJMD_E_INVALID; }
    LJ_CUDA(cudaSetDevice(h->p.device));
    LJ_CUDA(cudaEventSynchronize(h->ev1));
    LJ_CUDA(cudaEventElapsedTime(ms, h->ev0, h->ev1));
    return ljmd_check(h);
}

int ljmd_allpairs_mode(ljmd_t* h, int32_t* mode) {
    if (!h || !mode) { set_error("null argument"); return LJMD_E_INVALID; }
    *mode = (h->path == LJMD_PATH_ALLPAIRS) ? ap_mode(h) : 0;
    return 0;
}

int ljmd_launch_count(ljmd_t* h, int64_t* launches) {
    if (!h || !launches) { set_error("null argument"); return LJMD_E_INVALID; }
    *launches = h->launches;
    return 0;
}

int ljmd_pair_accel(int32_t law, const float* pos, const float* mass, int64_t n, float G, float* acc,
                    void* stream) {
    return pairlaw_accel(law, reinterpret_cast<const float2*>(pos), mass, n, G,
                         reinterpret_cast<float2*>(acc), reinterpret_cast<cudaStream_t>(stream));
}

int ljmd_fp32_peak_probe(int32_t device, int32_t packed, float* tflops) {
    if (!tflops) { set_error("null argument"); return LJMD_E_INVALID; }
    return fp32_peak_probe(device, packed, tflops);
}

}  // extern "C"
