// gpb200.cu -- the engine behind the C ABI of include/gpb200.h: device state, the blocked
// factorisation / inverse schedules, and the entry points the reference-side shim binds.
//
// Device layout (all FP64, row-major, leading dimension Npad = N rounded up to 128; the padding is
// an identity block, so L, L^-1, logdet and every solve are unaffected):
//   F     Npad x Npad   lower triangle: L (K_y = L L'; the reference's U = L', src/GP.jl:110).
//                       strict-upper tiles: scratch for the triangular-inverse merges (and Z' of gpb200_gpa_grad).
//   G     Npad x Npad   lower tiles: K_y -> Schur complements during the factorisation ->
//                       W = L^-1 (strictly-lower tiles) ; strictly-upper tiles: W' ;
//                       after gpb200_grad_prepare the lower triangle holds K_y^-1,
//                       after gpb200_gpa_grad -(P + P') of the latent-GP gradient.
//   Dinv / DinvT  Npad x 128   clean lower / upper copies of the inverted diagonal tiles.
//   x     N x d point-major (== Julia's d x N column-major), uploaded once (gpb200_set_data).
// The reference keeps four N x N host matrices per GPE (R, cK.mat, chol factors, ααinvcKI;
// test/memory.jl:14-19); this engine keeps two on the device and no distance cache.
//
// Every O(N^3) step is the NT DMMA GEMM of gemm_nt.cu:
//   Cholesky: recursive panel factorisation (chol_panel): leaf = potrf128 (tile factor + tile
//   inverse in one CTA) + a 128-wide TRSM GEMM through the inverted tile; every internal node is one
//   Schur-complement GEMM over a lower trapezoid with inner dimension = half the block, so ~98% of
//   the N^3/3 flops run with K >= 1024.  Option "nb" > 0 switches to a right-looking outer loop over
//   nb-wide panels (the form the multi-GPU block-column distribution uses).
//   Inverse: bottom-up *level-parallel* triangular inverse -- at level s every pair of adjacent
//   s x s diagonal blocks is merged independently, W21 = -W_C (L21 W_A), two batched GEMMs per
//   level, 2 log2(Npad/128) launches in total -- then K_y^-1 = W' W in ONE triangular SYRK launch.
//   N^3/3 + 2N^3/3 = N^3 flop per mll+gradient (the reference's potrs on the identity costs 7N^3/3).
#include <cuda.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <limits.h>
#include <nccl.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/gpb200.h"
#include "gemm_nt.cuh"
#include "gpa.cuh"
#include "gram.cuh"
#include "gram_fast.cuh"
#include "kprog.cuh"
#include "potrf_base.cuh"
#include "shard_kernels.cuh"
#include "vec.cuh"

namespace {
constexpr int TILE = 128;
constexpr double LOG2PI = 1.8378770664093453;
std::string g_create_error;
}  // namespace

// a virtual address range backed by physical memory only where `runs` say so (CUDA VMM: cuMemAddressReserve / cuMemMap)
struct VmBuf {
    CUdeviceptr base = 0;
    size_t va_size = 0;
    std::vector<std::pair<size_t, size_t>> runs;          // (offset, bytes) of every mapped run
    std::vector<CUmemGenericAllocationHandle> handles;    // one physical allocation per run
};

struct gpb200_handle {
    int device = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
    int64_t N = 0, Npad = 0, ld = 0;
    int d = 0;
    double* x = nullptr;
    KProg prog{};
    std::vector<double> theta;
    bool has_data = false, has_kernel = false, factored = false, inv_ready = false, alpha_ready = false;
    double *F = nullptr, *G = nullptr, *Dinv = nullptr, *DinvT = nullptr, *logd = nullptr;
    double *noise_var = nullptr, *r0 = nullptr, *r1 = nullptr, *y1 = nullptr, *alpha = nullptr, *scal = nullptr;
    double *part = nullptr, *trace_out = nullptr;
    double* tblk = nullptr;                    // Npad scratch vector (block right-hand sides of the sharded solves)
    // latent-GP gradient (gpb200_gpa_grad): Z' diagonal tiles [Npad x 128] and [Npad/128 x Npad] per-tile partial sums
    double *Zd = nullptr, *gpa_part = nullptr;
    int64_t gpa_npad = 0;                      // Npad the two buffers were sized for
    CUtensorMap mapZd{};
    bool chol_bar_ready = false;               // G's lower triangle holds -(P + P') of the last gpb200_gpa_grad
    cudaEvent_t ev_gpa[6] = {};                // phase boundaries of gpb200_unwhiten / gpb200_gpa_grad (timings [9..13])
    // TMA-staged SEIso kernels (gram_fast.cu): inputs stored [Npad x dxp] with an even, zero-padded dxp <= 8
    double *xp = nullptr, *xpt = nullptr;      // [Npad x dxp] and its transpose [dxp x Npad]
    int dxp = 0;
    CUtensorMap mapX{}, mapXT{};
    bool xmap_ok = false;
    int64_t capacity = 0;                      // option "capacity": rows reserved for gpb200_append (ElasticGPE's capacity)
    int gram_fast = 1;                         // option "gram_fast": 0 = always the generic kernels of gram.cu
    // cross-validation (gpb200_cv_*): K_y^-1 mirrored to a full symmetric matrix in G; two N x N temporaries
    bool g_sym = false;
    bool cv_m_ok = false;                                       // cvD holds M_j = Z_j K^-1 of the last cv_param call
    double *cvD = nullptr, *cvY = nullptr;
    CUtensorMap mapCvD{}, mapCvY{};
    double* cvblk = nullptr; long long* cvidx = nullptr; int64_t cvblk_cap = 0;
    // posterior sampling (gpb200_rand): M x M sub-engine for chol(Sigma* + nugget I), normal draws / samples staging
    gpb200_handle* sub = nullptr;
    bool cov_keep_device = false;              // predict: leave the full covariance in Kss (no D2H)
    double *rz = nullptr, *rout = nullptr;
    int64_t rz_rows = 0, rz_cols = 0;
    CUtensorMap mapRz{};
    int* info_dev = nullptr;
    int* flags = nullptr;                      // ready-flags of the single-launch triangular solves (2 x (Npad/128 + 1))
    int trsv_fused = 1;
    int max_resident_ctas = 0;
    int64_t n_noise = 1;
    double nugget = 0.0;
    CUtensorMap mapF{}, mapG{}, mapDinv{}, mapDinvT{};
    bool tma_ok = false;
    // predict workspace
    double *xs = nullptr, *Kst = nullptr, *Kss = nullptr, *pmu = nullptr, *pvar = nullptr, *pkdiag = nullptr;
    int64_t xs_cap = 0, Kst_rows = 0, Kss_rows = 0;
    CUtensorMap mapKst{};
    // options
    int nb = 0;                 // outer Cholesky block; 0 = fully recursive (one panel)
    int gemm_impl = 0;
    int lookahead = 1;          // factor the next diagonal tile on a side stream while the Schur update runs
    cudaStream_t st_side = nullptr;            // high-priority stream of the look-ahead chain
    cudaStream_t st_cur = nullptr;             // stream launch_gemm / the leaf use right now (st or st_side)
    cudaEvent_t ev_la0 = nullptr, ev_la2 = nullptr;
    // stats
    double ms[16] = {};
    int64_t launches = 0;
    bool own_stream = true;
    // per-launch GEMM profiling (option "profile"): event pairs + executed flops of every GEMM launch
    int profile = 0;
    std::vector<cudaEvent_t> pev;
    size_t pev_used = 0;
    double gemm_flops_exec = 0.0;
    int64_t gemm_launches = 0;
    // multi-GPU (one process per GPU): replicated F/G, block-column ownership, NCCL over NVLink
    int nranks = 1, rank = 0;
    ncclComm_t comm = nullptr;
    cudaStream_t st_comm = nullptr;
    int dist_nb = 0;                           // width of an owned block column; 0 = auto (~Npad/(8*nranks))
    double* pack[2] = {nullptr, nullptr};      // panel staging (double buffered)
    size_t pack_elems = 0;
    cudaEvent_t ev_packed[2] = {nullptr, nullptr}, ev_bcast[2] = {nullptr, nullptr}, ev_unpacked[2] = {nullptr, nullptr};
    cudaEvent_t ev_x = nullptr, ev_y = nullptr;
    double *ag_send = nullptr, *ag_recv = nullptr;
    size_t ag_send_elems = 0, ag_recv_elems = 0;
    // fused panel broadcast over NVLink peer memory (CUDA IPC): peers' F / Dinv / DinvT / logd / signal words
    bool p2p = false;
    int n_peer = 0;
    int peer_rank[7] = {0, 0, 0, 0, 0, 0, 0};
    double *peer_F[7] = {}, *peer_Dinv[7] = {}, *peer_DinvT[7] = {}, *peer_logd[7] = {};
    int* peer_sig[7] = {};
    int* sig = nullptr;                        // sig[q] = last panel published by rank q (epoch * 65536 + b + 1); sig[8] = watchdog
    int epoch = 0;
    int** peer_sig_dev = nullptr;              // device array: &peer_sig[q][rank]
    bool push_panel = false;                   // set while the owner factors a panel: leaf + leaf TRSM also store to the peers
    // ---- row-sharded storage (shard_impl.cuh): F / G are virtual address ranges, physical pages exist for owned rows only ----
    int shard_opt = -1;                        // option "shard": -1 auto (when replicated F+G would not fit), 0 never, 1 always
    int shard_rb_opt = 0;                      // option "shard_rb": ownership block in 128-row tiles (0 = auto)
    bool sharded = false;                      // current storage mode of F / G
    int rb = 4;                                // effective ownership block (tiles); panel width NBp = 128 * rb
    int shard_la = 1;                          // option "shard_la": look-ahead schedules of the sharded Cholesky / inverse
    int row_lim = 0;                           // chol_panel: rows below this limit only (diagonal block of a sharded panel); 0 = Npad
    VmBuf vmF, vmG;
    double* P[4] = {nullptr, nullptr, nullptr, nullptr};   // panel buffers, Npad x NBp (global row order); P[1], P[3] double as NBp x Npad row panels
    double* Sbuf = nullptr;                    // all-gather staging: nranks regions of S_per_rank doubles; scratch of the inverse sweep
    size_t S_per_rank = 0;
    CUtensorMap mapP[4] = {}, mapXR[2] = {}, mapS{};
    double* XRbig[2] = {nullptr, nullptr};     // row-panel forms X_J of a BATCH of panels (inverse sweep: batched LAUUM part)
    int xr_batch = 1;                          // panels per batch
    CUtensorMap mapXRbig[2] = {};
    double* red = nullptr;                     // small reduction scratch (local group all-reduce)
    int* redi = nullptr;
    struct gpb200_group* grp = nullptr;        // in-process group of virtual ranks on one device (gpb200_group_create)
    std::vector<cudaEvent_t> evring;
    size_t evring_next = 0;
    std::string err;
};

// in-process "communicator": R handles on one device acting as R ranks of the sharded schedules, driven in lock step by
// one host thread.  Collectives are device-to-device copies ordered by events (shard_impl.cuh).
struct gpb200_group {
    std::vector<gpb200_handle*> hs;
};


// ---- FITC (sparse/fully_indep_train_conditional.jl): two dense M x M sub-engines + N-chunk streaming ----
struct gpb200_fitc {
    gpb200_handle* eu = nullptr;     // K_uu  (+1e-10 I)            -> L_uu
    gpb200_handle* es = nullptr;     // Sigma_QR = K_uf L^-1 K_fu + K_uu (+1e-10 I) -> L_s
    int device = 0;
    int64_t N = 0, M = 0, Mpad = 0, Nc = 0;
    int d = 0;
    double *x = nullptr, *xs = nullptr, *lam = nullptr, *y = nullptr, *alpha = nullptr, *tmpn = nullptr;
    double *w = nullptr, *tmpc = nullptr, *zeroc = nullptr, *tmpc2 = nullptr;          // Nc
    double *bvec = nullptr, *uvec = nullptr, *tmpm = nullptr, *rhsm = nullptr, *scal = nullptr;   // Mpad
    double *bufA = nullptr, *bufB = nullptr;   // Nc x Mpad (K_fu chunk) ; Mpad x Nc (K_uf chunk)
    CUtensorMap mapA{}, mapB{}, mapB2{};
    // kernel-gradient workspace (allocated on first use)
    double *bufC = nullptr, *Hbuf = nullptr, *Wbuf = nullptr, *Tbuf = nullptr, *gvec = nullptr, *betav = nullptr;
    double *gpart = nullptr, *gacc = nullptr, *gtmp = nullptr;
    CUtensorMap mapAt{}, mapC{}, mapCt{}, mapH{}, mapT{};
    bool grad_ws = false;
    double* Kss = nullptr; int64_t Kss_rows = 0;      // full predictive covariance (gpb200_fitc_predict_cov)
    // multi-GPU (gpb200_fitc_comm_init): the N observations are sharded over the ranks, every M x M object is replicated;
    // exchanged: one all-reduce of the M x M accumulator Sigma_QR (and of H for the kernel gradient), M-vectors, scalars
    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;
    double Ntotal = 0.0;                              // observations over all ranks (mll's N log 2 pi)
    int mode = 0;                    // 0 FITC, 1 DTC, 2 SoR (Lambda = sigma^2 I; SoR also drops K_xx - Q_xx from the predictive variance)
    double noise_var = 0.0;
    bool has_data = false, has_kernel = false, factored = false, alpha_ready = false;
    std::string err;
};

namespace {

// ---- NCCL, bound at run time (dlopen) so that single-GPU use has no NCCL dependency -------------
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    bool ok = false;
} g_nccl;

bool nccl_load() {
    if (g_nccl.ok) return true;
    if (!g_nccl.lib) g_nccl.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl.lib) g_nccl.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!g_nccl.lib) return false;
    void* L = g_nccl.lib;
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))dlsym(L, "ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))dlsym(L, "ncclCommInitRank");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))dlsym(L, "ncclCommDestroy");
    g_nccl.Broadcast = (decltype(g_nccl.Broadcast))dlsym(L, "ncclBroadcast");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))dlsym(L, "ncclAllGather");
    g_nccl.AllReduce = (decltype(g_nccl.AllReduce))dlsym(L, "ncclAllReduce");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(L, "ncclGetErrorString");
    g_nccl.GroupStart = (decltype(g_nccl.GroupStart))dlsym(L, "ncclGroupStart");
    g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))dlsym(L, "ncclGroupEnd");
    g_nccl.ok = g_nccl.GetUniqueId && g_nccl.CommInitRank && g_nccl.CommDestroy && g_nccl.Broadcast &&
                g_nccl.AllGather && g_nccl.AllReduce && g_nccl.GetErrorString && g_nccl.GroupStart && g_nccl.GroupEnd;
    return g_nccl.ok;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,       \
                     cudaGetErrorString(e_));                                                      \
            h->err = buf_;                                                                         \
            (void)cudaGetLastError();                                                              \
            return GPB200_ECUDA;                                                                   \
        }                                                                                          \
    } while (0)

#define CKN(call)                                                                                  \
    do {                                                                                           \
        ncclResult_t r_ = (call);                                                                  \
        if (r_ != ncclSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,       \
                     g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error");            \
            h->err = buf_;                                                                         \
            return GPB200_ENCCL;                                                                   \
        }                                                                                          \
    } while (0)

int fail(gpb200_handle* h, int code, const char* msg) {
    if (h) h->err = msg;
    return code;
}

// unmap every peer buffer imported by gpb200_ipc_import (a realloc or a re-import makes them stale)
void close_peer_maps(gpb200_handle* h) {
    for (int q = 0; q < h->n_peer; ++q) {
        cudaIpcCloseMemHandle(h->peer_F[q]); cudaIpcCloseMemHandle(h->peer_Dinv[q]);
        cudaIpcCloseMemHandle(h->peer_DinvT[q]); cudaIpcCloseMemHandle(h->peer_logd[q]);
        cudaIpcCloseMemHandle(h->peer_sig[q]);
        h->peer_F[q] = h->peer_Dinv[q] = h->peer_DinvT[q] = h->peer_logd[q] = nullptr; h->peer_sig[q] = nullptr;
    }
    (void)cudaGetLastError();
    h->p2p = false; h->n_peer = 0;
}

void free_FG(gpb200_handle* h);               // shard_impl.cuh: F / G are cudaMalloc'ed (replicated) or VMM ranges (row-sharded)

void free_data(gpb200_handle* h) {
    free_FG(h);
    double** ptrs[] = {&h->x, &h->Dinv, &h->DinvT, &h->logd, &h->noise_var, &h->r0, &h->r1,
                       &h->y1, &h->alpha, &h->scal, &h->part, &h->trace_out, &h->xs, &h->Kst, &h->Kss,
                       &h->pmu, &h->pvar, &h->pkdiag, &h->tblk, &h->xp, &h->xpt, &h->Zd, &h->gpa_part};
    h->gpa_npad = 0; h->chol_bar_ready = false;
    h->xmap_ok = false;
    if (h->cvD) cudaFree(h->cvD);
    if (h->cvY) cudaFree(h->cvY);
    if (h->cvblk) cudaFree(h->cvblk);
    if (h->cvidx) cudaFree(h->cvidx);
    h->cvD = h->cvY = h->cvblk = nullptr; h->cvidx = nullptr; h->cvblk_cap = 0; h->g_sym = false; h->cv_m_ok = false;
    for (auto pp : ptrs) { if (*pp) cudaFree(*pp); *pp = nullptr; }
    if (h->info_dev) { cudaFree(h->info_dev); h->info_dev = nullptr; }
    if (h->flags) { cudaFree(h->flags); h->flags = nullptr; }
    close_peer_maps(h);                        // peers' mappings refer to the old buffers whether or not p2p is switched on
    if (h->sig) { cudaFree(h->sig); h->sig = nullptr; }
    if (h->peer_sig_dev) { cudaFree(h->peer_sig_dev); h->peer_sig_dev = nullptr; }
    for (int i = 0; i < 2; ++i) { if (h->pack[i]) cudaFree(h->pack[i]); h->pack[i] = nullptr; }
    if (h->ag_send) cudaFree(h->ag_send);
    if (h->ag_recv) cudaFree(h->ag_recv);
    h->ag_send = h->ag_recv = nullptr; h->pack_elems = h->ag_send_elems = h->ag_recv_elems = 0;
    h->xs_cap = h->Kst_rows = h->Kss_rows = 0;
    h->has_data = h->factored = h->inv_ready = h->alpha_ready = false;
}

GemmBuf bufF(gpb200_handle* h) { return GemmBuf{h->tma_ok ? &h->mapF : nullptr, h->F, h->ld}; }
GemmBuf bufG(gpb200_handle* h) { return GemmBuf{h->tma_ok ? &h->mapG : nullptr, h->G, h->ld}; }
GemmBuf bufDinv(gpb200_handle* h) { return GemmBuf{h->tma_ok ? &h->mapDinv : nullptr, h->Dinv, TILE}; }
GemmBuf bufDinvT(gpb200_handle* h) { return GemmBuf{h->tma_ok ? &h->mapDinvT : nullptr, h->DinvT, TILE}; }
GemmBuf bufNone() { return GemmBuf{nullptr, nullptr, 0}; }

// flops the GEMM launch executes (tile-granular: whole 128x128 tiles, clipped k ranges)
double gemm_exec_flops(const GemmDesc& d) {
    double total = 0.0;
    for (int z = 0; z < d.batch; ++z) {
        const int zo = z * d.zstep;
        const int Mz = std::min(d.M, d.m_lim - zo), Nz = std::min(d.N, d.n_lim - zo), Kz = std::min(d.K, d.k_lim - zo);
        if (Mz <= 0 || Nz <= 0 || Kz <= 0) continue;
        const int tm = Mz / TILE, tn = Nz / TILE;
        for (int bm = 0; bm < tm; ++bm) {
            if (d.bm_mod > 1 && (((bm + d.bm_off) / (d.bm_div > 0 ? d.bm_div : 1)) % d.bm_mod) != d.bm_rem) continue;
            const int bn_hi = (d.flags & GEMM_LOWER_ONLY) ? std::min(bm + 1, tn) : tn;
            for (int bn = 0; bn < bn_hi; ++bn) {
                if (d.bn_mod > 1 && (((bn + d.bn_off) / (d.bn_div > 0 ? d.bn_div : 1)) % d.bn_mod) != d.bn_rem) continue;
                int lo = (d.flags & GEMM_KLO_M) ? d.klo_off + bm * TILE : 0;
                if (d.flags & GEMM_KLO_N) lo = std::max(lo, bn * TILE);
                int hi = Kz;
                if (d.flags & GEMM_KHI_M) hi = std::min(hi, (bm + 1) * TILE);
                if (d.flags & GEMM_KHI_N) hi = std::min(hi, (bn + 1) * TILE);
                if (hi > lo) total += 2.0 * TILE * TILE * (double)(hi - lo);
            }
        }
    }
    return total;
}

cudaError_t launch_gemm(gpb200_handle* h, const GemmDesc& d) {
    ++h->launches;
    const int impl = h->tma_ok ? h->gemm_impl : 1;
    cudaStream_t stc = h->st_cur ? h->st_cur : h->st;
    if (!h->profile || stc != h->st) return gemm_nt_launch(d, impl, stc);
    if (h->pev_used + 2 > h->pev.size()) {
        const size_t old = h->pev.size();
        h->pev.resize(old + 512);
        for (size_t i = old; i < h->pev.size(); ++i) cudaEventCreate(&h->pev[i]);
    }
    cudaEventRecord(h->pev[h->pev_used++], h->st);
    cudaError_t e = gemm_nt_launch(d, impl, h->st);
    cudaEventRecord(h->pev[h->pev_used++], h->st);
    h->gemm_flops_exec += gemm_exec_flops(d);
    ++h->gemm_launches;
    return e;
}

// after a stream sync: fold the recorded GEMM launch durations into ms[6..8] and reset
void profile_collect(gpb200_handle* h) {
    if (!h->profile) return;
    double tot = 0.0;
    for (size_t i = 0; i + 1 < h->pev_used; i += 2) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->pev[i], h->pev[i + 1]) == cudaSuccess) tot += ms;
    }
    h->ms[6] += (double)h->gemm_launches;
    h->ms[7] += tot;
    h->ms[8] += h->gemm_flops_exec;
    h->pev_used = 0; h->gemm_flops_exec = 0.0; h->gemm_launches = 0;
}

// ---- pieces of the factorisation --------------------------------------------------------------

// F[r0.., p..p+128) = G[r0.., p..p+128) * W_pp'   (leaf panel TRSM through the inverted diagonal tile)
cudaError_t panel_trsm_leaf(gpb200_handle* h, int r0, int rows, int p) {
    GemmDesc g = gemm_desc_default();
    g.A = GemmOperand{bufG(h), bufNone(), r0, p};
    g.B = GemmOperand{bufDinv(h), bufNone(), p, 0};
    g.C = h->F; g.ldc = h->ld; g.c_row0 = r0; g.c_col0 = p;
    g.M = rows; g.N = TILE; g.K = TILE;
    if (h->push_panel) {                       // fused broadcast: the epilogue also writes the peers' factor
        g.n_peer = h->n_peer;
        for (int q = 0; q < h->n_peer; ++q) g.Cpeer[q] = h->peer_F[q];
    }
    return launch_gemm(h, g);
}
// Schur update of the lower trapezoid G[r0.., r0..r0+cols) -= F[r0.., p..p+k) F[r0..r0+cols, p..p+k)'
// (rows >= cols; cols == rows gives the classical trailing SYRK)
cudaError_t schur_update(gpb200_handle* h, int r0, int rows, int cols, int p, int k, int extra_flags = 0) {
    GemmDesc g = gemm_desc_default();
    g.A = GemmOperand{bufF(h), bufNone(), r0, p};
    g.B = GemmOperand{bufF(h), bufNone(), r0, p};
    g.C = h->G; g.ldc = h->ld; g.c_row0 = r0; g.c_col0 = r0;
    g.M = rows; g.N = cols; g.K = k;
    g.alpha = -1.0; g.beta = 1.0;
    g.flags = GEMM_LOWER_ONLY | extra_flags;
    return launch_gemm(h, g);
}
// merge of the inverses of two adjacent diagonal blocks [p,p+n1) and [p+n1,p+n1+n2):
//   T' = Wt_A * L21'  -> F strict-upper block (p, p+n1)
//   W21 = -W_C * T    -> G (p+n1, p)  and its transpose -> G (p, p+n1)
// batched over `batch` problems stepping 2*n1 along the diagonal (clipped at Npad).
cudaError_t merge_inverse(gpb200_handle* h, int p, int n1, int n2, int batch) {
    const int lim = (int)h->Npad - p - n1;     // rows available below the first block of problem 0
    {
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bufG(h), bufDinvT(h), p, p};
        g.B = GemmOperand{bufF(h), bufNone(), p + n1, p};
        g.C = h->F; g.ldc = h->ld; g.c_row0 = p; g.c_col0 = p + n1;
        g.M = n1; g.N = n2; g.K = n1;
        g.flags = GEMM_KLO_M;
        g.batch = batch; g.zstep = 2 * n1;
        g.n_lim = lim;
        cudaError_t e = launch_gemm(h, g);
        if (e != cudaSuccess) return e;
    }
    {
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bufG(h), bufDinv(h), p + n1, p + n1};
        g.B = GemmOperand{bufF(h), bufNone(), p, p + n1};
        g.C = h->G; g.ldc = h->ld; g.c_row0 = p + n1; g.c_col0 = p;
        g.Ct = h->G; g.ldct = h->ld; g.ct_row0 = p; g.ct_col0 = p + n1;
        g.M = n2; g.N = n1; g.K = n2;
        g.alpha = -1.0;
        g.flags = GEMM_KHI_M;
        g.batch = batch; g.zstep = 2 * n1;
        g.m_lim = lim; g.k_lim = lim;
        return launch_gemm(h, g);
    }
}

// Recursive panel Cholesky: factor columns [p, p+n) for ALL rows below (n <= s, s = 128 * 2^k,
// p aligned to s).  Every Schur update inside is one NT GEMM whose inner dimension is the half
// block size, so ~98% of the flops run with K >= 1024 (near-peak DMMA activity); only the
// 128-wide leaves (tile factorisation + TRSM through the inverted tile) are latency bound.
cudaError_t leaf_launch(gpb200_handle* h, int p, cudaStream_t st) {
    ++h->launches;
    PotrfPeers pp{};
    if (h->push_panel) {
        pp.n = h->n_peer;
        for (int q = 0; q < h->n_peer; ++q) { pp.F[q] = h->peer_F[q]; pp.Dinv[q] = h->peer_Dinv[q]; pp.DinvT[q] = h->peer_DinvT[q]; pp.logd[q] = h->peer_logd[q]; }
    }
    return potrf128_launch(h->G, h->ld, h->F, h->ld, h->Dinv, h->DinvT, h->logd, h->info_dev, p, 1, TILE, st, &pp);
}

// `leaf_done`: the tile at p was already factored by the look-ahead chain on the side stream (join it first).
// Look-ahead: once the left half of a node is done, the ONE tile of the Schur update the next leaf needs and
// that leaf run on a high-priority side stream while the main stream does the rest of the update -- the
// 125 us latency-bound leaf disappears behind the GEMM.
cudaError_t chol_panel(gpb200_handle* h, int p, int n, int s, bool leaf_done = false) {
    const int Np = h->row_lim > 0 ? h->row_lim : (int)h->Npad;
    cudaError_t e;
    if (s == TILE) {
        if (leaf_done) e = cudaStreamWaitEvent(h->st, h->ev_la2, 0);
        else e = leaf_launch(h, p, h->st);
        if (e != cudaSuccess) return e;
        const int below = Np - p - TILE;
        return below > 0 ? panel_trsm_leaf(h, p + TILE, below, p) : cudaSuccess;
    }
    const int hs = s / 2;
    if (n <= hs) return chol_panel(h, p, n, hs, leaf_done);
    if ((e = chol_panel(h, p, hs, hs, leaf_done)) != cudaSuccess) return e;
    const int rows = Np - p - hs, cols = n - hs;
    if (h->lookahead && h->st_side) {
        if ((e = cudaEventRecord(h->ev_la0, h->st)) != cudaSuccess) return e;
        if ((e = cudaStreamWaitEvent(h->st_side, h->ev_la0, 0)) != cudaSuccess) return e;
        h->st_cur = h->st_side;
        e = schur_update(h, p + hs, TILE, TILE, p, hs);                 // the next diagonal tile only
        h->st_cur = nullptr;
        if (e != cudaSuccess) return e;
        if ((e = leaf_launch(h, p + hs, h->st_side)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(h->ev_la2, h->st_side)) != cudaSuccess) return e;
        if ((e = schur_update(h, p + hs, rows, cols, p, hs, GEMM_SKIP_FIRST)) != cudaSuccess) return e;
        return chol_panel(h, p + hs, cols, hs, true);
    }
    if ((e = schur_update(h, p + hs, rows, cols, p, hs)) != cudaSuccess) return e;
    return chol_panel(h, p + hs, cols, hs);
}

cudaError_t cholesky(gpb200_handle* h) {
    const int Np = (int)h->Npad;
    // outer block: option "nb" (0 = one panel spanning the matrix: fully recursive)
    int NB = TILE;
    const int want = h->nb > 0 ? h->nb : Np;
    while (NB < want && NB < Np) NB *= 2;
    cudaError_t e;
    for (int p = 0; p < Np; p += NB) {
        const int n = (Np - p < NB) ? Np - p : NB;
        if ((e = chol_panel(h, p, n, NB)) != cudaSuccess) return e;
        const int rem = Np - p - n;
        if (rem > 0 && (e = schur_update(h, p + n, rem, rem, p, n)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// W = L^-1 from the factor: level-parallel triangular inverse (all pairs of adjacent s x s diagonal
// blocks merged at once, s = 128, 256, ...: 2 batched GEMM launches per level).  W' ends in G's
// strictly-upper tiles (diagonal tiles: DinvT).
cudaError_t inverse_merges(gpb200_handle* h) {
    const int Np = (int)h->Npad;
    cudaError_t e;
    for (long long s = TILE; s < Np; s *= 2) {
        const int batch = (int)((Np + 2 * s - 1) / (2 * s));
        const int n2 = (int)((Np - s < s) ? Np - s : s);
        if ((e = merge_inverse(h, 0, (int)s, n2, batch)) != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// K_y^-1 from the factor: the triangular inverse, then W'W.
cudaError_t inverse_from_factor(gpb200_handle* h) {
    const int Np = (int)h->Npad;
    cudaError_t e;
    if ((e = inverse_merges(h)) != cudaSuccess) return e;
    GemmDesc g = gemm_desc_default();
    g.A = GemmOperand{bufG(h), bufDinvT(h), 0, 0};
    g.B = GemmOperand{bufG(h), bufDinvT(h), 0, 0};
    g.C = h->G; g.ldc = h->ld; g.c_row0 = 0; g.c_col0 = 0;
    g.M = Np; g.N = Np; g.K = Np;
    g.flags = GEMM_LOWER_ONLY | GEMM_KLO_M;
    return launch_gemm(h, g);
}


// ================================================================================================
// multi-GPU schedules (nranks > 1).  Storage is replicated (every rank holds full F, G, Dinv);
// WORK is partitioned:
//   Gram / Cholesky : 1-D block-cyclic ownership of dist_nb-wide block columns.  The owner factors
//                     its panel (chol_panel), the panel is broadcast (NCCL over NVLink, on a side
//                     stream, double-buffered), every rank applies it to the block columns it owns.
//                     The owner of the NEXT panel updates and factors that panel first and ships it
//                     before finishing its remaining updates (look-ahead), so the broadcast and the
//                     latency-bound panel factorisation hide behind the other ranks' updates.
//   inverse         : small levels of the level-parallel triangular inverse are recomputed on every
//                     rank; from block size 128*nranks upwards each merge is split by column slices
//                     of W21 (no exchange between its two GEMMs), then all-gathered.
//   W'W + trace     : tile rows dealt round-robin; only the P+1 partial sums are all-reduced, K^-1
//                     itself is never exchanged.
// ================================================================================================
// rank q owns the 128-wide tile columns t with t % nranks == q of every W21 block; its "slice" is
// the concatenation of those tile columns (local column jl <-> global column ((jl/128)*nranks+q)*128 + jl%128)
__global__ void pack_slices_kernel(const double* __restrict__ G, long long ld, double* __restrict__ out,
                                   int s, int wr, int nranks, int self, int Np) {
    const int z = blockIdx.z;
    const int p = z * 2 * s;
    const int n2 = min(s, Np - p - s);
    const int i = blockIdx.y * 32 + threadIdx.y, jl = blockIdx.x * 32 + threadIdx.x;
    if (n2 <= 0 || i >= n2 || jl >= wr) return;
    const int gj = ((jl >> 7) * nranks + self) * 128 + (jl & 127);
    out[(long long)z * s * wr + (long long)i * wr + jl] = G[(long long)(p + s + i) * ld + p + gj];
}
// scatter the gathered W21 slices of all other ranks into G (lower block) and, transposed, into
// G's strict-upper block
__global__ void unpack_slices_kernel(double* __restrict__ G, long long ld, const double* __restrict__ in,
                                     long long per_rank, int s, int wr, int Np, int nranks, int self) {
    __shared__ double tile[32][33];
    const int batch = (Np + 2 * s - 1) / (2 * s);
    const int z = blockIdx.z % batch;
    const int q = blockIdx.z / batch;
    if (q == self) return;
    const int p = z * 2 * s;
    const int n2 = min(s, Np - p - s);
    if (n2 <= 0) return;
    const double* src = in + (long long)q * per_rank + (long long)z * s * wr;
    const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;            // 32 | 128: a block never straddles tiles
    if (i0 >= n2 || j0 >= wr) return;
    const int i = i0 + threadIdx.y, jl = j0 + threadIdx.x;
    double v = 0.0;
    if (i < n2 && jl < wr) {
        v = src[(long long)i * wr + jl];
        const int gj = ((jl >> 7) * nranks + q) * 128 + (jl & 127);
        G[(long long)(p + s + i) * ld + p + gj] = v;
    }
    tile[threadIdx.y][threadIdx.x] = v;
    __syncthreads();
    const int ti = i0 + threadIdx.x, tjl = j0 + threadIdx.y;
    if (ti < n2 && tjl < wr) {
        const int gj = ((tjl >> 7) * nranks + q) * 128 + (tjl & 127);
        G[(long long)(p + gj) * ld + p + s + ti] = tile[threadIdx.x][threadIdx.y];
    }
}

int dist_block(gpb200_handle* h) {
    int NB = TILE;
    if (h->dist_nb > 0) { while (NB < h->dist_nb && NB < h->Npad) NB *= 2; return NB; }
    const long long target = h->Npad / (8LL * h->nranks);           // ~8 block columns per rank (measured best at 2/4/8 GPUs)
    while (NB * 2 <= target && NB < 4096) NB *= 2;
    return NB < 256 ? (h->Npad >= 256 ? 256 : TILE) : NB;
}

int dist_alloc(gpb200_handle* h) {
    const size_t Np = (size_t)h->Npad;
    const size_t nbw = (size_t)dist_block(h);
    const size_t need_pack = Np * nbw + 2 * nbw * TILE + nbw + 16;
    if (need_pack > h->pack_elems) {
        for (int i = 0; i < 2; ++i) {
            if (h->pack[i]) cudaFree(h->pack[i]);
            h->pack[i] = nullptr;
            CK(cudaMalloc(&h->pack[i], sizeof(double) * need_pack));
        }
        h->pack_elems = need_pack;
    }
    const size_t need_recv = Np * Np / 4 + Np * TILE;
    const size_t need_send = need_recv / h->nranks + Np * TILE;
    if (need_recv > h->ag_recv_elems) {
        if (h->ag_recv) cudaFree(h->ag_recv);
        if (h->ag_send) cudaFree(h->ag_send);
        h->ag_recv = h->ag_send = nullptr;
        CK(cudaMalloc(&h->ag_recv, sizeof(double) * need_recv));
        CK(cudaMalloc(&h->ag_send, sizeof(double) * need_send));
        h->ag_recv_elems = need_recv; h->ag_send_elems = need_send;
    }
    return GPB200_OK;
}

size_t panel_count(gpb200_handle* h, int p, int n) {
    return (size_t)(h->Npad - p) * n + 2 * (size_t)n * TILE + (size_t)n;
}
// F[p.., p..p+n) + Dinv/DinvT rows p..p+n + logd[p..p+n)  <->  contiguous staging buffer
cudaError_t panel_pack(gpb200_handle* h, int p, int n, double* buf, bool unpack) {
    const size_t rows = (size_t)(h->Npad - p);
    double* fpan = h->F + (size_t)p * h->ld + p;
    cudaError_t e;
    if (!unpack) e = cudaMemcpy2DAsync(buf, sizeof(double) * n, fpan, sizeof(double) * h->ld, sizeof(double) * n, rows, cudaMemcpyDeviceToDevice, h->st);
    else         e = cudaMemcpy2DAsync(fpan, sizeof(double) * h->ld, buf, sizeof(double) * n, sizeof(double) * n, rows, cudaMemcpyDeviceToDevice, h->st);
    if (e != cudaSuccess) return e;
    double* b1 = buf + rows * n;
    double* b2 = b1 + (size_t)n * TILE;
    double* b3 = b2 + (size_t)n * TILE;
    const size_t tb = sizeof(double) * (size_t)n * TILE;
    if (!unpack) {
        if ((e = cudaMemcpyAsync(b1, h->Dinv + (size_t)p * TILE, tb, cudaMemcpyDeviceToDevice, h->st)) != cudaSuccess) return e;
        if ((e = cudaMemcpyAsync(b2, h->DinvT + (size_t)p * TILE, tb, cudaMemcpyDeviceToDevice, h->st)) != cudaSuccess) return e;
        return cudaMemcpyAsync(b3, h->logd + p, sizeof(double) * n, cudaMemcpyDeviceToDevice, h->st);
    }
    if ((e = cudaMemcpyAsync(h->Dinv + (size_t)p * TILE, b1, tb, cudaMemcpyDeviceToDevice, h->st)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(h->DinvT + (size_t)p * TILE, b2, tb, cudaMemcpyDeviceToDevice, h->st)) != cudaSuccess) return e;
    return cudaMemcpyAsync(h->logd + p, b3, sizeof(double) * n, cudaMemcpyDeviceToDevice, h->st);
}

int cholesky_dist(gpb200_handle* h) {
    const int Np = (int)h->Npad, R = h->nranks, me = h->rank;
    const int NB = dist_block(h);
    const int nblk = (Np + NB - 1) / NB;
    auto bp = [&](int b) { return b * NB; };
    auto bn = [&](int b) { return std::min(NB, Np - b * NB); };
    auto owner = [&](int b) { return b % R; };
    auto update = [&](int jb, int b) {      // block column jb <- panel b
        const int r0 = bp(jb);
        return schur_update(h, r0, Np - r0, bn(jb), bp(b), bn(b));
    };
    // panel 0
    if (owner(0) == me) {
        CK(chol_panel(h, 0, bn(0), NB));
        CK(panel_pack(h, 0, bn(0), h->pack[0], false));
        CK(cudaEventRecord(h->ev_packed[0], h->st));
        CK(cudaStreamWaitEvent(h->st_comm, h->ev_packed[0], 0));
    }
    CKN(g_nccl.Broadcast(h->pack[0], h->pack[0], panel_count(h, 0, bn(0)), ncclDouble, owner(0), h->comm, h->st_comm));
    CK(cudaEventRecord(h->ev_bcast[0], h->st_comm));
    for (int b = 0; b < nblk; ++b) {
        const int cur = b & 1, nxt = cur ^ 1;
        CK(cudaStreamWaitEvent(h->st, h->ev_bcast[cur], 0));
        if (owner(b) != me) CK(panel_pack(h, bp(b), bn(b), h->pack[cur], true));
        CK(cudaEventRecord(h->ev_unpacked[cur], h->st));
        bool did_next = false;
        if (b + 1 < nblk) {
            if (owner(b + 1) == me) {                         // look-ahead: next panel first
                CK(update(b + 1, b));
                CK(chol_panel(h, bp(b + 1), bn(b + 1), NB));
                CK(panel_pack(h, bp(b + 1), bn(b + 1), h->pack[nxt], false));
                CK(cudaEventRecord(h->ev_packed[nxt], h->st));
                CK(cudaStreamWaitEvent(h->st_comm, h->ev_packed[nxt], 0));
                did_next = true;
            } else if (b >= 1) {
                CK(cudaStreamWaitEvent(h->st_comm, h->ev_unpacked[nxt], 0));   // staging buffer free again
            }
            CKN(g_nccl.Broadcast(h->pack[nxt], h->pack[nxt], panel_count(h, bp(b + 1), bn(b + 1)), ncclDouble,
                                 owner(b + 1), h->comm, h->st_comm));
            CK(cudaEventRecord(h->ev_bcast[nxt], h->st_comm));
        }
        for (int jb = b + 1 + (did_next ? 1 : 0); jb < nblk; ++jb)
            if (owner(jb) == me) CK(update(jb, b));
    }
    // first failing pivot over all ranks
    CK(cudaEventRecord(h->ev_x, h->st));
    CK(cudaStreamWaitEvent(h->st_comm, h->ev_x, 0));
    CKN(g_nccl.AllReduce(h->info_dev, h->info_dev, 1, ncclInt32, ncclMin, h->comm, h->st_comm));
    CK(cudaEventRecord(h->ev_y, h->st_comm));
    CK(cudaStreamWaitEvent(h->st, h->ev_y, 0));
    return GPB200_OK;
}


// ---- device-side signalling for the fused (peer-memory) panel broadcast --------------------------
__global__ void signal_peers_kernel(int* const* peer_sig_words, int n_peer, int value) {
    // all panel stores of the preceding kernels are complete (stream order); make them visible
    // system-wide before the flag
    __threadfence_system();
    if ((int)threadIdx.x < n_peer)
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(peer_sig_words[threadIdx.x]), "r"(value) : "memory");
}
__global__ void wait_signal_kernel(const int* word, int target, int* err) {
    long long spins = 0;
    int v;
    do {
        asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(word) : "memory");
        if (v >= target) break;
        if (++spins > (1LL << 27)) { atomicExch(err, 1); break; }
        __nanosleep(100);
    } while (true);
}

// Cholesky over block columns with the panel broadcast FUSED into the kernels that produce the panel:
// the tile leaf and the 128-wide TRSM GEMM store their outputs into every peer's F / Dinv / DinvT / logd
// through NVLink-mapped pointers (CUDA IPC), then one tiny kernel raises a flag word in each peer; the
// peers' streams wait on that word with a one-thread kernel.  No staging copy, no NCCL on the panel path.
int cholesky_dist_p2p(gpb200_handle* h) {
    const int Np = (int)h->Npad, R = h->nranks, me = h->rank;
    const int NB = dist_block(h);
    const int nblk = (Np + NB - 1) / NB;
    auto bp = [&](int b) { return b * NB; };
    auto bn = [&](int b) { return std::min(NB, Np - b * NB); };
    auto owner = [&](int b) { return b % R; };
    auto update = [&](int jb, int b) {
        const int r0 = bp(jb);
        return schur_update(h, r0, Np - r0, bn(jb), bp(b), bn(b));
    };
    // start barrier: no rank may push a new panel into a peer's factor while that peer still reads the
    // previous evaluation's factor (inverse / predict); also makes the rare epoch wrap safe
    if (++h->epoch >= 32000) { h->epoch = 1; CK(cudaMemsetAsync(h->sig, 0, sizeof(int) * 8, h->st)); }
    const int base = h->epoch * 65536;
    CK(cudaEventRecord(h->ev_x, h->st));
    CK(cudaStreamWaitEvent(h->st_comm, h->ev_x, 0));
    CKN(g_nccl.AllReduce(h->sig + 12, h->sig + 12, 1, ncclInt32, ncclSum, h->comm, h->st_comm));
    CK(cudaEventRecord(h->ev_y, h->st_comm));
    CK(cudaStreamWaitEvent(h->st, h->ev_y, 0));
    auto factor_and_publish = [&](int b) -> int {
        h->push_panel = true;
        cudaError_t e = chol_panel(h, bp(b), bn(b), NB);
        h->push_panel = false;
        CK(e);
        ++h->launches;
        signal_peers_kernel<<<1, 32, 0, h->st>>>(h->peer_sig_dev, h->n_peer, base + b + 1);
        CK(cudaGetLastError());
        return GPB200_OK;
    };
    if (owner(0) == me) { int rc = factor_and_publish(0); if (rc) return rc; }
    for (int b = 0; b < nblk; ++b) {
        if (owner(b) != me) {
            ++h->launches;
            wait_signal_kernel<<<1, 1, 0, h->st>>>(h->sig + owner(b), base + b + 1, h->sig + 8);
            CK(cudaGetLastError());
        }
        bool did_next = false;
        if (b + 1 < nblk && owner(b + 1) == me) {
            CK(update(b + 1, b));
            int rc = factor_and_publish(b + 1);
            if (rc) return rc;
            did_next = true;
        }
        for (int jb = b + 1 + (did_next ? 1 : 0); jb < nblk; ++jb)
            if (owner(jb) == me) CK(update(jb, b));
    }
    // first failing pivot over all ranks; also the barrier that keeps the next evaluation from overwriting
    // a panel a slower peer is still reading
    CK(cudaEventRecord(h->ev_x, h->st));
    CK(cudaStreamWaitEvent(h->st_comm, h->ev_x, 0));
    CKN(g_nccl.AllReduce(h->info_dev, h->info_dev, 1, ncclInt32, ncclMin, h->comm, h->st_comm));
    CK(cudaEventRecord(h->ev_y, h->st_comm));
    CK(cudaStreamWaitEvent(h->st, h->ev_y, 0));
    return GPB200_OK;
}

int inverse_dist(gpb200_handle* h) {
    const int Np = (int)h->Npad, R = h->nranks, me = h->rank;
    for (long long s = TILE; s < Np; s *= 2) {
        const int batch = (int)((Np + 2 * s - 1) / (2 * s));
        const int n2 = (int)((Np - s < s) ? Np - s : s);
        const int tiles = (int)(s / TILE);
        if (tiles < R || tiles % R) {                        // small level: recompute everywhere
            CK(merge_inverse(h, 0, (int)s, n2, batch));
            continue;
        }
        const int wr = (int)(s / R);
        const int lim = Np - (int)s;
        {   // T'[own tile rows, :] = Wt_A[own tile rows, :] * L21'
            GemmDesc g = gemm_desc_default();
            g.A = GemmOperand{bufG(h), bufDinvT(h), 0, 0};
            g.B = GemmOperand{bufF(h), bufNone(), (int)s, 0};
            g.C = h->F; g.ldc = h->ld; g.c_row0 = 0; g.c_col0 = (int)s;
            g.M = (int)s; g.N = n2; g.K = (int)s;
            g.flags = GEMM_KLO_M;
            g.bm_mod = R; g.bm_rem = me;
            g.batch = batch; g.zstep = 2 * (int)s; g.n_lim = lim;
            CK(launch_gemm(h, g));
        }
        {   // W21[:, own tile columns] = -W_C * (T'[own tile rows, :])'
            GemmDesc g = gemm_desc_default();
            g.A = GemmOperand{bufG(h), bufDinv(h), (int)s, (int)s};
            g.B = GemmOperand{bufF(h), bufNone(), 0, (int)s};
            g.C = h->G; g.ldc = h->ld; g.c_row0 = (int)s; g.c_col0 = 0;
            g.Ct = h->G; g.ldct = h->ld; g.ct_row0 = 0; g.ct_col0 = (int)s;
            g.M = n2; g.N = (int)s; g.K = n2;
            g.alpha = -1.0; g.flags = GEMM_KHI_M;
            g.bn_mod = R; g.bn_rem = me;
            g.batch = batch; g.zstep = 2 * (int)s; g.m_lim = lim; g.k_lim = lim;
            CK(launch_gemm(h, g));
        }
        // exchange the column slices
        long long rows_total = 0;                                   // sum over problems of n2_z (only the last is short)
        for (int z = 0; z < batch; ++z) rows_total += std::max(0LL, std::min((long long)s, (long long)Np - z * 2 * s - s));
        const long long per_rank = rows_total * wr;
        if ((size_t)per_rank > h->ag_send_elems || (size_t)per_rank * R > h->ag_recv_elems)
            return fail(h, GPB200_ECUDA, "inverse_dist: exchange buffers too small");
        dim3 blk(32, 32), grd((wr + 31) / 32, (unsigned)((s + 31) / 32), (unsigned)batch);
        h->launches += 2;
        pack_slices_kernel<<<grd, blk, 0, h->st>>>(h->G, h->ld, h->ag_send, (int)s, wr, R, me, Np);
        CK(cudaGetLastError());
        CK(cudaEventRecord(h->ev_x, h->st));
        CK(cudaStreamWaitEvent(h->st_comm, h->ev_x, 0));
        CKN(g_nccl.AllGather(h->ag_send, h->ag_recv, (size_t)per_rank, ncclDouble, h->comm, h->st_comm));
        CK(cudaEventRecord(h->ev_y, h->st_comm));
        CK(cudaStreamWaitEvent(h->st, h->ev_y, 0));
        dim3 grd2((wr + 31) / 32, (unsigned)((s + 31) / 32), (unsigned)(batch * R));
        unpack_slices_kernel<<<grd2, blk, 0, h->st>>>(h->G, h->ld, h->ag_recv, per_rank, (int)s, wr, Np, R, me);
        CK(cudaGetLastError());
    }
    // W'W on this rank's tile rows only (K^-1 stays distributed; the trace needs no more)
    GemmDesc g = gemm_desc_default();
    g.A = GemmOperand{bufG(h), bufDinvT(h), 0, 0};
    g.B = GemmOperand{bufG(h), bufDinvT(h), 0, 0};
    g.C = h->G; g.ldc = h->ld; g.c_row0 = 0; g.c_col0 = 0;
    g.M = Np; g.N = Np; g.K = Np;
    g.flags = GEMM_LOWER_ONLY | GEMM_KLO_M;
    g.bm_mod = R; g.bm_rem = me;
    CK(launch_gemm(h, g));
    return GPB200_OK;
}

// alpha-type solve on device vectors: out = K_y^-1 rhs ; rhs (Npad, zero padded) is destroyed
cudaError_t solve_device(gpb200_handle* h, double* rhs, double* tmp, double* out) {
    const int nb = (int)(h->Npad / TILE);
    // single-launch flag-synchronised solves need all Npad/128 CTAs co-resident (8 CTAs of 256 threads per SM)
    if (h->trsv_fused && h->flags && nb <= h->max_resident_ctas) {
        cudaError_t e = trsv_lower_fwd_fused(h->F, h->ld, h->Dinv, rhs, tmp, h->Npad, h->flags, h->st, &h->launches);
        if (e != cudaSuccess) return e;
        return trsv_lower_bwd_fused(h->F, h->ld, h->DinvT, tmp, out, h->Npad, h->flags + nb + 1, h->st, &h->launches);
    }
    cudaError_t e = trsv_lower_fwd(h->F, h->ld, h->Dinv, rhs, tmp, h->Npad, h->st, &h->launches);
    if (e != cudaSuccess) return e;
    return trsv_lower_bwd(h->F, h->ld, h->DinvT, tmp, out, h->Npad, h->st, &h->launches);
}

// after a stream sync: did the watchdog of the single-launch solves fire?
int check_trsv_watchdog(gpb200_handle* h) {
    if (!h->trsv_fused || !h->flags) return GPB200_OK;
    const int nb = (int)(h->Npad / TILE);
    if (nb > h->max_resident_ctas) return GPB200_OK;
    int e[2] = {0, 0};
    CK(cudaMemcpy(&e[0], h->flags + nb, sizeof(int), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&e[1], h->flags + 2 * nb + 1, sizeof(int), cudaMemcpyDeviceToHost));
    if (e[0] || e[1]) return fail(h, GPB200_ECUDA, "triangular solve watchdog fired (a ready-flag never arrived)");
    return GPB200_OK;
}

int upload_padded(gpb200_handle* h, double* dst, const double* src_host) {
    CK(cudaMemsetAsync(dst, 0, sizeof(double) * h->Npad, h->st));
    CK(cudaMemcpyAsync(dst, src_host, sizeof(double) * h->N, cudaMemcpyHostToDevice, h->st));
    return GPB200_OK;
}

int ensure_predict_ws(gpb200_handle* h, int64_t Mc, bool want_cov) {
    const int64_t Mpad = (Mc + TILE - 1) / TILE * TILE;
    if (Mpad > h->xs_cap) {
        if (h->xs) cudaFree(h->xs);
        if (h->pmu) cudaFree(h->pmu);
        if (h->pvar) cudaFree(h->pvar);
        if (h->pkdiag) cudaFree(h->pkdiag);
        h->xs = h->pmu = h->pvar = h->pkdiag = nullptr; h->xs_cap = 0;
        CK(cudaMalloc(&h->xs, sizeof(double) * Mpad * h->d));
        CK(cudaMalloc(&h->pmu, sizeof(double) * Mpad));
        CK(cudaMalloc(&h->pvar, sizeof(double) * Mpad));
        CK(cudaMalloc(&h->pkdiag, sizeof(double) * Mpad));
        h->xs_cap = Mpad;
    }
    if (Mpad > h->Kst_rows) {
        if (h->Kst) cudaFree(h->Kst);
        h->Kst = nullptr; h->Kst_rows = 0;
        CK(cudaMalloc(&h->Kst, sizeof(double) * Mpad * h->Npad));
        h->Kst_rows = Mpad;
        if (h->tma_ok && !gemm_make_tensor_map(&h->mapKst, h->Kst, Mpad, h->Npad, h->Npad))
            return fail(h, GPB200_ECUDA, "cuTensorMapEncodeTiled failed for the predict buffer");
    }
    if (want_cov && Mpad > h->Kss_rows) {
        if (h->Kss) cudaFree(h->Kss);
        h->Kss = nullptr; h->Kss_rows = 0;
        CK(cudaMalloc(&h->Kss, sizeof(double) * Mpad * Mpad));
        h->Kss_rows = Mpad;
    }
    return GPB200_OK;
}

// Vt[:, c0..c0+n) <- solve against L[c0.., c0..] of handle h, in place on a row-major buffer
// (`rows` x h->Npad, leading dimension ldk): recursive blocked TRSM, leaves multiply by the inverted
// 128-tile, updates are NT GEMMs.  (whiten!, PDMats: x <- U^-T x.)
cudaError_t trsm_rec_buf(gpb200_handle* h, GemmBuf bk, int rows, int c0, int n) {
    double* kb = const_cast<double*>(bk.base);
    if (n == TILE) {
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bk, bufNone(), 0, c0};
        g.B = GemmOperand{bufDinv(h), bufNone(), c0, 0};
        g.C = kb; g.ldc = bk.ld; g.c_row0 = 0; g.c_col0 = c0;
        g.M = rows; g.N = TILE; g.K = TILE;
        return launch_gemm(h, g);
    }
    int n1 = TILE;
    while (n1 * 2 < n) n1 *= 2;
    const int n2 = n - n1;
    cudaError_t e;
    if ((e = trsm_rec_buf(h, bk, rows, c0, n1)) != cudaSuccess) return e;
    {
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bk, bufNone(), 0, c0};
        g.B = GemmOperand{bufF(h), bufNone(), c0 + n1, c0};
        g.C = kb; g.ldc = bk.ld; g.c_row0 = 0; g.c_col0 = c0 + n1;
        g.M = rows; g.N = n2; g.K = n1;
        g.alpha = -1.0; g.beta = 1.0;
        if ((e = launch_gemm(h, g)) != cudaSuccess) return e;
    }
    return trsm_rec_buf(h, bk, rows, c0 + n1, n2);
}
cudaError_t trsm_rec(gpb200_handle* h, int Mpad, int c0, int n) {
    GemmBuf bk{h->tma_ok ? &h->mapKst : nullptr, h->Kst, h->Npad};
    return trsm_rec_buf(h, bk, Mpad, c0, n);
}

// factor whatever SPD matrix sits in the lower tiles of h->G (padding must be identity)
int chol_inplace(gpb200_handle* h) {
    h->factored = h->inv_ready = h->alpha_ready = h->chol_bar_ready = false;
    const int init = INT_MAX;
    CK(cudaMemcpyAsync(h->info_dev, &init, sizeof(int), cudaMemcpyHostToDevice, h->st));
    CK(cholesky(h));
    int info = 0;
    CK(cudaMemcpyAsync(&info, h->info_dev, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    if (info != INT_MAX) {
        char buf[128];
        snprintf(buf, sizeof buf, "matrix is not positive definite; leading minor %d", info);
        h->err = buf;
        return info > h->N ? (int)h->N : info;
    }
    h->factored = true;
    return GPB200_OK;
}

float ev_ms(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

// Gram build / gradient trace dispatch: the TMA-staged SEIso kernels (gram_fast.cu) when the kernel program is the single
// SEIso leaf over all (<= 8) input dimensions, else the generic kernel-program kernels (gram.cu)
bool use_seiso_fast(gpb200_handle* h, SeIsoFast* sf) {
    return h->gram_fast && h->prog.fast && h->xmap_ok && h->xp && seiso_fast_prepare(h->prog.par[0], h->prog.par[1], sf);
}
cudaError_t launch_gram(gpb200_handle* h, double* G, int64_t ldg, int own_tiles, int nranks, int rank, int own_axis) {
    SeIsoFast sf;
    if (use_seiso_fast(h, &sf))
        return gram_seiso_tma_launch(&h->mapX, &h->mapXT, h->dxp, sf, h->N, h->Npad, h->noise_var, h->n_noise, h->nugget, G, ldg, h->st,
                                     own_tiles, nranks, rank, own_axis);
    return gram_lower_launch(h->prog, h->x, h->d, h->d, h->N, h->Npad, h->noise_var, h->n_noise, h->nugget, G, ldg, h->st,
                             own_tiles, nranks, rank, own_axis);
}
cudaError_t launch_trace(gpb200_handle* h, int bm_mod, int bm_rem, int bm_div) {
    SeIsoFast sf;
    if (use_seiso_fast(h, &sf))
        return trace_seiso_tma_launch(&h->mapX, &h->mapXT, h->dxp, sf, h->N, h->Npad, h->alpha, h->G, h->ld, h->part, h->trace_out, h->st,
                                      bm_mod, bm_rem, bm_div);
    return trace_launch(h->prog, h->x, h->d, h->d, h->N, h->Npad, h->alpha, h->G, h->ld, h->part, h->trace_out, h->st,
                        bm_mod, bm_rem, bm_div);
}

#include "shard_impl.cuh"

// collective entry points of a sharded handle: in an in-process group they must be called on the leader (it drives every
// virtual rank); per-rank state (host arguments) is replicated to every local handle here
int shard_entry(gpb200_handle* h, Locals& L) {
    L = locals(h);
    if (h->grp && L[0] != h) return fail(h, GPB200_ESTATE, "in-process group: call collective entry points on the leader (rank 0) handle");
    return GPB200_OK;
}
// debug getters with sharded storage: rows this rank owns, zeros elsewhere (the caller adds the ranks' pieces)
int copy_own_rows(gpb200_handle* h, double* dst_host, const double* src_dev) {
    const int64_t N = h->N;
    memset(dst_host, 0, sizeof(double) * (size_t)N * (size_t)N);
    for (int64_t t = 0; t * TILE < N; ++t) {
        if (owner_of_tile(h, t) != h->rank) continue;
        const int64_t r0 = t * TILE, nr = std::min<int64_t>(TILE, N - r0);
        CK(cudaMemcpy2DAsync(dst_host + r0 * N, sizeof(double) * N, src_dev + r0 * h->ld, sizeof(double) * h->ld, sizeof(double) * N, nr,
                             cudaMemcpyDeviceToHost, h->st));
    }
    return GPB200_OK;
}
int sync_all(const Locals& L) {
    for (auto* q : L) SCK(q, cudaStreamSynchronize(q->st));
    return GPB200_OK;
}

// latent-GP entry points: single-GPU handles with a resident factor; lazily sized workspace
int gpa_entry(gpb200_handle* h, const char* who) {
    char buf[160];
    if (h->nranks > 1 || h->sharded || h->grp) {
        snprintf(buf, sizeof buf, "%s: GPA runs on single-GPU handles only (not on replicated or row-sharded multi-rank storage)", who);
        return fail(h, GPB200_EINVAL, buf);
    }
    if (!h->factored) { snprintf(buf, sizeof buf, "%s: factorize first", who); return fail(h, GPB200_ESTATE, buf); }
    CK(cudaSetDevice(h->device));
    if (h->gpa_npad == h->Npad) return GPB200_OK;
    if (h->Zd) cudaFree(h->Zd);
    if (h->gpa_part) cudaFree(h->gpa_part);
    h->Zd = h->gpa_part = nullptr; h->gpa_npad = 0;
    CK(cudaMalloc(&h->Zd, sizeof(double) * (size_t)h->Npad * TILE));
    CK(cudaMalloc(&h->gpa_part, sizeof(double) * (size_t)(h->Npad / TILE) * (size_t)h->Npad));
    if (h->tma_ok && !gemm_make_tensor_map(&h->mapZd, h->Zd, h->Npad, TILE, TILE))
        return fail(h, GPB200_ECUDA, "cuTensorMapEncodeTiled failed for the GPA diagonal-tile buffer");
    for (auto& e : h->ev_gpa) if (!e) CK(cudaEventCreate(&e));
    h->gpa_npad = h->Npad;
    return GPB200_OK;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int gpb200_version(void) { return 100; }

const char* gpb200_last_error(gpb200_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int gpb200_create(gpb200_handle** out, int device) {
    if (!out) return GPB200_EINVAL;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) {
        g_create_error = std::string("no CUDA device available (") + cudaGetErrorString(e) +
                         "); libgpb200 has no CPU fallback";
        (void)cudaGetLastError();
        return GPB200_ECUDA;
    }
    if (device < 0 || device >= count) { g_create_error = "device index out of range"; return GPB200_EINVAL; }
    gpb200_handle* h = new gpb200_handle();
    h->device = device;
    auto bail = [&](const char* what, cudaError_t ce) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(ce);
        delete h;
        return GPB200_ECUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    if ((e = cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    cudaEventCreate(&h->ev0); cudaEventCreate(&h->ev1); cudaEventCreate(&h->ev2); cudaEventCreate(&h->ev3);
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&h->st_side, cudaStreamNonBlocking, hi) != cudaSuccess) { h->st_side = nullptr; (void)cudaGetLastError(); }
        cudaEventCreateWithFlags(&h->ev_la0, cudaEventDisableTiming);
        cudaEventCreateWithFlags(&h->ev_la2, cudaEventDisableTiming);
    }
    if ((e = gemm_nt_init()) != cudaSuccess) return bail("gemm_nt_init", e);
    const char* env = getenv("GPB200_GEMM");
    if (env) h->gemm_impl = atoi(env);
    env = getenv("GPB200_DIST_NB");
    if (env) { int v = atoi(env); if (v == 128 || v == 256 || v == 512 || v == 1024 || v == 2048 || v == 4096) h->dist_nb = v; }
    env = getenv("GPB200_SHARD_LA");
    if (env) h->shard_la = atoi(env) ? 1 : 0;
    env = getenv("GPB200_SHARD_RB");
    if (env) { int v = atoi(env); if (v == 1 || v == 2 || v == 4 || v == 8) h->shard_rb_opt = v; }
    env = getenv("GPB200_NB");
    if (env) { int v = atoi(env); if (v == 0 || v == 128 || v == 256 || v == 512 || v == 1024 || v == 2048 || v == 4096) h->nb = v; }
    *out = h;
    return GPB200_OK;
}

void gpb200_destroy(gpb200_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->grp) {                              // a group dissolves with its first destroyed member
        gpb200_group* g = h->grp;
        for (auto* m : g->hs) { if (m->st) cudaStreamSynchronize(m->st); }
        for (auto* m : g->hs) {                 // the survivors become ordinary single-rank handles (storage re-allocated at their next factorize)
            m->grp = nullptr; m->nranks = 1; m->rank = 0;
            m->factored = m->inv_ready = m->alpha_ready = false;
        }
        delete g;
    }
    if (h->st) cudaStreamSynchronize(h->st);
    if (h->sub) { h->sub->st = nullptr; h->sub->own_stream = false; gpb200_destroy(h->sub); h->sub = nullptr; }
    if (h->rz) cudaFree(h->rz);
    if (h->rout) cudaFree(h->rout);
    free_data(h);
    for (auto e : h->evring) cudaEventDestroy(e);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev2) cudaEventDestroy(h->ev2);
    if (h->ev3) cudaEventDestroy(h->ev3);
    if (h->ev_la0) cudaEventDestroy(h->ev_la0);
    if (h->ev_la2) cudaEventDestroy(h->ev_la2);
    for (auto e : h->ev_gpa) if (e) cudaEventDestroy(e);
    if (h->st_side) cudaStreamDestroy(h->st_side);
    for (auto e : h->pev) cudaEventDestroy(e);
    if (h->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(h->comm);
    for (int i = 0; i < 2; ++i) {
        if (h->ev_packed[i]) cudaEventDestroy(h->ev_packed[i]);
        if (h->ev_bcast[i]) cudaEventDestroy(h->ev_bcast[i]);
        if (h->ev_unpacked[i]) cudaEventDestroy(h->ev_unpacked[i]);
    }
    if (h->ev_x) cudaEventDestroy(h->ev_x);
    if (h->ev_y) cudaEventDestroy(h->ev_y);
    if (h->st_comm) cudaStreamDestroy(h->st_comm);
    if (h->st && h->own_stream) cudaStreamDestroy(h->st);
    delete h;
}

int gpb200_set_option(gpb200_handle* h, const char* key, int64_t value) {
    if (!h || !key) return GPB200_EINVAL;
    if (!strcmp(key, "nb")) {
        if (value != 0 && value != 128 && value != 256 && value != 512 && value != 1024 && value != 2048 && value != 4096)
            return fail(h, GPB200_EINVAL, "nb must be 0 (fully recursive) or 128 * 2^k <= 4096");
        h->nb = (int)value; h->factored = h->inv_ready = false; return GPB200_OK;
    }
    if (!strcmp(key, "gemm")) { h->gemm_impl = value ? 1 : 0; return GPB200_OK; }
    if (!strcmp(key, "dist_nb")) {
        if (value != 0 && value != 128 && value != 256 && value != 512 && value != 1024 && value != 2048 && value != 4096)
            return fail(h, GPB200_EINVAL, "dist_nb must be 0 (auto) or 128 * 2^k <= 4096");
        h->dist_nb = (int)value; h->factored = h->inv_ready = false; return GPB200_OK;
    }
    if (!strcmp(key, "lookahead")) { h->lookahead = value ? 1 : 0; return GPB200_OK; }
    if (!strcmp(key, "gram_fast")) { h->gram_fast = value ? 1 : 0; return GPB200_OK; }
    if (!strcmp(key, "leaf")) { potrf128_set_variant(value != 0); h->factored = h->inv_ready = false; return GPB200_OK; }
    if (!strcmp(key, "capacity")) {             // rows reserved by the next gpb200_set_data (>= N): room for gpb200_append
        if (value < 0 || value > ((int64_t)1 << 30)) return fail(h, GPB200_EINVAL, "capacity out of range");
        h->capacity = value; return GPB200_OK;
    }
    if (!strcmp(key, "shard")) {                // storage of F / G with several ranks: -1 auto, 0 replicated, 1 row-sharded
        if (value < -1 || value > 1) return fail(h, GPB200_EINVAL, "shard must be -1 (auto), 0 or 1");
        h->shard_opt = (int)value; h->factored = h->inv_ready = false; return GPB200_OK;
    }
    if (!strcmp(key, "shard_la")) { h->shard_la = value ? 1 : 0; return GPB200_OK; }
    if (!strcmp(key, "shard_rb")) {             // ownership block of the row-sharded storage in 128-row tiles (panel = 128 * rb)
        if (value != 0 && value != 1 && value != 2 && value != 4 && value != 8) return fail(h, GPB200_EINVAL, "shard_rb must be 0 (auto), 1, 2, 4 or 8");
        h->shard_rb_opt = (int)value; h->factored = h->inv_ready = false; return GPB200_OK;
    }
    if (!strcmp(key, "trsv_fused")) {            // 0: one launch per block step; 1: round-1 single-launch kernels; 2 (default): resident-tile kernels
        if (value < 0 || value > 2) return fail(h, GPB200_EINVAL, "trsv_fused must be 0, 1 or 2");
        h->trsv_fused = value ? 1 : 0;
        if (value) trsv_set_variant((int)value);
        return GPB200_OK;
    }
    if (!strcmp(key, "p2p")) {                 // 0: NCCL panel broadcast even if peer memory is mapped
        if (value && h->n_peer == 0) return fail(h, GPB200_ESTATE, "p2p: ipc_import first");
        h->p2p = value != 0; return GPB200_OK;
    }
    if (!strcmp(key, "profile")) {
        h->profile = value ? 1 : 0;
        h->ms[6] = h->ms[7] = h->ms[8] = 0.0;
        h->pev_used = 0; h->gemm_flops_exec = 0.0; h->gemm_launches = 0;
        return GPB200_OK;
    }
    return fail(h, GPB200_EINVAL, "unknown option");
}

int64_t gpb200_launch_count(gpb200_handle* h) { return h ? h->launches : 0; }

int gpb200_set_stream(gpb200_handle* h, void* stream) {
    if (!h) return GPB200_EINVAL;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->st));
    if (h->own_stream && h->st) cudaStreamDestroy(h->st);
    if (stream) { h->st = (cudaStream_t)stream; h->own_stream = false; }
    else {
        h->st = nullptr;
        CK(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking));
        h->own_stream = true;
    }
    return GPB200_OK;
}

int gpb200_get_timings(gpb200_handle* h, double* ms, int32_t n) {
    if (!h || !ms) return GPB200_EINVAL;
    for (int i = 0; i < n && i < 16; ++i) ms[i] = h->ms[i];
    return GPB200_OK;
}

int gpb200_set_data(gpb200_handle* h, int64_t N, int32_t d, const double* x, int64_t ldx) {
    if (!h) return GPB200_EINVAL;
    if (N <= 0 || d <= 0 || !x || ldx < d) return fail(h, GPB200_EINVAL, "set_data: bad N, d, x or ldx");
    if (d > GPB200_MAX_DIMS) return fail(h, GPB200_EINVAL, "set_data: d exceeds GPB200_MAX_DIMS");
    if (N > (int64_t)1 << 30) return fail(h, GPB200_EINVAL, "set_data: N too large");
    CK(cudaSetDevice(h->device));
    const int64_t Npad = (std::max<int64_t>(N, h->capacity) + TILE - 1) / TILE * TILE;
    const bool realloc = !h->has_data || Npad != h->Npad || d != h->d;
    if (realloc) {
        free_data(h);
        h->N = N; h->Npad = Npad; h->ld = Npad; h->d = d;
        CK(cudaMalloc(&h->x, sizeof(double) * Npad * d));      // Npad rows: N may grow up to Npad without realloc
        CK(cudaMalloc(&h->Dinv, sizeof(double) * Npad * TILE));
        CK(cudaMalloc(&h->DinvT, sizeof(double) * Npad * TILE));
        const size_t nv = sizeof(double) * Npad;
        CK(cudaMalloc(&h->logd, nv)); CK(cudaMalloc(&h->noise_var, nv)); CK(cudaMalloc(&h->r0, nv));
        CK(cudaMalloc(&h->r1, nv)); CK(cudaMalloc(&h->y1, nv)); CK(cudaMalloc(&h->alpha, nv)); CK(cudaMalloc(&h->tblk, nv));
        CK(cudaMalloc(&h->scal, sizeof(double) * 16));
        CK(cudaMalloc(&h->info_dev, sizeof(int)));
        CK(cudaMalloc(&h->flags, sizeof(int) * 2 * (Npad / TILE + 1)));
        CK(cudaMalloc(&h->sig, sizeof(int) * 16));
        CK(cudaMemsetAsync(h->sig, 0, sizeof(int) * 16, h->st));
        {
            int sms = 0;
            CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
            h->max_resident_ctas = sms * 4;            // conservative: 4 CTAs of 256 threads per SM
        }
        const int64_t T = Npad / TILE;
        CK(cudaMalloc(&h->part, sizeof(double) * (size_t)(T * (T + 1) / 2) * (GPB200_MAX_THETA + 1)));
        CK(cudaMalloc(&h->trace_out, sizeof(double) * (GPB200_MAX_THETA + 1)));
        // F / G: replicated (cudaMalloc) or row-sharded (virtual range, owned rows mapped) -- decided by the communicator,
        // the problem size and option "shard"; re-checked at every factorize (the communicator may be joined later)
        int rc_fg = ensure_storage(h);
        if (rc_fg != GPB200_OK) return rc_fg;
    }
    h->N = N;
    // x arrives as Julia's d x N column-major (ld = ldx): point i is the contiguous run x[i*ldx .. +d)
    CK(cudaMemcpy2DAsync(h->x, sizeof(double) * d, x, sizeof(double) * ldx, sizeof(double) * d, N,
                         cudaMemcpyHostToDevice, h->st));
    // second copy with an even row length for the TMA-staged SEIso kernels (row pitch must be a multiple of 16 bytes)
    h->xmap_ok = false;
    if (d <= 8) {
        h->dxp = (d + 1) / 2 * 2;
        if (!h->xp) CK(cudaMalloc(&h->xp, sizeof(double) * Npad * h->dxp));
        CK(cudaMemsetAsync(h->xp, 0, sizeof(double) * Npad * h->dxp, h->st));
        CK(cudaMemcpy2DAsync(h->xp, sizeof(double) * h->dxp, x, sizeof(double) * ldx, sizeof(double) * d, N,
                             cudaMemcpyHostToDevice, h->st));
        if (!h->xpt) CK(cudaMalloc(&h->xpt, sizeof(double) * Npad * h->dxp));
        ++h->launches;
        CK(shard_transpose(h->xpt, Npad, h->xp, h->dxp, Npad, h->dxp, h->st));
        h->xmap_ok = gemm_make_tensor_map_plain(&h->mapX, h->xp, N, h->dxp, h->dxp, TILE, h->dxp) &&
                     gemm_make_tensor_map_plain(&h->mapXT, h->xpt, h->dxp, N, Npad, h->dxp, TILE);
    }
    CK(cudaStreamSynchronize(h->st));
    h->has_data = true;
    h->factored = h->inv_ready = h->alpha_ready = false;
    return GPB200_OK;
}

int gpb200_set_kernel(gpb200_handle* h, int32_t n_ops, const int32_t* ops, int32_t n_dims, const int32_t* dims,
                      int32_t n_theta) {
    if (!h) return GPB200_EINVAL;
    if (n_ops <= 0 || n_ops > GPB200_MAX_OPS || !ops) return fail(h, GPB200_EINVAL, "set_kernel: bad n_ops");
    if (n_theta < 0 || n_theta > GPB200_MAX_THETA) return fail(h, GPB200_EINVAL, "set_kernel: too many parameters");
    if (n_dims < 0 || n_dims > GPB200_MAX_DIMS || (n_dims > 0 && !dims)) return fail(h, GPB200_EINVAL, "set_kernel: bad dims");
    KProg P{};
    P.n_ops = n_ops; P.n_theta = n_theta;
    int stack[GPB200_MAX_OPS]; int sp = 0; int tcount = 0;
    for (int q = 0; q < n_ops; ++q) {
        const int32_t* o = ops + q * GPB200_OP_STRIDE;
        P.op[q] = o[0]; P.toff[q] = o[1]; P.nth[q] = o[2]; P.doff[q] = o[3]; P.nd[q] = o[4]; P.extra[q] = o[5];
        if (o[0] == GPB200_OP_SUM || o[0] == GPB200_OP_PROD) {
            if (sp < 2) return fail(h, GPB200_EINVAL, "set_kernel: malformed program (stack underflow)");
            const int right = stack[--sp]; const int left = stack[--sp];
            if (right != q - 1) return fail(h, GPB200_EINVAL, "set_kernel: program is not in post-order");
            P.left[q] = left; P.nth[q] = 0;
            stack[sp++] = q;
        } else {
            if (o[0] < GPB200_OP_SE_ISO || o[0] > GPB200_OP_CONST) return fail(h, GPB200_EINVAL, "set_kernel: unknown opcode");
            if (o[1] < 0 || o[2] < 0 || o[1] + o[2] > n_theta) return fail(h, GPB200_EINVAL, "set_kernel: theta range");
            if (o[3] < 0 || o[4] < 0 || o[3] + o[4] > n_dims) return fail(h, GPB200_EINVAL, "set_kernel: dims range");
            int expect = -1;
            switch (o[0]) {
            case GPB200_OP_SE_ISO: case GPB200_OP_MAT12_ISO: case GPB200_OP_MAT32_ISO: case GPB200_OP_MAT52_ISO:
            case GPB200_OP_POLY: expect = 2; break;
            case GPB200_OP_SE_ARD: case GPB200_OP_MAT12_ARD: case GPB200_OP_MAT32_ARD: case GPB200_OP_MAT52_ARD:
                expect = o[4] + 1; break;
            case GPB200_OP_RQ_ISO: case GPB200_OP_PERIODIC: expect = 3; break;
            case GPB200_OP_RQ_ARD: expect = o[4] + 2; break;
            case GPB200_OP_LIN_ISO: case GPB200_OP_NOISE: case GPB200_OP_CONST: expect = 1; break;
            case GPB200_OP_LIN_ARD: expect = o[4]; break;
            }
            if (o[2] != expect) return fail(h, GPB200_EINVAL, "set_kernel: wrong parameter count for a leaf");
            tcount += o[2];
            stack[sp++] = q;
        }
    }
    if (sp != 1 || tcount != n_theta) return fail(h, GPB200_EINVAL, "set_kernel: malformed program");
    for (int i = 0; i < n_dims; ++i) {
        if (dims[i] < 0 || (h->has_data && dims[i] >= h->d)) return fail(h, GPB200_EINVAL, "set_kernel: dim index out of range");
        P.dims[i] = dims[i];
    }
    // single SEIso leaf over dims 0..nd-1 == the whole input: specialised kernels
    P.fast = 0;
    if (n_ops == 1 && P.op[0] == GPB200_OP_SE_ISO && h->has_data && P.nd[0] == h->d) {
        bool ident = true;
        for (int i = 0; i < P.nd[0]; ++i) ident = ident && (P.dims[P.doff[0] + i] == i);
        P.fast = ident ? 1 : 0;
    }
    h->prog = P;
    h->theta.assign(n_theta, 0.0);
    h->has_kernel = true;
    h->factored = h->inv_ready = false;
    return GPB200_OK;
}

int gpb200_factorize(gpb200_handle* h, const double* theta, const double* log_noise, int64_t n_noise,
                     double extra_nugget) {
    if (!h) return GPB200_EINVAL;
    if (!h->has_data || !h->has_kernel) return fail(h, GPB200_ESTATE, "factorize: set_data and set_kernel first");
    if ((h->prog.n_theta > 0 && !theta) || !log_noise) return fail(h, GPB200_EINVAL, "factorize: null theta/log_noise");
    if (n_noise != 1 && n_noise != h->N) return fail(h, GPB200_EINVAL, "factorize: n_noise must be 1 or N");
    for (int i = 0; i < h->prog.n_theta; ++i)
        if (!isfinite(theta[i])) return fail(h, GPB200_EINVAL, "factorize: non-finite hyper-parameter");
    CK(cudaSetDevice(h->device));
    h->factored = h->inv_ready = h->alpha_ready = false; h->g_sym = false; h->cv_m_ok = false; h->chol_bar_ready = false;
    std::vector<double> nv((size_t)n_noise);
    for (int64_t i = 0; i < n_noise; ++i) {
        if (!isfinite(log_noise[i])) return fail(h, GPB200_EINVAL, "factorize: non-finite logNoise");
        nv[i] = exp(2.0 * log_noise[i]);
    }
    Locals L;
    { int rc = shard_entry(h, L); if (rc) return rc; }
    for (auto* q : L) { int rc = ensure_storage(q); if (rc) { if (q != h) h->err = q->err; return rc; } }
    const int init = INT_MAX;
    for (auto* q : L) {                                    // (an in-process group: every virtual rank gets the arguments)
        if (!q->has_data || !q->has_kernel || q->prog.n_theta != h->prog.n_theta || q->N != h->N)
            return fail(h, GPB200_ESTATE, "factorize: every handle of the group needs the same set_data / set_kernel");
        q->factored = q->inv_ready = q->alpha_ready = false;
        for (int i = 0; i < q->prog.n_theta; ++i) q->theta[i] = theta[i];
        kprog_set_theta(q->prog, theta);
        SCK(q, cudaMemcpyAsync(q->noise_var, nv.data(), sizeof(double) * n_noise, cudaMemcpyHostToDevice, q->st));
        q->n_noise = n_noise; q->nugget = extra_nugget;
        SCK(q, cudaMemcpyAsync(q->info_dev, &init, sizeof(int), cudaMemcpyHostToDevice, q->st));
    }
    if (h->sharded) {
        // row-sharded storage: own rows of the Gram matrix, then the all-gathered-panel Cholesky (shard_impl.cuh)
        CK(cudaEventRecord(h->ev0, h->st));
        for (auto* q : L) {
            ++q->launches;
            SCK(q, launch_gram(q, q->G, q->ld, q->rb, q->nranks, q->rank, 1));
        }
        CK(cudaEventRecord(h->ev1, h->st));
        { int rc = h->shard_la ? shard_cholesky_la(L) : shard_cholesky(L); if (rc) { if (L[0] != h) h->err = L[0]->err; return rc; } }
        CK(cudaEventRecord(h->ev2, h->st));
        int info_s = 0;
        CK(cudaMemcpyAsync(&info_s, h->info_dev, sizeof(int), cudaMemcpyDeviceToHost, h->st));
        { int rc = sync_all(L); if (rc) return rc; }
        for (auto* q : L) profile_collect(q);
        h->ms[0] = ev_ms(h->ev0, h->ev1);
        h->ms[1] = ev_ms(h->ev1, h->ev2);
        if (info_s != INT_MAX) {
            char buf[128];
            snprintf(buf, sizeof buf, "matrix is not positive definite; leading minor %d", info_s);
            h->err = buf;
            return info_s > h->N ? (int)h->N : info_s;
        }
        for (auto* q : L) q->factored = true;
        return GPB200_OK;
    }

    CK(cudaEventRecord(h->ev0, h->st));
    ++h->launches;
    if (h->nranks > 1) {
        int rc = dist_alloc(h);
        if (rc) return rc;
        const int NBd = dist_block(h);
        CK(launch_gram(h, h->G, h->ld, NBd / TILE, h->nranks, h->rank, 0));
        CK(cudaEventRecord(h->ev1, h->st));
        rc = h->p2p ? cholesky_dist_p2p(h) : cholesky_dist(h);
        if (rc) return rc;
    } else {
        CK(launch_gram(h, h->G, h->ld, 0, 1, 0, 0));
        CK(cudaEventRecord(h->ev1, h->st));
        CK(cholesky(h));
    }
    CK(cudaEventRecord(h->ev2, h->st));
    int info = 0;
    CK(cudaMemcpyAsync(&info, h->info_dev, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    h->ms[0] = ev_ms(h->ev0, h->ev1);
    h->ms[1] = ev_ms(h->ev1, h->ev2);
    if (h->p2p) {
        int wd = 0;
        CK(cudaMemcpy(&wd, h->sig + 8, sizeof(int), cudaMemcpyDeviceToHost));
        if (wd) return fail(h, GPB200_ECUDA, "panel signal watchdog fired (a peer never published its panel)");
    }
    if (info != INT_MAX) {
        char buf[128];
        snprintf(buf, sizeof buf, "matrix is not positive definite; leading minor %d", info);
        h->err = buf;
        return info > h->N ? (int)h->N : info;
    }
    h->factored = true;
    return GPB200_OK;
}

int gpb200_logdet(gpb200_handle* h, double* logdet) {
    if (!h || !logdet) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "logdet: factorize first");
    CK(cudaSetDevice(h->device));
    ++h->launches;
    CK(sum_launch(h->logd, h->Npad, h->scal, h->st));
    CK(cudaMemcpyAsync(logdet, h->scal, sizeof(double), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPB200_OK;
}

int gpb200_solve(gpb200_handle* h, const double* rhs, double* out) {
    if (!h || !rhs || !out) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "solve: factorize first");
    CK(cudaSetDevice(h->device));
    if (h->sharded) {
        Locals L;
        { int rc = shard_entry(h, L); if (rc) return rc; }
        for (auto* q : L) { int rc = upload_padded(q, q->r1, rhs); if (rc) return rc; }
        { int rc = shard_solve(L, &gpb200_handle::r1, &gpb200_handle::y1, &gpb200_handle::r0); if (rc) { if (L[0] != h) h->err = L[0]->err; return rc; } }
        CK(cudaMemcpyAsync(out, h->r0, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
        return sync_all(L);
    }
    int rc = upload_padded(h, h->r1, rhs);
    if (rc) return rc;
    CK(solve_device(h, h->r1, h->y1, h->r0));
    CK(cudaMemcpyAsync(out, h->r0, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return check_trsv_watchdog(h);
}

int gpb200_mll(gpb200_handle* h, const double* y_minus_mean, double* alpha, double* mll) {
    if (!h || !y_minus_mean || !mll) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "mll: factorize first");
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev0, h->st));
    Locals Ls;
    if (h->sharded) { int rc = shard_entry(h, Ls); if (rc) return rc; }
    int rc = upload_padded(h, h->r0, y_minus_mean);
    if (rc) return rc;
    if (h->sharded) {
        for (auto* q : Ls) if (q != h) { rc = upload_padded(q, q->r0, y_minus_mean); if (rc) return rc; }
        rc = shard_solve(Ls, &gpb200_handle::r0, &gpb200_handle::y1, &gpb200_handle::alpha);
        if (rc) { if (Ls[0] != h) h->err = Ls[0]->err; return rc; }
        for (auto* q : Ls) q->alpha_ready = true;
    } else {
        CK(cudaMemcpyAsync(h->r1, h->r0, sizeof(double) * h->Npad, cudaMemcpyDeviceToDevice, h->st));
        CK(solve_device(h, h->r1, h->y1, h->alpha));
    }
    h->launches += 2;
    CK(dot_launch(h->r0, h->alpha, h->Npad, h->scal + 0, h->st));
    CK(sum_launch(h->logd, h->Npad, h->scal + 1, h->st));
    double s[2];
    CK(cudaMemcpyAsync(s, h->scal, sizeof(double) * 2, cudaMemcpyDeviceToHost, h->st));
    if (alpha) CK(cudaMemcpyAsync(alpha, h->alpha, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaEventRecord(h->ev1, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (h->sharded) { int rcs = sync_all(Ls); if (rcs) return rcs; }
    h->ms[2] = ev_ms(h->ev0, h->ev1);
    if (!h->sharded) { int rcw = check_trsv_watchdog(h); if (rcw) return rcw; }
    *mll = -(s[0] + s[1] + LOG2PI * (double)h->N) / 2.0;    // src/GPE.jl:210
    h->alpha_ready = true;
    return GPB200_OK;
}

int gpb200_grad_prepare(gpb200_handle* h) {
    if (!h) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "grad_prepare: factorize first");
    if (h->inv_ready) return GPB200_OK;
    h->g_sym = false; h->cv_m_ok = false; h->chol_bar_ready = false;
    CK(cudaSetDevice(h->device));
    CK(cudaEventRecord(h->ev0, h->st));
    if (h->sharded) {
        Locals L;
        { int rc = shard_entry(h, L); if (rc) return rc; }
        { int rc = h->shard_la ? shard_inverse_la(L) : shard_inverse(L); if (rc) { if (L[0] != h) h->err = L[0]->err; return rc; } }
        CK(cudaEventRecord(h->ev1, h->st));
        { int rc = sync_all(L); if (rc) return rc; }
        for (auto* q : L) { profile_collect(q); q->inv_ready = true; }
        h->ms[3] = ev_ms(h->ev0, h->ev1);
        return GPB200_OK;
    }
    if (h->nranks > 1) { int rc = inverse_dist(h); if (rc) return rc; }
    else CK(inverse_from_factor(h));
    CK(cudaEventRecord(h->ev1, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    h->ms[3] = ev_ms(h->ev0, h->ev1);
    h->inv_ready = true;
    return GPB200_OK;
}

int gpb200_grad_kernel(gpb200_handle* h, const double* alpha, double* dmll_kernel, double* trA) {
    if (!h) return GPB200_EINVAL;
    if (!h->inv_ready) return fail(h, GPB200_ESTATE, "grad_kernel: grad_prepare first");
    if (!alpha && !h->alpha_ready) return fail(h, GPB200_ESTATE, "grad_kernel: no alpha (call mll or pass alpha)");
    CK(cudaSetDevice(h->device));
    Locals Lg;
    if (h->sharded) { int rc = shard_entry(h, Lg); if (rc) return rc; } else Lg = Locals{h};
    if (alpha) {
        for (auto* q : Lg) {
            int rc = upload_padded(q, q->alpha, alpha);
            if (rc) return rc;
            q->alpha_ready = true;
        }
    }
    CK(cudaEventRecord(h->ev0, h->st));
    if (h->sharded) {
        // fused trace over the own rows of K^-1 (block-cyclic tile rows), P+1 partial sums summed over the ranks
        for (auto* q : Lg) {
            q->launches += 2;
            SCK(q, launch_trace(q, q->nranks, q->rank, q->rb));
        }
        int rc = coll_allreduce_sum(Lg, [&](gpb200_handle* q) { return q->trace_out; }, (size_t)trace_num_acc(h->prog));
        if (rc) { if (Lg[0] != h) h->err = Lg[0]->err; return rc; }
    } else {
    h->launches += 2;
    CK(launch_trace(h, h->nranks, h->rank, 1));
    }
    if (!h->sharded && h->nranks > 1) {                    // P+1 partial sums, summed over ranks
        CK(cudaEventRecord(h->ev_x, h->st));
        CK(cudaStreamWaitEvent(h->st_comm, h->ev_x, 0));
        CKN(g_nccl.AllReduce(h->trace_out, h->trace_out, (size_t)trace_num_acc(h->prog), ncclDouble, ncclSum, h->comm, h->st_comm));
        CK(cudaEventRecord(h->ev_y, h->st_comm));
        CK(cudaStreamWaitEvent(h->st, h->ev_y, 0));
    }
    CK(cudaEventRecord(h->ev1, h->st));
    const int np = h->prog.n_theta;
    std::vector<double> out((size_t)np + 1);
    CK(cudaMemcpyAsync(out.data(), h->trace_out, sizeof(double) * (np + 1), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (h->sharded) { int rcs = sync_all(Lg); if (rcs) return rcs; }
    h->ms[4] = ev_ms(h->ev0, h->ev1);
    if (dmll_kernel) for (int p = 0; p < np; ++p) dmll_kernel[p] = out[p];
    if (trA) *trA = out[np];
    return GPB200_OK;
}

int gpb200_unwhiten(gpb200_handle* h, const double* v, double* f) {
    if (!h || !v || !f) return GPB200_EINVAL;
    { int rc = gpa_entry(h, "unwhiten"); if (rc) return rc; }
    int rc = upload_padded(h, h->r0, v);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_gpa[0], h->st));
    CK(gpa_trmv(h->F, h->ld, h->Npad, false, h->r0, h->gpa_part, h->r1, h->st, &h->launches));
    CK(cudaEventRecord(h->ev_gpa[1], h->st));
    CK(cudaMemcpyAsync(f, h->r1, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    h->ms[9] = ev_ms(h->ev_gpa[0], h->ev_gpa[1]);
    return GPB200_OK;
}

// Closed-form reverse-mode Cholesky (DESIGN.md section 9.4).  With W = L^-1, w = L' g and Phi(X) = tril(X) with the
// diagonal halved, the reference's chol_unblocked_rev! on tril(g v') contracted with dK (GPA.jl:164-173) equals
// 1/2 sum_ij (P + P')_ij dK_ij with P = W' Z, Z = Phi(w v') W.  Schedule (launches only, all on the stream):
//   w = L' g ; the inverse merges (W' in G's upper tiles) ; the row scan (Z' into F's upper tiles + Zd) ;
//   G_lower = -(W' Z + Z' W) as two NT GEMMs over k >= row ; the kernel-gradient trace with alpha = 0 (A = -G).
int gpb200_gpa_grad(gpb200_handle* h, const double* v, const double* dl_df, double* dll_v, double* dll_kernel) {
    if (!h || !v || !dl_df) return GPB200_EINVAL;
    { int rc = gpa_entry(h, "gpa_grad"); if (rc) return rc; }
    // G's lower triangle is about to be overwritten: K^-1, its symmetric mirror and the CV products are gone
    h->inv_ready = h->g_sym = h->cv_m_ok = h->chol_bar_ready = false;
    int rc = upload_padded(h, h->r0, v);
    if (!rc) rc = upload_padded(h, h->r1, dl_df);
    if (rc) return rc;
    const int Np = (int)h->Npad;
    cudaEvent_t* ev = h->ev_gpa;
    CK(cudaEventRecord(ev[0], h->st));
    CK(gpa_trmv(h->F, h->ld, h->Npad, true, h->r1, h->gpa_part, h->y1, h->st, &h->launches));
    CK(cudaEventRecord(ev[1], h->st));
    CK(inverse_merges(h));
    CK(cudaEventRecord(ev[2], h->st));
    CK(gpa_row_scan(h->G, h->ld, h->DinvT, h->r0, h->y1, h->Npad, h->gpa_part, h->F, h->Zd, h->st, &h->launches));
    CK(cudaEventRecord(ev[3], h->st));
    const GemmBuf bZd{h->tma_ok ? &h->mapZd : nullptr, h->Zd, TILE};
    for (int pass = 0; pass < 2; ++pass) {                 // P = W'Z (A = W', B = Z'), then P' (A = Z', B = W')
        const GemmOperand Wt{bufG(h), bufDinvT(h), 0, 0}, Zt{bufF(h), bZd, 0, 0};
        GemmDesc g = gemm_desc_default();
        g.A = pass == 0 ? Wt : Zt;
        g.B = pass == 0 ? Zt : Wt;
        g.C = h->G; g.ldc = h->ld; g.c_row0 = 0; g.c_col0 = 0;
        g.M = Np; g.N = Np; g.K = Np;
        g.alpha = -1.0; g.beta = pass == 0 ? 0.0 : 1.0;
        g.flags = GEMM_LOWER_ONLY | GEMM_KLO_M;
        CK(launch_gemm(h, g));
    }
    CK(cudaEventRecord(ev[4], h->st));
    CK(cudaMemsetAsync(h->alpha, 0, sizeof(double) * h->Npad, h->st));
    h->alpha_ready = false;
    h->launches += 2;
    CK(launch_trace(h, 1, 0, 1));
    CK(cudaEventRecord(ev[5], h->st));
    const int np = h->prog.n_theta;
    std::vector<double> out((size_t)np + 1);
    CK(cudaMemcpyAsync(out.data(), h->trace_out, sizeof(double) * (np + 1), cudaMemcpyDeviceToHost, h->st));
    if (dll_v) CK(cudaMemcpyAsync(dll_v, h->y1, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    h->ms[10] = ev_ms(ev[0], ev[1]);
    h->ms[11] = ev_ms(ev[1], ev[2]);
    h->ms[12] = ev_ms(ev[2], ev[3]);
    h->ms[13] = ev_ms(ev[3], ev[4]);
    h->ms[4] = ev_ms(ev[4], ev[5]);
    if (dll_kernel) for (int p = 0; p < np; ++p) dll_kernel[p] = out[p];
    h->chol_bar_ready = true;
    return GPB200_OK;
}

int gpb200_get_chol_bar(gpb200_handle* h, double* out) {
    if (!h || !out) return GPB200_EINVAL;
    if (!h->chol_bar_ready) return fail(h, GPB200_ESTATE, "get_chol_bar: gpa_grad first");
    CK(cudaSetDevice(h->device));
    const int64_t N = h->N;
    CK(cudaMemcpy2DAsync(out, sizeof(double) * N, h->G, sizeof(double) * h->ld, sizeof(double) * N, N,
                         cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    for (int64_t i = 0; i < N; ++i) {                      // G holds -(P + P') in its lower triangle
        for (int64_t j = 0; j < i; ++j) out[j * N + i] = out[i * N + j] = -out[i * N + j];
        out[i * N + i] = -out[i * N + i];
    }
    return GPB200_OK;
}

int gpb200_predict(gpb200_handle* h, int64_t M, const double* xs, int64_t ldxs, const double* alpha,
                   double* mu, double* var, double* cov) {
    if (!h) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "predict: factorize first");
    if (M <= 0 || !xs || ldxs < h->d || !mu) return fail(h, GPB200_EINVAL, "predict: bad M, xs, ldxs or mu");
    if (!alpha && !h->alpha_ready) return fail(h, GPB200_ESTATE, "predict: no alpha (call mll or pass alpha)");
    CK(cudaSetDevice(h->device));
    if (alpha) {
        int rc = upload_padded(h, h->alpha, alpha);
        if (rc) return rc;
        h->alpha_ready = true;
    }
    // chunk the test points so that the M_c x Npad workspace stays below ~16 GB
    int64_t cap = (int64_t)(16.0e9 / (8.0 * (double)h->Npad)) / TILE * TILE;
    if (const char* env = getenv("GPB200_PREDICT_CHUNK")) {            // testing hook: force small chunks
        const int64_t v = atoll(env) / TILE * TILE;
        if (v >= TILE && v < cap) cap = v;
    }
    if (cap < TILE) cap = TILE;
    if (h->sharded && cap > h->Npad) cap = h->Npad;       // a block of V' travels through the Npad x NBp panel buffer
    if (cov) cap = (M + TILE - 1) / TILE * TILE;          // full covariance needs all of V at once
    if (cov && h->sharded && cap > h->Npad) return fail(h, GPB200_EINVAL, "predict: full covariance of more than Npad test points is not supported with sharded storage");
    const bool need_v = (var != nullptr) || (cov != nullptr);
    Locals Lp;
    if (h->sharded) {
        int rc = shard_entry(h, Lp); if (rc) return rc;
        if (alpha) for (auto* q : Lp) if (q != h) { rc = upload_padded(q, q->alpha, alpha); if (rc) return rc; }
    }
    CK(cudaEventRecord(h->ev2, h->st));
    for (int64_t m0 = 0; h->sharded && m0 < M; m0 += cap) {
        // row-sharded factor: K*' on every rank, the triangular solve runs over column blocks owned like the rows of L
        const int64_t Mc = (M - m0 < cap) ? M - m0 : cap;
        const int64_t Mpad = (Mc + TILE - 1) / TILE * TILE;
        for (auto* q : Lp) {
            int rc = ensure_predict_ws(q, Mc, cov != nullptr);
            if (rc) { if (q != h) h->err = q->err; return rc; }
            SCK(q, cudaMemcpy2DAsync(q->xs, sizeof(double) * q->d, xs + m0 * ldxs, sizeof(double) * ldxs, sizeof(double) * q->d, Mc,
                                     cudaMemcpyHostToDevice, q->st));
            ++q->launches;
            SCK(q, crossgram_launch(q->prog, q->xs, q->d, Mc, Mpad, q->x, q->d, q->N, q->Npad, q->d, q->Kst, q->Npad, q->st));
            if (need_v) {
                ++q->launches;
                SCK(q, kdiag_launch(q->prog, q->xs, q->d, Mc, q->pvar, q->st));           // running variance starts at k**
                if (cov) { ++q->launches; SCK(q, gram_full_launch(q->prog, q->xs, q->d, Mc, Mpad, q->d, q->Kss, Mpad, q->st)); }
            }
        }
        ++h->launches;
        CK(rowdot_launch(h->Kst, h->Npad, h->alpha, Mc, h->Npad, h->pmu, h->st));          // GP.jl:26
        CK(cudaMemcpyAsync(mu + m0, h->pmu, sizeof(double) * Mc, cudaMemcpyDeviceToHost, h->st));
        if (need_v) {
            int rc = shard_predict_solve(Lp, (int)Mpad, Mc, var != nullptr, cov != nullptr);
            if (rc) { if (Lp[0] != h) h->err = Lp[0]->err; return rc; }
            if (var) CK(cudaMemcpyAsync(var + m0, h->pvar, sizeof(double) * Mc, cudaMemcpyDeviceToHost, h->st));
            if (cov && !h->cov_keep_device) CK(cudaMemcpy2DAsync(cov, sizeof(double) * M, h->Kss, sizeof(double) * Mpad, sizeof(double) * M, M,
                                          cudaMemcpyDeviceToHost, h->st));
        }
        { int rc = sync_all(Lp); if (rc) return rc; }
    }
    for (int64_t m0 = 0; !h->sharded && m0 < M; m0 += cap) {
        const int64_t Mc = (M - m0 < cap) ? M - m0 : cap;
        const int64_t Mpad = (Mc + TILE - 1) / TILE * TILE;
        int rc = ensure_predict_ws(h, Mc, cov != nullptr);
        if (rc) return rc;
        CK(cudaMemcpy2DAsync(h->xs, sizeof(double) * h->d, xs + m0 * ldxs, sizeof(double) * ldxs,
                             sizeof(double) * h->d, Mc, cudaMemcpyHostToDevice, h->st));
        h->launches += 2;
        CK(crossgram_launch(h->prog, h->xs, h->d, Mc, Mpad, h->x, h->d, h->N, h->Npad, h->d, h->Kst, h->Npad, h->st));
        CK(rowdot_launch(h->Kst, h->Npad, h->alpha, Mc, h->Npad, h->pmu, h->st));          // GP.jl:26
        CK(cudaMemcpyAsync(mu + m0, h->pmu, sizeof(double) * Mc, cudaMemcpyDeviceToHost, h->st));
        if (need_v) {
            CK(trsm_rec(h, (int)Mpad, 0, (int)h->Npad));                                   // whiten!, GP.jl:27
            if (var) {
                h->launches += 2;
                CK(kdiag_launch(h->prog, h->xs, h->d, Mc, h->pkdiag, h->st));
                CK(rowvar_launch(h->Kst, h->Npad, h->pkdiag, Mc, h->Npad, h->pvar, h->st));
                CK(cudaMemcpyAsync(var + m0, h->pvar, sizeof(double) * Mc, cudaMemcpyDeviceToHost, h->st));
            }
            if (cov) {                                                                      // GP.jl:51-54
                ++h->launches;
                CK(gram_full_launch(h->prog, h->xs, h->d, Mc, Mpad, h->d, h->Kss, Mpad, h->st));
                GemmBuf bk{h->tma_ok ? &h->mapKst : nullptr, h->Kst, h->Npad};
                GemmDesc g = gemm_desc_default();
                g.A = GemmOperand{bk, bufNone(), 0, 0};
                g.B = GemmOperand{bk, bufNone(), 0, 0};
                g.C = h->Kss; g.ldc = Mpad; g.M = (int)Mpad; g.N = (int)Mpad; g.K = (int)h->Npad;
                g.alpha = -1.0; g.beta = 1.0;
                CK(launch_gemm(h, g));
                if (!h->cov_keep_device)
                    CK(cudaMemcpy2DAsync(cov, sizeof(double) * M, h->Kss, sizeof(double) * Mpad, sizeof(double) * M, M,
                                         cudaMemcpyDeviceToHost, h->st));
            }
        }
        CK(cudaStreamSynchronize(h->st));
    }
    CK(cudaEventRecord(h->ev3, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    h->ms[5] = ev_ms(h->ev2, h->ev3);
    return GPB200_OK;
}

// rand(gp, X, n) (src/GP.jl:120-146): posterior draws  mu* + chol(Sigma* + nugget I) Z  entirely on the device: full predictive
// covariance (predictMVN), make_posdef!(Sigma; nugget) with the engine's own Cholesky on an M x M sub-engine, unwhiten! as one
// triangular NT GEMM.  z / samples are Julia's M x nsamp column-major matrices (== nsamp x M row-major).
int gpb200_rand(gpb200_handle* h, int64_t M, const double* xs, int64_t ldxs, const double* alpha, int64_t nsamp,
                const double* z, double nugget, double* mu_minus_mean, double* samples) {
    if (!h) return GPB200_EINVAL;
    if (M <= 0 || nsamp <= 0 || !z || !samples || !mu_minus_mean) return fail(h, GPB200_EINVAL, "rand: bad M, nsamp, z, mu or samples");
    if (!(nugget >= 0.0)) return fail(h, GPB200_EINVAL, "rand: nugget must be >= 0");
    CK(cudaSetDevice(h->device));
    static double cov_flag;                                     // non-null marker: the covariance stays in h->Kss
    h->cov_keep_device = true;
    int rc = gpb200_predict(h, M, xs, ldxs, alpha, mu_minus_mean, nullptr, &cov_flag);
    h->cov_keep_device = false;
    if (rc) return rc;
    const int64_t Mpad = (M + TILE - 1) / TILE * TILE, Spad = (nsamp + TILE - 1) / TILE * TILE;
    // sub-engine of size M (shares this handle's stream)
    if (!h->sub) {
        rc = gpb200_create(&h->sub, h->device);
        if (rc) return fail(h, rc, "rand: could not create the M x M sub-engine");
        cudaStreamDestroy(h->sub->st);
        h->sub->own_stream = false;
    }
    gpb200_handle* sb = h->sub;
    sb->st = h->st;
    if (!sb->has_data || sb->N != M) {
        std::vector<double> dummy((size_t)M, 0.0);
        rc = gpb200_set_data(sb, M, 1, dummy.data(), 1);
        if (rc) { h->err = "rand: " + sb->err; return rc; }
    }
    ++h->launches;
    CK(spd_from_cov_launch(sb->G, sb->ld, h->Kss, Mpad, M, Mpad, nugget, h->st));
    rc = chol_inplace(sb);
    if (rc) { h->err = "rand: predictive covariance + nugget is not positive definite: " + sb->err; return rc; }
    // draws: Zt (nsamp x M, zero padded) on the device
    if (Spad > h->rz_rows || Mpad > h->rz_cols) {
        if (h->rz) cudaFree(h->rz);
        if (h->rout) cudaFree(h->rout);
        h->rz = h->rout = nullptr; h->rz_rows = h->rz_cols = 0;
        CK(cudaMalloc(&h->rz, sizeof(double) * Spad * Mpad));
        CK(cudaMalloc(&h->rout, sizeof(double) * Spad * Mpad));
        h->rz_rows = Spad; h->rz_cols = Mpad;
    }
    const int64_t ldz = h->rz_cols;
    if (h->tma_ok && !gemm_make_tensor_map(&h->mapRz, h->rz, h->rz_rows, ldz, ldz)) return fail(h, GPB200_ECUDA, "rand: tensor map");
    CK(cudaMemsetAsync(h->rz, 0, sizeof(double) * h->rz_rows * ldz, h->st));
    CK(cudaMemcpy2DAsync(h->rz, sizeof(double) * ldz, z, sizeof(double) * M, sizeof(double) * M, nsamp, cudaMemcpyHostToDevice, h->st));
    {   // out[s, m] = sum_{k <= m} Zt[s, k] L[m, k]       (unwhiten!: L Z)
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{GemmBuf{h->tma_ok ? &h->mapRz : nullptr, h->rz, ldz}, bufNone(), 0, 0};
        g.B = GemmOperand{bufF(sb), bufNone(), 0, 0};
        g.C = h->rout; g.ldc = ldz; g.M = (int)Spad; g.N = (int)Mpad; g.K = (int)Mpad;
        g.flags = GEMM_KHI_N;
        CK(launch_gemm(h, g));
    }
    ++h->launches;
    CK(add_rowvec_launch(h->rout, ldz, h->pmu, nsamp, M, h->st));                          // + mu (K*' alpha part)
    CK(cudaMemcpy2DAsync(samples, sizeof(double) * M, h->rout, sizeof(double) * ldz, sizeof(double) * M, nsamp, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPB200_OK;
}

// ---- ElasticGPE append! (src/GPEelastic.jl:13-22): extend the factor by k new observations -----------------------------
// The reference appends rows to an elastic Cholesky (ElasticPDMats.append!, a rank-k extension) and keeps the hyper-parameters
// (update_target!(gp, kern=false, noise=false)).  Here the rows live inside the capacity reserved at set_data (option
// "capacity"): only the block rows from the first touched 128-row tile on are rebuilt --
//   Gram rows r >= c0;  L[r, 0:c0] = K[r, 0:c0] L11^-T (whitening TRSM against the existing factor);
//   Schur complement of the trailing block (one GEMM with K = c0);  Cholesky of that small trailing block --
// i.e. O(k N^2) instead of O(N^3).  Returns GPB200_EINVAL if N + k exceeds the capacity (the caller refits).
int gpb200_append(gpb200_handle* h, int64_t k, const double* xnew, int64_t ldx) {
    if (!h) return GPB200_EINVAL;
    if (k <= 0 || !xnew || ldx < h->d) return fail(h, GPB200_EINVAL, "append: bad k, x or ldx");
    if (!h->factored) return fail(h, GPB200_ESTATE, "append: factorize first");
    if (h->nranks > 1) return fail(h, GPB200_ESTATE, "append: single-GPU handles only");
    if (h->n_noise != 1) return fail(h, GPB200_ESTATE, "append: scalar logNoise only (per-point noise needs a refit)");
    if (h->N + k > h->Npad) return fail(h, GPB200_EINVAL, "append: capacity exceeded (set option \"capacity\" before set_data, or refit)");
    CK(cudaSetDevice(h->device));
    const int64_t Nold = h->N, Nnew = Nold + k;
    const int d = h->d, Np = (int)h->Npad;
    const int c0 = (int)(Nold / TILE * TILE);                       // first tile row that changes
    CK(cudaMemcpy2DAsync(h->x + Nold * d, sizeof(double) * d, xnew, sizeof(double) * ldx, sizeof(double) * d, k, cudaMemcpyHostToDevice, h->st));
    h->xmap_ok = false;
    if (h->xp) {
        CK(cudaMemcpy2DAsync(h->xp + Nold * h->dxp, sizeof(double) * h->dxp, xnew, sizeof(double) * ldx, sizeof(double) * d, k, cudaMemcpyHostToDevice, h->st));
        ++h->launches;
        CK(shard_transpose(h->xpt, Np, h->xp, h->dxp, Np, h->dxp, h->st));
        h->xmap_ok = gemm_make_tensor_map_plain(&h->mapX, h->xp, Nnew, h->dxp, h->dxp, TILE, h->dxp) &&
                     gemm_make_tensor_map_plain(&h->mapXT, h->xpt, h->dxp, Nnew, Np, h->dxp, TILE);
    }
    h->N = Nnew;
    h->inv_ready = h->alpha_ready = false; h->g_sym = false; h->cv_m_ok = false; h->chol_bar_ready = false;
    const int init = INT_MAX;
    CK(cudaMemcpyAsync(h->info_dev, &init, sizeof(int), cudaMemcpyHostToDevice, h->st));
    ++h->launches;
    // Gram rows >= c0 (columns <= row), identity beyond the new N
    CK(gram_lower_launch(h->prog, h->x, d, d, Nnew, Np, h->noise_var, 1, h->nugget, h->G, h->ld, h->st, 0, 1, 0, 0, c0 / TILE));
    cudaError_t e = cudaSuccess;
    if (c0 > 0) {
        // rows >= c0 of G against the existing factor: G[r, 0:c0] <- G[r, 0:c0] L11^-T, then keep them as rows of L
        CUtensorMap sub{};
        double* gsub = h->G + (size_t)c0 * h->ld;
        const bool tma = h->tma_ok && gemm_make_tensor_map(&sub, gsub, Np - c0, Np, h->ld);
        GemmBuf bk{tma ? &sub : nullptr, gsub, h->ld};
        const int impl_save = h->gemm_impl;
        if (!tma) h->gemm_impl = 1;
        e = trsm_rec_buf(h, bk, Np - c0, 0, c0);
        h->gemm_impl = impl_save;
        CK(e);
        CK(cudaMemcpy2DAsync(h->F + (size_t)c0 * h->ld, sizeof(double) * h->ld, gsub, sizeof(double) * h->ld, sizeof(double) * c0, Np - c0,
                             cudaMemcpyDeviceToDevice, h->st));
        // Schur complement of the trailing block:  G[r, c] -= sum_{k < c0} L[r, k] L[c, k],  r >= c >= c0
        CK(schur_update(h, c0, Np - c0, Np - c0, 0, c0));
    }
    // factor the trailing block tile by tile (right-looking, 128-wide panels)
    for (int p = c0; p < Np; p += TILE) {
        CK(chol_panel(h, p, TILE, TILE));
        const int rem = Np - p - TILE;
        if (rem > 0) CK(schur_update(h, p + TILE, rem, rem, p, TILE));
    }
    int info = 0;
    CK(cudaMemcpyAsync(&info, h->info_dev, sizeof(int), cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    if (info != INT_MAX) {
        h->factored = false;
        char buf[128];
        snprintf(buf, sizeof buf, "append: extended matrix is not positive definite; leading minor %d", info);
        h->err = buf;
        return info > h->N ? (int)h->N : info;
    }
    return GPB200_OK;
}

// ---- cross-validation on the resident inverse (src/crossvalidation.jl) --------------------------------------------
// The reference forms inv(Sigma) and, per hyper-parameter j, Z_j = inv(Sigma) dK_j and Z_j inv(Sigma) on the host
// (crossvalidation.jl:86-108, 270-283).  Here K_y^-1 already sits on the device after gpb200_grad_prepare; per parameter:
// D = dK_j (recomputed from x), Y' = K^-1 D, M_j = Y' K^-1 -- two NT DMMA GEMMs -- and the two N-vectors every LOO / fold
// formula needs: Z_j alpha = Y' alpha and diag(M_j).  Fold formulas read principal sub-blocks through gpb200_cv_block.
static int cv_prepare(gpb200_handle* h) {
    if (!h->inv_ready) return fail(h, GPB200_ESTATE, "cv: grad_prepare first (K_y^-1 must be resident)");
    if (h->nranks > 1) return fail(h, GPB200_ESTATE, "cv: K^-1 is distributed over the ranks; single-GPU handles only");
    const size_t nn = sizeof(double) * (size_t)h->Npad * (size_t)h->Npad;
    if (!h->cvD || !h->cvY) {
        if (h->cvD) { cudaFree(h->cvD); h->cvD = nullptr; }
        if (h->cvY) { cudaFree(h->cvY); h->cvY = nullptr; }
        h->cv_m_ok = false;
        if (cudaMalloc(&h->cvD, nn) != cudaSuccess || cudaMalloc(&h->cvY, nn) != cudaSuccess) {
            (void)cudaGetLastError();
            if (h->cvD) { cudaFree(h->cvD); h->cvD = nullptr; }
            h->cvY = nullptr;
            return fail(h, GPB200_ECUDA, "cv: out of device memory for the two N x N work matrices");
        }
        if (h->tma_ok && !(gemm_make_tensor_map(&h->mapCvD, h->cvD, h->Npad, h->Npad, h->Npad) &&
                           gemm_make_tensor_map(&h->mapCvY, h->cvY, h->Npad, h->Npad, h->Npad)))
            return fail(h, GPB200_ECUDA, "cv: cuTensorMapEncodeTiled failed");
    }
    if (!h->g_sym) {
        ++h->launches;
        CK(symmetrize_launch(h->G, h->ld, h->Npad, h->st));      // lower K^-1 -> full symmetric (the W' scratch above it is dead)
        h->g_sym = true;
    }
    return GPB200_OK;
}

int gpb200_cv_param(gpb200_handle* h, int32_t param, const double* alpha, double* Zj_alpha, double* diag_ZjSinv) {
    if (!h || !Zj_alpha || !diag_ZjSinv) return GPB200_EINVAL;
    if (param < -1 || param >= h->prog.n_theta) return fail(h, GPB200_EINVAL, "cv_param: parameter index out of range");
    if (!alpha && !h->alpha_ready) return fail(h, GPB200_ESTATE, "cv_param: no alpha (call mll or pass alpha)");
    CK(cudaSetDevice(h->device));
    int rc = cv_prepare(h);
    if (rc) return rc;
    if (alpha) { rc = upload_padded(h, h->alpha, alpha); if (rc) return rc; h->alpha_ready = true; }
    const int Np = (int)h->Npad;
    GemmBuf bD{h->tma_ok ? &h->mapCvD : nullptr, h->cvD, h->Npad}, bY{h->tma_ok ? &h->mapCvY : nullptr, h->cvY, h->Npad};
    const double* Yt = h->cvY;
    if (param >= 0) {
        ++h->launches;
        CK(gram_grad_full_launch(h->prog, h->x, h->d, h->d, h->N, h->Npad, param, h->cvD, h->Npad, h->st));
        GemmDesc g = gemm_desc_default();                           // Y' = K^-1 D   (both symmetric: NT form)
        g.A = GemmOperand{bufG(h), bufNone(), 0, 0};
        g.B = GemmOperand{bD, bufNone(), 0, 0};
        g.C = h->cvY; g.ldc = h->Npad; g.M = Np; g.N = Np; g.K = Np;
        CK(launch_gemm(h, g));
    } else {
        Yt = h->G;                                                  // noise: Z = K^-1 (crossvalidation.jl:124-126)
    }
    h->launches += 2;
    CK(rowdot_launch(Yt, h->Npad, h->alpha, h->N, h->Npad, h->r1, h->st));              // Z_j alpha
    CK(rowdot2_launch(h->G, Yt, h->Npad, h->N, h->Npad, h->y1, h->st));                 // diag(Z_j K^-1) = rowwise <K^-1_i, Y'_i>
    {   // M_j = Y' K^-1  -> cvD (fold sub-blocks)
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{param >= 0 ? bY : bufG(h), bufNone(), 0, 0};
        g.B = GemmOperand{bufG(h), bufNone(), 0, 0};
        g.C = h->cvD; g.ldc = h->Npad; g.M = Np; g.N = Np; g.K = Np;
        CK(launch_gemm(h, g));
    }
    h->cv_m_ok = true;
    CK(cudaMemcpyAsync(Zj_alpha, h->r1, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaMemcpyAsync(diag_ZjSinv, h->y1, sizeof(double) * h->N, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    profile_collect(h);
    return GPB200_OK;
}

int gpb200_cv_block(gpb200_handle* h, int32_t which, int64_t nV, const int64_t* idx, double* out) {
    if (!h || !idx || !out || nV <= 0 || which < 0 || which > 1) return GPB200_EINVAL;
    CK(cudaSetDevice(h->device));
    int rc = cv_prepare(h);
    if (rc) return rc;
    if (which == 1 && !h->cv_m_ok) return fail(h, GPB200_ESTATE, "cv_block: which = 1 reads M_j of the last cv_param call; call cv_param first");
    for (int64_t a = 0; a < nV; ++a)
        if (idx[a] < 0 || idx[a] >= h->N) return fail(h, GPB200_EINVAL, "cv_block: index out of range");
    if (nV > h->cvblk_cap) {
        if (h->cvblk) cudaFree(h->cvblk);
        if (h->cvidx) cudaFree(h->cvidx);
        h->cvblk = nullptr; h->cvidx = nullptr; h->cvblk_cap = 0;
        CK(cudaMalloc(&h->cvblk, sizeof(double) * nV * nV));
        CK(cudaMalloc(&h->cvidx, sizeof(long long) * nV));
        h->cvblk_cap = nV;
    }
    static_assert(sizeof(long long) == sizeof(int64_t), "index width");
    CK(cudaMemcpyAsync(h->cvidx, idx, sizeof(long long) * nV, cudaMemcpyHostToDevice, h->st));
    ++h->launches;
    CK(gather_block_launch(h->cvblk, which == 0 ? h->G : h->cvD, h->Npad, h->cvidx, nV, h->st));
    CK(cudaMemcpyAsync(out, h->cvblk, sizeof(double) * nV * nV, cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPB200_OK;
}

int gpb200_get_gram(gpb200_handle* h, double* K) {
    if (!h || !K) return GPB200_EINVAL;
    if (!h->has_data || !h->has_kernel) return fail(h, GPB200_ESTATE, "get_gram: set_data and set_kernel first");
    CK(cudaSetDevice(h->device));
    double* tmp = nullptr;
    const size_t nn = sizeof(double) * (size_t)h->Npad * (size_t)h->Npad;
    CK(cudaMalloc(&tmp, nn));
    cudaError_t e = launch_gram(h, tmp, h->Npad, 0, 1, 0, 0);
    if (e == cudaSuccess)
        e = cudaMemcpy2DAsync(K, sizeof(double) * h->N, tmp, sizeof(double) * h->Npad, sizeof(double) * h->N, h->N,
                              cudaMemcpyDeviceToHost, h->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->st);
    cudaFree(tmp);
    CK(e);
    const int64_t N = h->N;
    for (int64_t i = 0; i < N; ++i)
        for (int64_t j = i + 1; j < N; ++j) K[i * N + j] = K[j * N + i];
    return GPB200_OK;
}

int gpb200_get_factor(gpb200_handle* h, double* U) {
    if (!h || !U) return GPB200_EINVAL;
    if (!h->factored) return fail(h, GPB200_ESTATE, "get_factor: factorize first");
    CK(cudaSetDevice(h->device));
    const int64_t N = h->N;
    if (h->sharded) { int rc = copy_own_rows(h, U, h->F); if (rc) return rc; }
    else
    CK(cudaMemcpy2DAsync(U, sizeof(double) * N, h->F, sizeof(double) * h->ld, sizeof(double) * N, N,
                         cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    // row-major lower L == column-major upper U; clear the other triangle (scratch on the device)
    for (int64_t j = 0; j < N; ++j)
        for (int64_t i = j + 1; i < N; ++i) U[j * N + i] = 0.0;
    return GPB200_OK;
}

int gpb200_get_inverse(gpb200_handle* h, double* Kinv) {
    if (!h || !Kinv) return GPB200_EINVAL;
    if (!h->inv_ready) return fail(h, GPB200_ESTATE, "get_inverse: grad_prepare first");
    if (h->nranks > 1 && !h->sharded) return fail(h, GPB200_ESTATE, "get_inverse: K^-1 is distributed over the ranks (tile rows round-robin)");
    CK(cudaSetDevice(h->device));
    const int64_t N = h->N;
    if (h->sharded) { int rc = copy_own_rows(h, Kinv, h->G); if (rc) return rc; }     // own rows only (others zero): sum over the ranks
    else
    CK(cudaMemcpy2DAsync(Kinv, sizeof(double) * N, h->G, sizeof(double) * h->ld, sizeof(double) * N, N,
                         cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    for (int64_t i = 0; i < N; ++i)
        for (int64_t j = i + 1; j < N; ++j) Kinv[i * N + j] = Kinv[j * N + i];
    return GPB200_OK;
}

int gpb200_get_inverse_diag(gpb200_handle* h, double* diag) {
    if (!h || !diag) return GPB200_EINVAL;
    if (!h->inv_ready) return fail(h, GPB200_ESTATE, "get_inverse_diag: grad_prepare first");
    if (h->nranks > 1) return fail(h, GPB200_ESTATE, "get_inverse_diag: K^-1 is distributed over the ranks");
    CK(cudaSetDevice(h->device));
    // strided gather of G[i,i]: pitch (ld+1) doubles, one double per row
    CK(cudaMemcpy2DAsync(diag, sizeof(double), h->G, sizeof(double) * (h->ld + 1), sizeof(double), h->N,
                         cudaMemcpyDeviceToHost, h->st));
    CK(cudaStreamSynchronize(h->st));
    return GPB200_OK;
}

int gpb200_dgemm_nt_device(gpb200_handle* h, int impl, int64_t M, int64_t N, int64_t K, double alpha,
                           const double* dA, int64_t lda, const double* dB, int64_t ldb, double beta, double* dC,
                           int64_t ldc, int lower_only, int reps, double* ms) {
    if (!h || !dA || !dB || !dC) return GPB200_EINVAL;
    if (M % TILE || N % TILE || K % 16 || M <= 0 || N <= 0 || K <= 0 || reps < 1)
        return fail(h, GPB200_EINVAL, "dgemm_nt: M,N multiples of 128, K multiple of 16");
    CK(cudaSetDevice(h->device));
    CUtensorMap ma{}, mb{};
    const bool tma = gemm_make_tensor_map(&ma, dA, M, K, lda) && gemm_make_tensor_map(&mb, dB, N, K, ldb);
    if (impl == 0 && !tma) return fail(h, GPB200_ECUDA, "dgemm_nt: TMA descriptors unavailable");
    GemmDesc g = gemm_desc_default();
    g.A = GemmOperand{GemmBuf{&ma, dA, lda}, bufNone(), 0, 0};
    g.B = GemmOperand{GemmBuf{&mb, dB, ldb}, bufNone(), 0, 0};
    g.C = dC; g.ldc = ldc; g.M = (int)M; g.N = (int)N; g.K = (int)K;
    g.alpha = alpha; g.beta = beta;
    g.flags = lower_only ? GEMM_LOWER_ONLY : 0;
    CK(cudaEventRecord(h->ev0, h->st));
    for (int r = 0; r < reps; ++r) { ++h->launches; CK(gemm_nt_launch(g, impl, h->st)); }
    CK(cudaEventRecord(h->ev1, h->st));
    CK(cudaStreamSynchronize(h->st));
    if (ms) *ms = ev_ms(h->ev0, h->ev1);
    return GPB200_OK;
}

int gpb200_fp64_peak(gpb200_handle* h, double* tflops_dmma, double* tflops_dfma) {
    if (!h) return GPB200_EINVAL;
    CK(cudaSetDevice(h->device));
    double t[2] = {0, 0};
    CK(fp64_peak_measure(h->st, t));
    if (tflops_dmma) *tflops_dmma = t[0];
    if (tflops_dfma) *tflops_dfma = t[1];
    return GPB200_OK;
}


#define GPB200_IPC_BYTES 512
int gpb200_ipc_export(gpb200_handle* h, char* out) {
    if (!h || !out) return GPB200_EINVAL;
    if (!h->has_data) return fail(h, GPB200_ESTATE, "ipc_export: set_data first (buffers must exist)");
    CK(cudaSetDevice(h->device));
    memset(out, 0, GPB200_IPC_BYTES);
    cudaIpcMemHandle_t hd[5];
    CK(cudaIpcGetMemHandle(&hd[0], h->F));
    CK(cudaIpcGetMemHandle(&hd[1], h->Dinv));
    CK(cudaIpcGetMemHandle(&hd[2], h->DinvT));
    CK(cudaIpcGetMemHandle(&hd[3], h->logd));
    CK(cudaIpcGetMemHandle(&hd[4], h->sig));
    static_assert(5 * sizeof(cudaIpcMemHandle_t) + 16 <= GPB200_IPC_BYTES, "ipc blob too small");
    memcpy(out, hd, sizeof hd);
    const int64_t np = h->Npad;
    memcpy(out + sizeof hd, &np, sizeof np);
    return GPB200_OK;
}

int gpb200_ipc_import(gpb200_handle* h, int nranks, const char* all) {
    if (!h || !all) return GPB200_EINVAL;
    if (nranks != h->nranks || nranks < 2 || nranks > 8) return fail(h, GPB200_EINVAL, "ipc_import: call comm_init first; 2..8 ranks");
    CK(cudaSetDevice(h->device));
    close_peer_maps(h);                        // re-import: drop the previous mappings first
    int n = 0;
    for (int q = 0; q < nranks; ++q) {
        if (q == h->rank) continue;
        const char* blob = all + (size_t)q * GPB200_IPC_BYTES;
        cudaIpcMemHandle_t hd[5];
        memcpy(hd, blob, sizeof hd);
        int64_t np = 0;
        memcpy(&np, blob + sizeof hd, sizeof np);
        if (np != h->Npad) return fail(h, GPB200_EINVAL, "ipc_import: peers hold a different problem size");
        void* ptr[5];
        for (int k = 0; k < 5; ++k) CK(cudaIpcOpenMemHandle(&ptr[k], hd[k], cudaIpcMemLazyEnablePeerAccess));
        h->peer_rank[n] = q;
        h->peer_F[n] = (double*)ptr[0]; h->peer_Dinv[n] = (double*)ptr[1]; h->peer_DinvT[n] = (double*)ptr[2];
        h->peer_logd[n] = (double*)ptr[3]; h->peer_sig[n] = (int*)ptr[4];
        ++n;
    }
    h->n_peer = n;
    int* words[7];
    for (int q = 0; q < n; ++q) words[q] = h->peer_sig[q] + h->rank;
    if (!h->peer_sig_dev) CK(cudaMalloc(&h->peer_sig_dev, sizeof(int*) * 8));
    CK(cudaMemcpy(h->peer_sig_dev, words, sizeof(int*) * n, cudaMemcpyHostToDevice));
    h->p2p = true;
    return GPB200_OK;
}

int gpb200_nccl_unique_id(char* id128) {
    if (!id128) return GPB200_EINVAL;
    if (!nccl_load()) { g_create_error = "libnccl.so.2 could not be loaded"; return GPB200_ENCCL; }
    ncclUniqueId id;
    if (g_nccl.GetUniqueId(&id) != ncclSuccess) { g_create_error = "ncclGetUniqueId failed"; return GPB200_ENCCL; }
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    memcpy(id128, &id, 128);
    return GPB200_OK;
}

int gpb200_comm_init(gpb200_handle* h, int nranks, int rank, const char* id128) {
    if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return GPB200_EINVAL;
    if (nranks & (nranks - 1)) return fail(h, GPB200_EINVAL, "comm_init: number of ranks must be a power of two");
    if (h->grp) return fail(h, GPB200_ESTATE, "comm_init: handle belongs to an in-process group");
    if (!nccl_load()) return fail(h, GPB200_ENCCL, "libnccl.so.2 could not be loaded");
    CK(cudaSetDevice(h->device));
    if (h->comm) { g_nccl.CommDestroy(h->comm); h->comm = nullptr; }
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    CKN(g_nccl.CommInitRank(&h->comm, nranks, id, rank));
    if (!h->st_comm) CK(cudaStreamCreateWithFlags(&h->st_comm, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        if (!h->ev_packed[i]) CK(cudaEventCreateWithFlags(&h->ev_packed[i], cudaEventDisableTiming));
        if (!h->ev_bcast[i]) CK(cudaEventCreateWithFlags(&h->ev_bcast[i], cudaEventDisableTiming));
        if (!h->ev_unpacked[i]) CK(cudaEventCreateWithFlags(&h->ev_unpacked[i], cudaEventDisableTiming));
    }
    if (!h->ev_x) CK(cudaEventCreateWithFlags(&h->ev_x, cudaEventDisableTiming));
    if (!h->ev_y) CK(cudaEventCreateWithFlags(&h->ev_y, cudaEventDisableTiming));
    h->nranks = nranks; h->rank = rank;
    h->factored = h->inv_ready = false;
    return GPB200_OK;
}


int gpb200_storage_info(gpb200_handle* h, int64_t* out, int32_t n) {
    if (!h || !out) return GPB200_EINVAL;
    int64_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    v[6] = h->tma_ok ? 1 : 0;
    v[0] = h->sharded ? 1 : 0;
    v[1] = h->sharded ? (int64_t)vm_mapped_bytes(h->vmF) : (h->F ? (int64_t)sizeof(double) * h->Npad * h->Npad : 0);
    v[2] = h->sharded ? (int64_t)vm_mapped_bytes(h->vmG) : (h->G ? (int64_t)sizeof(double) * h->Npad * h->Npad : 0);
    v[3] = h->sharded ? h->rb : 0;
    v[4] = h->nranks;
    v[5] = h->rank;
    for (int i = 0; i < n && i < 8; ++i) out[i] = v[i];
    return GPB200_OK;
}

int gpb200_group_create(gpb200_handle** hs, int n) {
    if (!hs || n < 1 || n > 8) return GPB200_EINVAL;
    for (int i = 0; i < n; ++i) {
        if (!hs[i]) return GPB200_EINVAL;
        if (hs[i]->grp || hs[i]->comm) return fail(hs[i], GPB200_ESTATE, "group_create: handle already belongs to a group / communicator");
        if (hs[i]->device != hs[0]->device) return fail(hs[i], GPB200_EINVAL, "group_create: all handles must live on one device");
        for (int j = 0; j < i; ++j) if (hs[j] == hs[i]) return fail(hs[i], GPB200_EINVAL, "group_create: duplicate handle");
    }
    gpb200_group* g = new gpb200_group();
    for (int i = 0; i < n; ++i) {
        g->hs.push_back(hs[i]);
        hs[i]->grp = g; hs[i]->nranks = n; hs[i]->rank = i;
        hs[i]->factored = hs[i]->inv_ready = false;
    }
    return GPB200_OK;
}

// ================================================================================================
// FITC -- Fully Independent Training Conditional (src/sparse/fully_indep_train_conditional.jl)
//   update_cK! (:134-156), `\` (:33-36), logdet (:77), dmll_noise (:243-257), predictMVN (:324-332 ->
//   determ_train_conditional.jl:41-59 -> subsetofregressors.jl:302-321).
// The reference materialises K_uf (M x N) and several copies; here N is streamed in chunks through two
// staging buffers and only M x M state persists (H7 of SURVEY.md §7.2): per chunk a cross-Gram, a
// recursive TRSM against L_uu for diag(Q_ff), and one rank-Nc SYRK into Sigma_QR -- all on the DMMA GEMM.
// ================================================================================================
#define FCK(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__,       \
                     cudaGetErrorString(e_));                                                      \
            f->err = buf_;                                                                         \
            (void)cudaGetLastError();                                                              \
            return GPB200_ECUDA;                                                                   \
        }                                                                                          \
    } while (0)
#define FSUB(call, who)                                                                            \
    do {                                                                                           \
        int rc_ = (call);                                                                          \
        if (rc_ != GPB200_OK) { f->err = std::string(#call) + ": " + (who)->err; return rc_; }     \
    } while (0)

#define FCKN(call)                                                                                 \
    do {                                                                                           \
        ncclResult_t r_ = (call);                                                                  \
        if (r_ != ncclSuccess) {                                                                   \
            f->err = std::string(#call) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "nccl error"); \
            return GPB200_ENCCL;                                                                   \
        }                                                                                          \
    } while (0)
// in-place sum over the ranks of a device vector (no-op on one rank)
static int fitc_allreduce(gpb200_fitc* f, double* v, size_t n) {
    if (f->nranks <= 1 || n == 0) return GPB200_OK;
    FCKN(g_nccl.AllReduce(v, v, n, ncclDouble, ncclSum, f->comm, f->eu->st));
    return GPB200_OK;
}

int gpb200_fitc_comm_init(gpb200_fitc* f, int nranks, int rank, const char* id128) {
    if (!f || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return GPB200_EINVAL;
    if (!nccl_load()) { f->err = "libnccl.so.2 could not be loaded"; return GPB200_ENCCL; }
    FCK(cudaSetDevice(f->device));
    if (f->comm) { g_nccl.CommDestroy(f->comm); f->comm = nullptr; }
    ncclUniqueId id;
    memcpy(&id, id128, 128);
    FCKN(g_nccl.CommInitRank(&f->comm, nranks, id, rank));
    f->nranks = nranks; f->rank = rank;
    f->factored = f->alpha_ready = false;
    return GPB200_OK;
}

void gpb200_fitc_destroy(gpb200_fitc* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    if (f->eu && f->eu->st) cudaStreamSynchronize(f->eu->st);
    double** ptrs[] = {&f->x, &f->xs, &f->lam, &f->y, &f->alpha, &f->tmpn, &f->w, &f->tmpc, &f->zeroc, &f->tmpc2,
                       &f->bvec, &f->uvec, &f->tmpm, &f->rhsm, &f->scal, &f->bufA, &f->bufB,
                       &f->bufC, &f->Hbuf, &f->Wbuf, &f->Tbuf, &f->gvec, &f->betav, &f->gpart, &f->gacc, &f->gtmp};
    for (auto pp : ptrs) { if (*pp) cudaFree(*pp); *pp = nullptr; }
    if (f->Kss) cudaFree(f->Kss);
    if (f->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(f->comm);
    if (f->es) { f->es->st = nullptr; f->es->own_stream = false; gpb200_destroy(f->es); }
    if (f->eu) gpb200_destroy(f->eu);
    delete f;
}

int gpb200_fitc_create(gpb200_fitc** out, int device) {
    if (!out) return GPB200_EINVAL;
    *out = nullptr;
    gpb200_fitc* f = new gpb200_fitc();
    f->device = device;
    int rc = gpb200_create(&f->eu, device);
    if (rc == GPB200_OK) rc = gpb200_create(&f->es, device);
    if (rc != GPB200_OK) { if (f->eu) gpb200_destroy(f->eu); delete f; return rc; }
    // one stream for both sub-engines
    cudaStreamDestroy(f->es->st);
    f->es->st = f->eu->st; f->es->own_stream = false;
    *out = f;
    return GPB200_OK;
}

const char* gpb200_fitc_last_error(gpb200_fitc* f) { return f ? f->err.c_str() : g_create_error.c_str(); }

int gpb200_fitc_set_data(gpb200_fitc* f, int64_t N, int32_t d, const double* x, int64_t ldx, int64_t M,
                         const double* xu, int64_t ldxu) {
    if (!f) return GPB200_EINVAL;
    if (N <= 0 || M <= 0 || d <= 0 || !x || !xu || ldx < d || ldxu < d) { f->err = "fitc_set_data: bad arguments"; return GPB200_EINVAL; }
    FCK(cudaSetDevice(f->device));
    FSUB(gpb200_set_data(f->eu, M, d, xu, ldxu), f->eu);
    FSUB(gpb200_set_data(f->es, M, d, xu, ldxu), f->es);
    cudaStream_t st = f->eu->st;
    double** ptrs[] = {&f->x, &f->xs, &f->lam, &f->y, &f->alpha, &f->tmpn, &f->w, &f->tmpc, &f->zeroc, &f->tmpc2,
                       &f->bvec, &f->uvec, &f->tmpm, &f->rhsm, &f->scal, &f->bufA, &f->bufB,
                       &f->bufC, &f->Hbuf, &f->Wbuf, &f->Tbuf, &f->gvec, &f->betav, &f->gpart, &f->gacc, &f->gtmp};
    for (auto pp : ptrs) { if (*pp) cudaFree(*pp); *pp = nullptr; }
    f->grad_ws = false;
    f->N = N; f->M = M; f->d = d; f->Mpad = f->eu->Npad;
    // chunk of data rows: two staging buffers of ~2 GB each at most
    int64_t nc = (int64_t)(2.0e9 / (8.0 * (double)f->Mpad)) / TILE * TILE;
    const int64_t Nceil = (N + TILE - 1) / TILE * TILE;
    if (nc > 32768) nc = 32768;                       // grid.y limit of the row-scaling kernel
    if (nc > Nceil) nc = Nceil;
    if (nc < TILE) nc = TILE;
    f->Nc = nc;
    FCK(cudaMalloc(&f->x, sizeof(double) * N * d));
    FCK(cudaMalloc(&f->xs, sizeof(double) * nc * d));
    for (double** p : {&f->lam, &f->y, &f->alpha, &f->tmpn}) FCK(cudaMalloc(p, sizeof(double) * (N + TILE)));
    for (double** p : {&f->w, &f->tmpc, &f->zeroc, &f->tmpc2}) FCK(cudaMalloc(p, sizeof(double) * nc));
    for (double** p : {&f->bvec, &f->uvec, &f->tmpm, &f->rhsm}) FCK(cudaMalloc(p, sizeof(double) * f->Mpad));
    FCK(cudaMalloc(&f->scal, sizeof(double) * 16));
    FCK(cudaMalloc(&f->bufA, sizeof(double) * nc * f->Mpad));
    FCK(cudaMalloc(&f->bufB, sizeof(double) * nc * f->Mpad));
    FCK(cudaMemsetAsync(f->zeroc, 0, sizeof(double) * nc, st));
    FCK(cudaMemcpy2DAsync(f->x, sizeof(double) * d, x, sizeof(double) * ldx, sizeof(double) * d, N, cudaMemcpyHostToDevice, st));
    if (f->eu->tma_ok) {
        const bool ok = gemm_make_tensor_map(&f->mapA, f->bufA, nc, f->Mpad, f->Mpad) &&
                        gemm_make_tensor_map(&f->mapB, f->bufB, f->Mpad, nc, nc) &&
                        gemm_make_tensor_map(&f->mapB2, f->bufB, nc, f->Mpad, f->Mpad);
        if (!ok) { f->err = "fitc_set_data: cuTensorMapEncodeTiled failed"; return GPB200_ECUDA; }
    }
    FCK(cudaStreamSynchronize(st));
    f->has_data = true; f->factored = f->alpha_ready = false;
    return GPB200_OK;
}

int gpb200_fitc_set_kernel(gpb200_fitc* f, int32_t n_ops, const int32_t* ops, int32_t n_dims, const int32_t* dims,
                           int32_t n_theta) {
    if (!f) return GPB200_EINVAL;
    FSUB(gpb200_set_kernel(f->eu, n_ops, ops, n_dims, dims, n_theta), f->eu);
    FSUB(gpb200_set_kernel(f->es, n_ops, ops, n_dims, dims, n_theta), f->es);
    f->has_kernel = true; f->factored = f->alpha_ready = false;
    return GPB200_OK;
}

// K_fu chunk (rows r0..r0+nc of x against the inducing points) into bufA [Nc x Mpad]
static cudaError_t fitc_kfu(gpb200_fitc* f, const double* xrows, int64_t nc) {
    ++f->eu->launches;
    return crossgram_launch(f->eu->prog, xrows, f->d, nc, f->Nc, f->eu->x, f->d, f->M, f->Mpad, f->d, f->bufA, f->Mpad, f->eu->st);
}
// K_uf chunk into bufB [Mpad x Nc]
static cudaError_t fitc_kuf(gpb200_fitc* f, const double* xrows, int64_t nc) {
    ++f->eu->launches;
    return crossgram_launch(f->eu->prog, f->eu->x, f->d, f->M, f->Mpad, xrows, f->d, nc, f->Nc, f->d, f->bufB, f->Nc, f->eu->st);
}

int gpb200_fitc_factorize(gpb200_fitc* f, const double* theta, double log_noise) {
    if (!f) return GPB200_EINVAL;
    if (!f->has_data || !f->has_kernel) { f->err = "fitc_factorize: set_data and set_kernel first"; return GPB200_ESTATE; }
    if (!isfinite(log_noise)) { f->err = "fitc_factorize: non-finite logNoise"; return GPB200_EINVAL; }
    FCK(cudaSetDevice(f->device));
    f->factored = f->alpha_ready = false;
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    // K_uu + 1e-10 I and its factor (fitc.jl:139-141)
    const double ln_off = -1000.0;                          // exp(2*ln) == 0: no noise on K_uu
    FSUB(gpb200_factorize(eu, theta, &ln_off, 1, 1e-10), eu);
    // Sigma_QR starts as K_uu (+ the second 1e-10 nugget of make_posdef!, fitc.jl:153)
    kprog_set_theta(es->prog, theta);
    for (int i = 0; i < es->prog.n_theta; ++i) es->theta[i] = theta[i];
    const double zero = 0.0;
    FCK(cudaMemcpyAsync(es->noise_var, &zero, sizeof(double), cudaMemcpyHostToDevice, st));
    es->n_noise = 1; es->nugget = 2e-10;
    ++es->launches;
    if (f->rank == 0) FCK(gram_lower_launch(es->prog, es->x, f->d, f->d, f->M, f->Mpad, es->noise_var, 1, 2e-10, es->G, es->ld, st));
    else FCK(cudaMemsetAsync(es->G, 0, sizeof(double) * (size_t)f->Mpad * (size_t)f->Mpad, st));     // K_uu (+ nuggets, identity padding) enters the sum once
    f->noise_var = exp(2.0 * log_noise);
    GemmBuf bA{eu->tma_ok ? &f->mapA : nullptr, f->bufA, f->Mpad};
    GemmBuf bB{eu->tma_ok ? &f->mapB : nullptr, f->bufB, f->Nc};
    for (int64_t r0 = 0; r0 < f->N; r0 += f->Nc) {
        const int64_t nc = std::min(f->Nc, f->N - r0);
        const double* xr = f->x + r0 * f->d;
        if (f->mode == 0) {
            // Lambda_i = sigma^2 + K_ii - |L_uu^-1 K_ui|^2   (fitc.jl:146-148)
            FCK(fitc_kfu(f, xr, nc));
            FCK(trsm_rec_buf(eu, bA, (int)f->Nc, 0, (int)f->Mpad));
            eu->launches += 3;
            FCK(kdiag_launch(eu->prog, xr, f->d, nc, f->tmpc, st));
            FCK(rowvar_launch(f->bufA, f->Mpad, f->tmpc, nc, f->Mpad, f->tmpc2, st));
            FCK(ew_launch(0, nc, f->lam + r0, f->tmpc2, nullptr, nullptr, f->noise_var, st));
        } else {
            // SoR / DTC: Lambda = sigma^2 I   (subsetofregressors.jl:100: exp(-2 logNoise) * Kuf * Kfu + Kuu)
            ++eu->launches;
            FCK(ew_launch(0, nc, f->lam + r0, f->zeroc, nullptr, nullptr, f->noise_var, st));
        }
        // Sigma_QR += K_uf Lambda^-1 K_fu   (fitc.jl:150), as (K_uf Lambda^-1/2)(K_uf Lambda^-1/2)'
        FCK(fitc_kuf(f, xr, nc));
        ++eu->launches;
        FCK(scale_launch(0, f->bufB, f->Nc, f->Mpad, nc, f->lam + r0, st));
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bB, bufNone(), 0, 0};
        g.B = GemmOperand{bB, bufNone(), 0, 0};
        g.C = es->G; g.ldc = es->ld; g.M = (int)f->Mpad; g.N = (int)f->Mpad; g.K = (int)f->Nc;
        g.alpha = 1.0; g.beta = 1.0; g.flags = GEMM_LOWER_ONLY;
        FCK(launch_gemm(es, g));
    }
    // multi-GPU: Sigma_QR = K_uu + sum over ranks of K_uf L^-1 K_fu  -- the one M x M exchange of the FITC likelihood
    { int rca = fitc_allreduce(f, es->G, (size_t)f->Mpad * (size_t)f->Mpad); if (rca) return rca; }
    int rc = chol_inplace(es);
    if (rc != GPB200_OK) { f->err = "fitc_factorize (Sigma_QR): " + es->err; return rc; }
    f->factored = true;
    return GPB200_OK;
}

// alpha = Sigma^-1 r (fitc.jl:33-36), logdet (fitc.jl:77), mll (GPE.jl:210)
int gpb200_fitc_mll(gpb200_fitc* f, const double* y_minus_mean, double* alpha, double* mll, double* logdet) {
    if (!f || !y_minus_mean || !mll) return GPB200_EINVAL;
    if (!f->factored) { f->err = "fitc_mll: factorize first"; return GPB200_ESTATE; }
    FCK(cudaSetDevice(f->device));
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    FCK(cudaMemcpyAsync(f->y, y_minus_mean, sizeof(double) * f->N, cudaMemcpyHostToDevice, st));
    // b = K_uf Lambda^-1 r
    FCK(cudaMemsetAsync(f->bvec, 0, sizeof(double) * f->Mpad, st));
    for (int64_t r0 = 0; r0 < f->N; r0 += f->Nc) {
        const int64_t nc = std::min(f->Nc, f->N - r0);
        FCK(fitc_kuf(f, f->x + r0 * f->d, nc));
        eu->launches += 3;
        FCK(cudaMemsetAsync(f->w, 0, sizeof(double) * f->Nc, st));
        FCK(ew_launch(1, nc, f->w, f->y + r0, f->lam + r0, nullptr, 0.0, st));
        FCK(rowdot_launch(f->bufB, f->Nc, f->w, f->M, f->Nc, f->tmpm, st));
        FCK(ew_launch(2, f->M, f->bvec, f->tmpm, nullptr, nullptr, 0.0, st));
    }
    { int rca = fitc_allreduce(f, f->bvec, (size_t)f->Mpad); if (rca) return rca; }              // b summed over the ranks' rows
    // u = Sigma_QR^-1 b   (== get_alpha_u, fitc.jl:279-286)
    FCK(cudaMemcpyAsync(f->rhsm, f->bvec, sizeof(double) * f->Mpad, cudaMemcpyDeviceToDevice, st));
    FCK(solve_device(es, f->rhsm, f->tmpm, f->uvec));
    // alpha = Lambda^-1 (r - K_fu u)
    for (int64_t r0 = 0; r0 < f->N; r0 += f->Nc) {
        const int64_t nc = std::min(f->Nc, f->N - r0);
        FCK(fitc_kfu(f, f->x + r0 * f->d, nc));
        eu->launches += 2;
        FCK(rowdot_launch(f->bufA, f->Mpad, f->uvec, nc, f->Mpad, f->tmpc, st));
        FCK(ew_launch(3, nc, f->alpha + r0, f->y + r0, f->tmpc, f->lam + r0, 0.0, st));
    }
    eu->launches += 5;
    FCK(dot_launch(f->y, f->alpha, f->N, f->scal + 0, st));
    FCK(sum_launch(es->logd, es->Npad, f->scal + 1, st));
    FCK(sum_launch(eu->logd, eu->Npad, f->scal + 2, st));
    FCK(ew_launch(4, f->N, f->tmpn, f->lam, nullptr, nullptr, 0.0, st));
    FCK(sum_launch(f->tmpn, f->N, f->scal + 3, st));
    double s[5];
    if (f->nranks > 1) {
        // r'alpha, sum log Lambda and N are sums over the ranks' rows; the two M x M log-determinants are replicated
        const double nloc = (double)f->N;
        FCK(cudaMemcpyAsync(f->scal + 8, f->scal + 0, sizeof(double), cudaMemcpyDeviceToDevice, st));
        FCK(cudaMemcpyAsync(f->scal + 9, f->scal + 3, sizeof(double), cudaMemcpyDeviceToDevice, st));
        FCK(cudaMemcpyAsync(f->scal + 10, &nloc, sizeof(double), cudaMemcpyHostToDevice, st));
        { int rca = fitc_allreduce(f, f->scal + 8, 3); if (rca) return rca; }
        FCK(cudaMemcpyAsync(f->scal + 0, f->scal + 8, sizeof(double), cudaMemcpyDeviceToDevice, st));
        FCK(cudaMemcpyAsync(f->scal + 3, f->scal + 9, sizeof(double), cudaMemcpyDeviceToDevice, st));
        FCK(cudaMemcpyAsync(f->scal + 4, f->scal + 10, sizeof(double), cudaMemcpyDeviceToDevice, st));
    }
    FCK(cudaMemcpyAsync(s, f->scal, sizeof(double) * 5, cudaMemcpyDeviceToHost, st));
    if (alpha) FCK(cudaMemcpyAsync(alpha, f->alpha, sizeof(double) * f->N, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    f->Ntotal = f->nranks > 1 ? s[4] : (double)f->N;
    const double ld = s[1] - s[2] + s[3];
    if (logdet) *logdet = ld;
    *mll = -(s[0] + ld + LOG2PI * f->Ntotal) / 2.0;
    f->alpha_ready = true;
    return GPB200_OK;
}

// dmll_noise (fitc.jl:243-257): sigma^2 * (alpha.alpha - sum 1/Lambda + |L_s^-1 K_uf Lambda^-1|_F^2)
int gpb200_fitc_grad_noise(gpb200_fitc* f, double* dmll_noise) {
    if (!f || !dmll_noise) return GPB200_EINVAL;
    if (!f->factored || !f->alpha_ready) { f->err = "fitc_grad_noise: factorize and mll first"; return GPB200_ESTATE; }
    FCK(cudaSetDevice(f->device));
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    GemmBuf bA{eu->tma_ok ? &f->mapA : nullptr, f->bufA, f->Mpad};
    for (int64_t r0 = 0; r0 < f->N; r0 += f->Nc) {
        const int64_t nc = std::min(f->Nc, f->N - r0);
        FCK(fitc_kfu(f, f->x + r0 * f->d, nc));
        eu->launches += 2;
        FCK(scale_launch(1, f->bufA, f->Mpad, nc, f->Mpad, f->lam + r0, st));
        FCK(trsm_rec_buf(es, bA, (int)f->Nc, 0, (int)f->Mpad));
        FCK(rowvar_launch(f->bufA, f->Mpad, f->zeroc, nc, f->Mpad, f->tmpn + r0, st));     // = -|row|^2
    }
    eu->launches += 4;
    FCK(sum_launch(f->tmpn, f->N, f->scal + 0, st));
    FCK(dot_launch(f->alpha, f->alpha, f->N, f->scal + 1, st));
    FCK(ew_launch(5, f->N, f->tmpn, f->lam, nullptr, nullptr, 0.0, st));
    FCK(sum_launch(f->tmpn, f->N, f->scal + 2, st));
    { int rca = fitc_allreduce(f, f->scal, 3); if (rca) return rca; }                             // sums over the ranks' rows
    double s[3];
    FCK(cudaMemcpyAsync(s, f->scal, sizeof(double) * 3, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    *dmll_noise = f->noise_var * (s[1] - s[2] - s[0]);
    return GPB200_OK;
}

// predictive mean / variance (fitc.jl:324-332 -> dtc.jl:41-59 -> sor.jl:302-321):
//   mu = K_xu u ;  var = k_xx - |L_uu^-1 k_ux|^2 + |L_s^-1 k_ux|^2
int gpb200_fitc_predict(gpb200_fitc* f, int64_t Ms, const double* xs, int64_t ldxs, double* mu, double* var) {
    if (!f || Ms <= 0 || !xs || ldxs < f->d || !mu) return GPB200_EINVAL;
    if (!f->factored || !f->alpha_ready) { f->err = "fitc_predict: factorize and mll first"; return GPB200_ESTATE; }
    FCK(cudaSetDevice(f->device));
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    GemmBuf bA{eu->tma_ok ? &f->mapA : nullptr, f->bufA, f->Mpad};
    GemmBuf bB2{eu->tma_ok ? &f->mapB2 : nullptr, f->bufB, f->Mpad};
    for (int64_t m0 = 0; m0 < Ms; m0 += f->Nc) {
        const int64_t mc = std::min(f->Nc, Ms - m0);
        FCK(cudaMemcpy2DAsync(f->xs, sizeof(double) * f->d, xs + m0 * ldxs, sizeof(double) * ldxs, sizeof(double) * f->d,
                              mc, cudaMemcpyHostToDevice, st));
        FCK(fitc_kfu(f, f->xs, mc));
        ++eu->launches;
        FCK(rowdot_launch(f->bufA, f->Mpad, f->uvec, mc, f->Mpad, f->tmpc, st));
        FCK(cudaMemcpyAsync(mu + m0, f->tmpc, sizeof(double) * mc, cudaMemcpyDeviceToHost, st));
        if (var) {
            FCK(cudaMemcpyAsync(f->bufB, f->bufA, sizeof(double) * f->Nc * f->Mpad, cudaMemcpyDeviceToDevice, st));
            FCK(trsm_rec_buf(eu, bA, (int)f->Nc, 0, (int)f->Mpad));
            FCK(trsm_rec_buf(es, bB2, (int)f->Nc, 0, (int)f->Mpad));
            eu->launches += 4;
            FCK(kdiag_launch(eu->prog, f->xs, f->d, mc, f->tmpc, st));
            FCK(rowvar_launch(f->bufA, f->Mpad, f->tmpc, mc, f->Mpad, f->tmpc2, st));       // k_xx - q
            FCK(rowvar_launch(f->bufB, f->Mpad, f->zeroc, mc, f->Mpad, f->w, st));          // -s
            if (f->mode == 2) {                                                             // SoR: K_xu S^-1 K_ux only (sor.jl:302-321)
                FCK(cudaMemsetAsync(f->tmpc2, 0, sizeof(double) * mc, st));
            }
            FCK(ew_launch(6, mc, f->tmpc, f->tmpc2, f->w, nullptr, 0.0, st));               // [k_xx - q] + s
            FCK(cudaMemcpyAsync(var + m0, f->tmpc, sizeof(double) * mc, cudaMemcpyDeviceToHost, st));
        }
        FCK(cudaStreamSynchronize(st));
    }
    return GPB200_OK;
}


// predictMVN with the FULL predictive covariance (fitc.jl:324-332 -> determ_train_conditional.jl:41-59 ->
// subsetofregressors.jl:302-321):  Sigma* = K** - K*u K_uu^-1 Ku* + K*u S^-1 Ku*   (FITC, DTC);   K*u S^-1 Ku*   (SoR)
// = K** - A A' + B B' with A = K*u L_uu^-T, B = K*u L_s^-T: two whitening TRSMs and two NT GEMMs.  Ms <= one staging chunk.
int gpb200_fitc_predict_cov(gpb200_fitc* f, int64_t Ms, const double* xs, int64_t ldxs, double* mu, double* cov) {
    if (!f || Ms <= 0 || !xs || ldxs < f->d || !mu || !cov) return GPB200_EINVAL;
    if (!f->factored || !f->alpha_ready) { f->err = "fitc_predict_cov: factorize and mll first"; return GPB200_ESTATE; }
    if (Ms > f->Nc) { f->err = "fitc_predict_cov: too many test points for one staging chunk"; return GPB200_EINVAL; }
    FCK(cudaSetDevice(f->device));
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    const int64_t Mspad = (Ms + TILE - 1) / TILE * TILE;
    if (Mspad > f->Kss_rows) {
        if (f->Kss) cudaFree(f->Kss);
        f->Kss = nullptr; f->Kss_rows = 0;
        FCK(cudaMalloc(&f->Kss, sizeof(double) * Mspad * Mspad));
        f->Kss_rows = Mspad;
    }
    GemmBuf bA{eu->tma_ok ? &f->mapA : nullptr, f->bufA, f->Mpad};
    GemmBuf bB2{eu->tma_ok ? &f->mapB2 : nullptr, f->bufB, f->Mpad};
    FCK(cudaMemcpy2DAsync(f->xs, sizeof(double) * f->d, xs, sizeof(double) * ldxs, sizeof(double) * f->d, Ms, cudaMemcpyHostToDevice, st));
    FCK(fitc_kfu(f, f->xs, Ms));                                         // bufA = K*u  (Ms x Mpad, zero padded rows)
    ++eu->launches;
    FCK(rowdot_launch(f->bufA, f->Mpad, f->uvec, Ms, f->Mpad, f->tmpc, st));
    FCK(cudaMemcpyAsync(mu, f->tmpc, sizeof(double) * Ms, cudaMemcpyDeviceToHost, st));
    FCK(cudaMemcpyAsync(f->bufB, f->bufA, sizeof(double) * f->Nc * f->Mpad, cudaMemcpyDeviceToDevice, st));
    FCK(trsm_rec_buf(es, bB2, (int)Mspad, 0, (int)f->Mpad));             // B = K*u L_s^-T
    ++eu->launches;
    if (f->mode != 2) {
        FCK(trsm_rec_buf(eu, bA, (int)Mspad, 0, (int)f->Mpad));         // A = K*u L_uu^-T
        FCK(gram_full_launch(eu->prog, f->xs, f->d, Ms, Mspad, f->d, f->Kss, Mspad, st));
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bA, bufNone(), 0, 0};
        g.B = GemmOperand{bA, bufNone(), 0, 0};
        g.C = f->Kss; g.ldc = Mspad; g.M = (int)Mspad; g.N = (int)Mspad; g.K = (int)f->Mpad;
        g.alpha = -1.0; g.beta = 1.0;
        FCK(launch_gemm(eu, g));
    } else {
        FCK(cudaMemsetAsync(f->Kss, 0, sizeof(double) * Mspad * Mspad, st));
    }
    {
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bB2, bufNone(), 0, 0};
        g.B = GemmOperand{bB2, bufNone(), 0, 0};
        g.C = f->Kss; g.ldc = Mspad; g.M = (int)Mspad; g.N = (int)Mspad; g.K = (int)f->Mpad;
        g.alpha = 1.0; g.beta = 1.0;
        FCK(launch_gemm(es, g));
    }
    FCK(cudaMemcpy2DAsync(cov, sizeof(double) * Ms, f->Kss, sizeof(double) * Mspad, sizeof(double) * Ms, Ms, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    return GPB200_OK;
}

// Kernel-parameter gradient of the FITC mll: dmll_kern!(::FullyIndepStrat) (fitc.jl:200-234) on top of
// dmll_kern!(::SubsetOfRegsStrategy) (subsetofregressors.jl:219-253), regrouped so that every
// parameter shares the same three weighted traces (kernel derivatives recomputed on the fly):
//   dmll_p = 1/2 [ <W_fu, dK_fu/dθ_p> + <W_uu, dK_uu/dθ_p> + sum_i g_i dK_ii/dθ_p ]
//   g_i   = alpha_i^2 - (Sigma^-1)_ii ,  (Sigma^-1)_ii = 1/L_i - K_fu,i S^-1 K_uf,i / L_i^2      (trinvAB, fitc.jl:63-67)
//   W_fu  = 2 alpha beta' - 2 L^-1 K_fu S^-1 - 2 diag(g) K_fu K_uu^-1 ,  beta = K_uu^-1 K_uf alpha   (sor.jl:147)
//   W_uu  = -beta beta' + K_uu^-1 - S^-1 + K_uu^-1 (K_uf diag(g) K_fu) K_uu^-1
// with S = Sigma_QR, L = Lambda; uses Sigma^-1 K_fu K_uu^-1 = L^-1 K_fu S^-1 and
// K_uu^-1 K_uf Sigma^-1 K_fu K_uu^-1 = K_uu^-1 - S^-1 (both follow from S = K_uu + K_uf L^-1 K_fu).
// All O(M^2 N) work is NT GEMMs against the explicit M x M inverses (grad_prepare of the sub-engines).
int gpb200_fitc_grad_kernel(gpb200_fitc* f, double* dmll_kernel) {
    if (!f || !dmll_kernel) return GPB200_EINVAL;
    if (!f->factored || !f->alpha_ready) { f->err = "fitc_grad_kernel: factorize and mll first"; return GPB200_ESTATE; }
    FCK(cudaSetDevice(f->device));
    gpb200_handle *eu = f->eu, *es = f->es;
    cudaStream_t st = eu->st;
    const int np = eu->prog.n_theta;
    const int64_t Mp = f->Mpad, Nc = f->Nc;
    if (!f->grad_ws) {
        FCK(cudaMalloc(&f->bufC, sizeof(double) * Nc * Mp));
        for (double** p : {&f->Hbuf, &f->Wbuf, &f->Tbuf}) FCK(cudaMalloc(p, sizeof(double) * Mp * Mp));
        FCK(cudaMalloc(&f->gvec, sizeof(double) * (f->N + TILE)));
        FCK(cudaMalloc(&f->betav, sizeof(double) * Mp));
        const size_t tiles = (size_t)std::max((Nc / TILE) * (Mp / TILE), (Mp / TILE) * (Mp / TILE));
        FCK(cudaMalloc(&f->gpart, sizeof(double) * tiles * GPB200_MAX_THETA));
        FCK(cudaMalloc(&f->gacc, sizeof(double) * GPB200_MAX_THETA));
        FCK(cudaMalloc(&f->gtmp, sizeof(double) * GPB200_MAX_THETA));
        if (eu->tma_ok) {
            const bool ok = gemm_make_tensor_map(&f->mapAt, f->bufA, Mp, Nc, Nc) && gemm_make_tensor_map(&f->mapC, f->bufC, Nc, Mp, Mp) &&
                            gemm_make_tensor_map(&f->mapCt, f->bufC, Mp, Nc, Nc) && gemm_make_tensor_map(&f->mapH, f->Hbuf, Mp, Mp, Mp) &&
                            gemm_make_tensor_map(&f->mapT, f->Tbuf, Mp, Mp, Mp);
            if (!ok) { f->err = "fitc_grad_kernel: cuTensorMapEncodeTiled failed"; return GPB200_ECUDA; }
        }
        f->grad_ws = true;
    }
    // explicit K_uu^-1 and Sigma_QR^-1 (full symmetric) in the sub-engines' G buffers
    FSUB(gpb200_grad_prepare(eu), eu);
    FSUB(gpb200_grad_prepare(es), es);
    eu->launches += 2;
    FCK(symmetrize_launch(eu->G, eu->ld, Mp, st));
    FCK(symmetrize_launch(es->G, es->ld, Mp, st));
    const bool tma = eu->tma_ok;
    GemmBuf bA{tma ? &f->mapA : nullptr, f->bufA, Mp}, bAt{tma ? &f->mapAt : nullptr, f->bufA, Nc};
    GemmBuf bCt{tma ? &f->mapCt : nullptr, f->bufC, Nc};
    GemmBuf bH{tma ? &f->mapH : nullptr, f->Hbuf, Mp}, bT{tma ? &f->mapT : nullptr, f->Tbuf, Mp};
    // beta = K_uu^-1 (K_uf alpha)
    FCK(cudaMemsetAsync(f->rhsm, 0, sizeof(double) * Mp, st));
    for (int64_t r0 = 0; r0 < f->N; r0 += Nc) {
        const int64_t nc = std::min(Nc, f->N - r0);
        FCK(fitc_kuf(f, f->x + r0 * f->d, nc));
        eu->launches += 2;
        FCK(cudaMemsetAsync(f->w, 0, sizeof(double) * Nc, st));
        FCK(cudaMemcpyAsync(f->w, f->alpha + r0, sizeof(double) * nc, cudaMemcpyDeviceToDevice, st));
        FCK(rowdot_launch(f->bufB, Nc, f->w, f->M, Nc, f->tmpm, st));
        FCK(ew_launch(2, f->M, f->rhsm, f->tmpm, nullptr, nullptr, 0.0, st));
    }
    { int rca = fitc_allreduce(f, f->rhsm, (size_t)Mp); if (rca) return rca; }                    // K_uf alpha over all rows
    FCK(solve_device(eu, f->rhsm, f->tmpm, f->betav));
    FCK(cudaMemsetAsync(f->gacc, 0, sizeof(double) * GPB200_MAX_THETA, st));
    FCK(cudaMemsetAsync(f->Hbuf, 0, sizeof(double) * Mp * Mp, st));
    for (int64_t r0 = 0; r0 < f->N; r0 += Nc) {
        const int64_t nc = std::min(Nc, f->N - r0);
        const double* xr = f->x + r0 * f->d;
        FCK(fitc_kfu(f, xr, nc));                                         // bufA = K_fu chunk
        {   // P2 = K_fu S^-1 -> bufB (as Nc x Mpad)
            GemmDesc g = gemm_desc_default();
            g.A = GemmOperand{bA, bufNone(), 0, 0};
            g.B = GemmOperand{bufG(es), bufNone(), 0, 0};
            g.C = f->bufB; g.ldc = Mp; g.M = (int)Nc; g.N = (int)Mp; g.K = (int)Mp;
            FCK(launch_gemm(es, g));
        }
        eu->launches += 2;
        FCK(rowdot2_launch(f->bufA, f->bufB, Mp, nc, Mp, f->tmpc, st));
        if (f->mode == 0) FCK(fitc_g_launch(nc, f->alpha + r0, f->lam + r0, f->tmpc, f->gvec + r0, st));
        else FCK(cudaMemsetAsync(f->gvec + r0, 0, sizeof(double) * nc, st));       // SoR part only (sor.jl:219-253)
        {   // P1 = K_fu K_uu^-1 -> bufC
            GemmDesc g = gemm_desc_default();
            g.A = GemmOperand{bA, bufNone(), 0, 0};
            g.B = GemmOperand{bufG(eu), bufNone(), 0, 0};
            g.C = f->bufC; g.ldc = Mp; g.M = (int)Nc; g.N = (int)Mp; g.K = (int)Mp;
            FCK(launch_gemm(eu, g));
        }
        eu->launches += 4;
        FCK(fitc_wfu_launch(f->bufB, f->bufC, Mp, nc, f->M, f->alpha + r0, f->lam + r0, f->gvec + r0, f->betav, st));
        FCK(trace_rect_launch(eu->prog, xr, f->d, nc, eu->x, f->d, f->M, f->d, f->bufB, Mp, f->gpart, f->gtmp, st));
        FCK(ew_launch(2, np, f->gacc, f->gtmp, nullptr, nullptr, 0.0, st));
        if (f->mode != 0) continue;                                       // no Lambda-derivative terms for SoR / DTC
        // diagonal term sum_i g_i dK_ii/dθ_p (scratch: bufC as np x nc)
        FCK(kdiag_grad_launch(eu->prog, xr, f->d, nc, f->gvec + r0, f->bufC, st));
        for (int p = 0; p < np; ++p) { ++eu->launches; FCK(sum_launch(f->bufC + (size_t)p * nc, nc, f->gtmp + p, st)); }
        FCK(ew_launch(2, np, f->gacc, f->gtmp, nullptr, nullptr, 0.0, st));
        // H += K_uf diag(g) K_fu
        ++eu->launches;
        FCK(crossgram_launch(eu->prog, eu->x, f->d, f->M, Mp, xr, f->d, nc, Nc, f->d, f->bufA, Nc, st));   // bufA = K_uf chunk (Mpad x Nc)
        FCK(cudaMemcpyAsync(f->bufC, f->bufA, sizeof(double) * Mp * Nc, cudaMemcpyDeviceToDevice, st));
        ++eu->launches;
        FCK(colscale_launch(f->bufC, Nc, Mp, nc, f->gvec + r0, st));
        {
            GemmDesc g = gemm_desc_default();
            g.A = GemmOperand{bAt, bufNone(), 0, 0};
            g.B = GemmOperand{bCt, bufNone(), 0, 0};
            g.C = f->Hbuf; g.ldc = Mp; g.M = (int)Mp; g.N = (int)Mp; g.K = (int)Nc;
            g.alpha = 1.0; g.beta = 1.0;
            FCK(launch_gemm(eu, g));
        }
    }
    // multi-GPU: the per-row traces and H = K_uf diag(g) K_fu are sums over the ranks' rows; the M x M part below is replicated
    { int rca = fitc_allreduce(f, f->gacc, (size_t)np); if (rca) return rca; }
    { int rca = fitc_allreduce(f, f->Hbuf, (size_t)Mp * (size_t)Mp); if (rca) return rca; }
    {   // T = K_uu^-1 H ; Wbuf = K_uu^-1 T' = K_uu^-1 H K_uu^-1
        GemmDesc g = gemm_desc_default();
        g.A = GemmOperand{bufG(eu), bufNone(), 0, 0};
        g.B = GemmOperand{bH, bufNone(), 0, 0};
        g.C = f->Tbuf; g.ldc = Mp; g.M = (int)Mp; g.N = (int)Mp; g.K = (int)Mp;
        FCK(launch_gemm(eu, g));
        g.B = GemmOperand{bT, bufNone(), 0, 0};
        g.C = f->Wbuf;
        FCK(launch_gemm(eu, g));
    }
    eu->launches += 4;
    FCK(fitc_wuu_launch(f->Wbuf, f->Wbuf, eu->G, es->G, Mp, f->M, f->betav, st));
    FCK(trace_rect_launch(eu->prog, eu->x, f->d, f->M, eu->x, f->d, f->M, f->d, f->Wbuf, Mp, f->gpart, f->gtmp, st));
    FCK(ew_launch(2, np, f->gacc, f->gtmp, nullptr, nullptr, 0.0, st));
    std::vector<double> out((size_t)std::max(np, 1));
    FCK(cudaMemcpyAsync(out.data(), f->gacc, sizeof(double) * np, cudaMemcpyDeviceToHost, st));
    FCK(cudaStreamSynchronize(st));
    for (int p = 0; p < np; ++p) dmll_kernel[p] = 0.5 * out[p];
    return GPB200_OK;
}

int gpb200_fitc_set_mode(gpb200_fitc* f, int mode) {
    if (!f || mode < 0 || mode > 2) return GPB200_EINVAL;
    f->mode = mode; f->factored = f->alpha_ready = false;
    return GPB200_OK;
}

int64_t gpb200_fitc_launch_count(gpb200_fitc* f) { return f ? f->eu->launches + f->es->launches : 0; }

}  // extern "C"
