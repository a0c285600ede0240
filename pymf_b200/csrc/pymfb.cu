// pymfb.cu - context, scheduling of the per-iteration kernels, and the C ABI (include/pymfb.h).
//
// Path served: pymf.NMF.factorize -> update_w / update_h / frobenius_norm / converged
// (pymf/nmf.py:100-202).  State kept on the device between iterations:
//   W (d x kp), H (kp x ldh) ping-pong pairs; P = [X H^T | H H^T] local partials;
//   AB = the same after the all-reduce over ranks; G = W^T W; ||X||^2.
// One iteration (W, then H, then error - the reference's order, :183-190):
//   W  <- W * A / (W B + 1e-9)                 k_update_w           (replicated, O(d k^2))
//   G  <- W^T W                                k_ltr_partial + sum  (replicated, O(d k^2))
//   H  <- H * (W^T X) / (G H + 1e-9)           H-update pass        (streams X)
//   P  <- [X H^T | H H^T]                      X H^T pass           (streams X)
//   AB <- allreduce(P)                         NCCL (world > 1)
//   ferr_i = sqrt(xx - 2<W,A> + <G,B>)         k_err (fp64), device-side stop flag
#include <cuda_runtime.h>
#include <chrono>
#include <dlfcn.h>
#include <immintrin.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <ctype.h>
#include <stdlib.h>
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/pymfb.h"
#include "common.cuh"
#include "kernels_simt.cuh"
#include "kernels_tc.cuh"
#include "kernels_ts2.cuh"
#include "kernels_tc2.cuh"
#include "kernels_fused.cuh"
#include "kernels_svd.cuh"
#include "kernels_sparse.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

using namespace pymfb;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
static int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return 1;
}
#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e_ = (call);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return fail("%s:%d %s -> %s%s", __FILE__, __LINE__, #call, cudaGetErrorString(e_), fault_note()); \
    } while (0)
// Device-side watchdogs (bounded barrier / flag waits in the persistent kernels) leave a note in this mapped
// host buffer before they trap, so that a protocol bug reads "which wait, which CTA" instead of only
// "unspecified launch failure".  [0] = code (0 = none), [1] = CTA, [2] = aux, [3] = thread.
static int* g_fault_host = nullptr;
static int* g_fault_dev = nullptr;
static int* fault_buffer() {
    if (!g_fault_host) {
        if (cudaHostAlloc((void**)&g_fault_host, 64 * sizeof(int), cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); g_fault_host = nullptr; return nullptr; }
        memset(g_fault_host, 0, 64 * sizeof(int));
        if (cudaHostGetDevicePointer((void**)&g_fault_dev, g_fault_host, 0) != cudaSuccess) { cudaGetLastError(); g_fault_dev = nullptr; }
    }
    return g_fault_dev;
}
static const char* fault_note() {
    static thread_local char buf[160];
    buf[0] = 0;
    if (g_fault_host && g_fault_host[0] != 0)
        snprintf(buf, sizeof(buf), " [device watchdog: wait code %d, CTA %d, aux %d, thread %d]", g_fault_host[0], g_fault_host[1],
                 g_fault_host[2], g_fault_host[3]);
    return buf;
}
#define CK(call)                      \
    do {                              \
        int r_ = (call);              \
        if (r_ != 0) return r_;       \
    } while (0)

// ------------------------------------------------------------------------------------------
// NCCL through dlopen (so that the library loads on a box without NCCL / without a GPU)
// ------------------------------------------------------------------------------------------
struct Uid128 { char b[128]; };   // ncclUniqueId (passed by value)
namespace {
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(void*) = nullptr;
    int (*CommInitRank)(void**, int, Uid128, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
    int (*CommDestroy)(void*) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    // optional (NCCL >= 2.19): user-buffer registration, so that the all-reduce runs in place on the buffer the
    // pass epilogues write (zero-copy / NVLS-capable) instead of staging through NCCL's own buffers
    int (*MemAlloc)(void**, size_t) = nullptr;
    int (*MemFree)(void*) = nullptr;
    int (*CommRegister)(void*, void*, size_t, void**) = nullptr;
    int (*CommDeregister)(void*, void*) = nullptr;
};
}  // namespace
static NcclApi g_nccl;
static const int kNcclFloat32 = 7, kNcclFloat64 = 8, kNcclSum = 0;

static int nccl_load() {
    if (g_nccl.lib) return 0;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* h = nullptr;
    for (const char* nm : names) { h = dlopen(nm, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL); if (h) break; }
    if (!h) for (const char* nm : names) { h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
    if (!h) return fail("cannot dlopen libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(void*))dlsym(h, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void**, int, Uid128, int))dlsym(h, "ncclCommInitRank");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))dlsym(h, "ncclAllReduce");
    g_nccl.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
    g_nccl.MemAlloc = (int (*)(void**, size_t))dlsym(h, "ncclMemAlloc");
    g_nccl.MemFree = (int (*)(void*))dlsym(h, "ncclMemFree");
    g_nccl.CommRegister = (int (*)(void*, void*, size_t, void**))dlsym(h, "ncclCommRegister");
    g_nccl.CommDeregister = (int (*)(void*, void*))dlsym(h, "ncclCommDeregister");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy)
        return fail("libnccl is missing required symbols");
    g_nccl.lib = h;
    return 0;
}
#define NC(call)                                                                         \
    do {                                                                                 \
        int r_ = (call);                                                                 \
        if (r_ != 0)                                                                     \
            return fail("%s:%d %s -> nccl error %d (%s)", __FILE__, __LINE__, #call, r_, \
                        g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?");        \
    } while (0)

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
// Host-side scheduling state that decides which kernels an iteration launches and on which buffers.
struct LoopState {
    int wcur, hcur; bool ab, g, xx, hs0, hs1; int ht;
    bool operator==(const LoopState& o) const {
        return wcur == o.wcur && hcur == o.hcur && ab == o.ab && g == o.g && xx == o.xx && hs0 == o.hs0 && hs1 == o.hs1 &&
               ht == o.ht;
    }
};

// Sparse X on the device (kernels_sparse.cuh): CSC and the column-panel CSR built from it.
struct SparseX {
    int64_t nnz = 0;
    int64_t* colptr = nullptr;     // n_local + 1
    int32_t* rowidx = nullptr;     // nnz
    float* vals = nullptr;         // nnz rounded up to a multiple of 4, zero-padded
    int64_t pw = 0;                // columns per CSR panel
    int npanels = 0;
    int64_t* rowptr = nullptr;     // npanels * d + 1
    int32_t* ccol = nullptr;       // nnz: column of each CSR entry
    float* cval = nullptr;         // nnz
};
static void sparse_free(SparseX& s) {
    cudaFree(s.colptr); cudaFree(s.rowidx); cudaFree(s.vals); cudaFree(s.rowptr); cudaFree(s.ccol); cudaFree(s.cval);
    s = SparseX();
}

struct pymfb_ctx {
    int device = 0;
    int64_t d = 0, n_loc = 0, n_glob = 0, col0 = 0;
    int k = 0, kp = 0, kb = 0;     // kp: padded k; kb: SIMT k block
    int sm_count = 148;
    cudaStream_t stream = nullptr;

    const float* X = nullptr;      // d x ldx
    float* X_own = nullptr;
    int64_t own_ldx = 0, own_xps = 0;    // layout of X_own (ensure_own_x)
    int own_xsh = kNoPanelShift;
    size_t own_bytes = 0;
    int64_t xps = 0;               // layout of X (common.cuh): floats between column panels, 0 = row-major
    int xsh = kNoPanelShift;       // log2(panel width)
    int64_t ldx = 0;

    float* W[2] = {nullptr, nullptr};   // d x kp
    float* H[2] = {nullptr, nullptr};   // kp x ldh
    int wcur = 0, hcur = 0;
    int64_t ldh = 0;
    bool w_set = false, h_set = false;

    float* P = nullptr;            // [A (d x kp) | B (kp x kp)]: local partials, all-reduced IN PLACE over the ranks
    float* AB = nullptr;           // alias of P (the reduced values)
    bool p_nccl = false;           // P comes from ncclMemAlloc and is registered with the communicator
    void* p_reg = nullptr;         // ncclCommRegister handle
    int64_t ab_count = 0;
    float* G = nullptr;            // kp x kp
    float* Gpart = nullptr;        // g_splits x kp x kp
    int g_splits = 1;
    int64_t g_rows_per_split = 0;
    double* red_scratch = nullptr; // fp64 block partials (k_err, k_xx)
    DevState* st = nullptr;
    double* ferr_dev = nullptr;
    int ferr_cap = 0;
    float* flush_buf = nullptr;
    size_t flush_bytes = 0;

    // error mode: direct residual for small problems, trace identity otherwise
    bool err_direct = false;
    int err_mode_opt = PYMFB_ERR_AUTO;     // what pymfb_set_option(PYMFB_OPT_ERR_MODE) asked for
    bool err_auto_switched = false;        // err_direct was turned on by note_cancellation
    float* Wt = nullptr;           // kp x ldwt (direct mode)
    int64_t ldwt = 0;
    double* resid_part = nullptr;

    bool ab_valid = false;         // AB matches the current H (and X)
    bool p_zeroed = false;         // P was cleared by the SIMT H-update kernel and not written since
    bool g_valid = false;          // G matches the current W
    bool xx_valid = false;

    int path_opt = PYMFB_PATH_AUTO;
    int path = PYMFB_PATH_SIMT;
    TcPlan tc;                     // tensor-core plan (kernels_tc.cuh)
    FusedPlan fused;               // one-pass kernel plan (kernels_fused.cuh)

    void* comm = nullptr;
    bool comm_owned = true;        // false: attached by pymfb_comm_attach, the caller destroys it
    int world = 1, rank = 0;

    int64_t launches = 0;
    int nndsvd_path_opt = PYMFB_PATH_AUTO;
    int nndsvd_path = 0;                  // pass family of the last pymfb_nndsvd (PYMFB_PATH_SIMT / _TC), 0 = none yet
    double nndsvd_change = 0.0;           // its last sweep-to-sweep change of the Ritz values (pymfb_nndsvd_info)
    float* xpart_simt = nullptr;         // SIMT X H^T pass: copies of [A | B] for the deterministic combine of the column splits
    bool deterministic_simt = true;       // PYMFB_DETERMINISTIC=0: fp32 atomics
    bool uw_smem_set = false;      // k_update_w's dynamic shared memory attribute raised (k > 1536)
    bool last_upload_pinned = false;
    cudaEvent_t panel_ev[2] = {nullptr, nullptr};     // panel-streamed ingest: last DMA that read panel buffer `slot`
    void* panel_stage[2] = {nullptr, nullptr};        // fp64 panels: device staging for the cast
    size_t panel_stage_bytes[2] = {0, 0};
    bool panel_open = false;
    void* stage = nullptr;         // factor transfer staging (factor_stage)
    size_t stage_bytes = 0;

    // SIMT H-update: splits of the contraction over d when there are few column tiles (k_h_update_simt)
    int hsplit = 1;
    int64_t h_rows_per_split = 0;
    float* h_cpart = nullptr;      // tiles x hsplit x KB x TILE_N partial W^T X
    unsigned* h_tickets = nullptr; // one arrival counter per (column tile, k block)

    // Semi-NMF (pymf/snmf.py): variant switch and its buffers (allocated by pymfb_set_variant)
    int variant = PYMFB_VARIANT_NMF;
    float* Gpos = nullptr;         // kp x kp   (|G| + G)/2
    float* Gneg = nullptr;         // kp x kp   (|G| - G)/2
    float* Dp = nullptr;           // kp x ldh  G+ H  (tensor-core path only)
    float* Dn = nullptr;           // kp x ldh  G- H
    double* inv_work = nullptr;    // k x 2k    Gauss-Jordan tableau
    double* Binv = nullptr;        // k x k     (H H^T)^-1

    // CUDA graph of two steady-state iterations (launch-bound problems), see graph_build
    int graph_opt = PYMFB_GRAPH_AUTO;
    cudaGraphExec_t graph_exec = nullptr;
    unsigned graph_key = 0;
    LoopState graph_state = {0, 0, false, false, false, false, false, -1};
    int64_t graph_launches = 0, graph_replays = 0;

    // BNMF penalty (pymf/bnmf.py:70-90): weights of the current iteration and their growth per H update; 0 = NMF
    double lam_w = 0.0, lam_h = 0.0, inc_w = 1.0, inc_h = 1.0;

    // sparse X (pymfb_upload_x_csc): current instead of X while `sparse`
    bool sparse = false;
    SparseX sx;
    float* Ht = nullptr;           // n_loc x kp: H^T of H[ht_of] (-1: of neither buffer), gathered by the X H^T pass
    int ht_of = -1;
    float* GH = nullptr;           // kp x ldh: G H for the sparse H update (NMF / BNMF)
    float* hh_part = nullptr;      // hh_splits x kp x kp: row-split partials of H H^T = (H^T)^T H^T
    int hh_splits = 1;
    int64_t hh_rows_per_split = 0;

    // per-kernel timing (CUDA events on the launch stream)
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev[2];
    std::vector<cudaEvent_t> ev_pool;
};

// d * n_local * kp at or below which the error is a direct residual pass (2^28 MACs ~ a few us)
static const double kDirectErrMaxWork = 268435456.0;
static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
// Leading dimension of a row-major matrix with n columns: a multiple of 32 floats, plus PYMFB_LD_PAD floats
// (experiment knob, default 0) when the plain value is a large power-of-two multiple.
static inline int64_t padded_ld(int64_t n) {
    int64_t ld = round_up(n, 32);
    static const int64_t pad = [] { const char* e = getenv("PYMFB_LD_PAD"); return e ? (int64_t)atoll(e) : (int64_t)0; }();
    if (pad > 0 && ld % 4096 == 0) ld += round_up(pad, 32);
    return ld;
}
static inline int grid_for(int64_t count, int block, int cap) {
    int64_t g = (count + block - 1) / block;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, cap));
}

static int plan_tc(pymfb_ctx* c) {
    if (tc_plan(c->tc, c->device, c->sm_count, c->d, c->n_loc, c->k, c->kp, c->X, c->ldx, c->ldh, c->H[0], c->H[1], c->xps, c->xsh))
        return fail("tcgen05 plan failed: %s", c->tc.err.c_str());
    if (ts2_prepare(c->tc)) return fail("CTA-pair kernel setup failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (tc2_prepare(c->tc)) return fail("CTA-pair SS kernel setup failed: %s", cudaGetErrorString(cudaGetLastError()));
    fused_release(c->fused);
    if (fused_wanted(c->tc) && fused_plan(c->fused, c->tc)) return fail("fused-kernel plan failed: %s", cudaGetErrorString(cudaGetLastError()));
    return 0;
}

static int timing_begin(pymfb_ctx* c, int which, cudaEvent_t* e0, cudaEvent_t* e1) {
    *e0 = *e1 = nullptr;
    if (!c->timing || c->ev[which].size() >= 4096) return 0;
    CU(cudaEventCreate(e0));
    CU(cudaEventCreate(e1));
    CU(cudaEventRecord(*e0, c->stream));
    return 0;
}
static int timing_end(pymfb_ctx* c, int which, cudaEvent_t e0, cudaEvent_t e1) {
    if (!e0) return 0;
    CU(cudaEventRecord(e1, c->stream));
    c->ev[which].push_back({e0, e1});
    return 0;
}

// ------------------------------------------------------------------------------------------
// kernel scheduling helpers
// ------------------------------------------------------------------------------------------
static int resolve_path(pymfb_ctx* c) {
    if (c->sparse) {
        if (c->path_opt == PYMFB_PATH_SIMT || c->path_opt == PYMFB_PATH_TC)
            return fail("sparse data runs on its own passes: the dense kernel families (path simt / tc) do not apply");
        c->path = PYMFB_PATH_SPARSE;
        return 0;
    }
    std::string why;
    bool ok = tc_supported(c->d, c->n_loc, c->kp, c->ldx, c->X, &why);
    if (c->path_opt == PYMFB_PATH_SIMT) { c->path = PYMFB_PATH_SIMT; return 0; }
    if (c->path_opt == PYMFB_PATH_TC) {
        if (!ok) return fail("tcgen05 path not available for this shape: %s", why.c_str());
        c->path = PYMFB_PATH_TC;
        return 0;
    }
    c->path = ok ? PYMFB_PATH_TC : PYMFB_PATH_SIMT;
    return 0;
}

// G = W^T W (deterministic two-stage sum)
static int launch_gram_w(pymfb_ctx* c) {
    const float* W = c->W[c->wcur];
    dim3 grid((unsigned)((c->kp + TILE_N - 1) / TILE_N), (unsigned)(c->kp / c->kb), (unsigned)c->g_splits);
    if (c->kb == 16)
        k_ltr_partial_simt<16><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, W, c->kp, W, c->kp, c->kp, c->d,
                                                                     c->g_rows_per_split, c->Gpart, c->kp, c->kp);
    else
        k_ltr_partial_simt<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, W, c->kp, W, c->kp, c->kp, c->d,
                                                                     c->g_rows_per_split, c->Gpart, c->kp, c->kp);
    const int64_t cnt = (int64_t)c->kp * c->kp;
    k_sum_partials<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>(c->st, c->Gpart, c->g_splits, cnt, c->G);
    c->launches += 2;
    CU(cudaGetLastError());
    if (c->path == PYMFB_PATH_TC && tc_after_gram(c->tc, c->st, c->W[c->wcur], c->G, c->stream, &c->launches)) return fail("split kernel launch failed");
    if (c->variant == PYMFB_VARIANT_SNMF) {
        k_split_posneg<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>(c->st, c->G, cnt, c->Gpos, c->Gneg);
        c->launches += 1;
        CU(cudaGetLastError());
    }
    c->g_valid = true;
    return 0;
}

static int launch_update_w(pymfb_ctx* c) {
    const float* A = c->AB;
    const float* B = c->AB + c->d * c->kp;
    unsigned grid = (unsigned)((c->d + UW_ROWS - 1) / UW_ROWS);
    size_t smem = (size_t)UW_ROWS * c->kp * sizeof(float);
    if (smem > 48 * 1024 && !c->uw_smem_set) {     // k > 1536: beyond the default dynamic shared-memory limit
        CU(cudaFuncSetAttribute(k_update_w, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CU(cudaFuncSetAttribute(k_update_w_snmf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        c->uw_smem_set = true;
    }
    if (c->variant == PYMFB_VARIANT_SNMF) {      // W = A B^-1 (pymf/snmf.py:67-70); the old W is not an input
        k_inv_f64<<<1, 256, 0, c->stream>>>(c->st, B, c->kp, c->k, c->inv_work, c->Binv);
        k_update_w_snmf<<<grid, SIMT_THREADS, smem, c->stream>>>(c->st, A, c->Binv, c->W[c->wcur ^ 1], c->d, c->kp, c->k);
        c->launches += 2;
        CU(cudaGetLastError());
        c->wcur ^= 1;
        c->g_valid = false;
        return 0;
    }
    k_update_w<<<grid, SIMT_THREADS, smem, c->stream>>>(c->st, c->W[c->wcur], A, B, c->W[c->wcur ^ 1], c->d, c->kp, (float)c->lam_w);
    c->launches += 1;
    CU(cudaGetLastError());
    c->wcur ^= 1;
    c->g_valid = false;
    return 0;
}

// k block of the sparse passes: the widest of 128 / 64 / 32 / 16 that divides kp
static int sparse_kblk(int kp) { return kp % 128 == 0 ? 128 : kp % 64 == 0 ? 64 : kp % 32 == 0 ? 32 : 16; }

// Sparse H update: D = G H (G+ H, G- H for Semi-NMF), then H[hcur^1] and Ht from the CSC
static int launch_h_update_sparse(pymfb_ctx* c, bool snmf) {
    const float* Hc = c->H[c->hcur];
    dim3 gg((unsigned)((c->n_loc + TILE_N - 1) / TILE_N), (unsigned)(c->kp / c->kb));
    if (snmf) {
        if (c->kb == 16) k_gh_posneg_simt<16><<<gg, SIMT_THREADS, 0, c->stream>>>(c->st, c->Gpos, c->Gneg, Hc, c->ldh, c->n_loc, c->kp, c->Dp, c->Dn);
        else k_gh_posneg_simt<32><<<gg, SIMT_THREADS, 0, c->stream>>>(c->st, c->Gpos, c->Gneg, Hc, c->ldh, c->n_loc, c->kp, c->Dp, c->Dn);
    } else {
        if (c->kb == 16) sp::k_gh_simt<16><<<gg, SIMT_THREADS, 0, c->stream>>>(c->st, c->G, Hc, c->ldh, c->n_loc, c->kp, c->GH);
        else sp::k_gh_simt<32><<<gg, SIMT_THREADS, 0, c->stream>>>(c->st, c->G, Hc, c->ldh, c->n_loc, c->kp, c->GH);
    }
    const SparseX& s = c->sx;
    const float* D = snmf ? c->Dp : c->GH;
    const float* Dn = snmf ? c->Dn : nullptr;
    const int kblk = sparse_kblk(c->kp);
    const int tcol = (sp::SP_THREADS / (kblk / 4)) * sp::SP_COLS_PER_GROUP;
    dim3 grid((unsigned)((c->n_loc + tcol - 1) / tcol), (unsigned)(c->kp / kblk));
#define SP_HU(KBLK) sp::k_h_update_csc<KBLK><<<grid, sp::SP_THREADS, 0, c->stream>>>(c->st, s.colptr, s.rowidx, s.vals, \
        c->W[c->wcur], c->kp, Hc, c->H[c->hcur ^ 1], c->ldh, c->Ht, D, Dn, (float)c->lam_h, c->n_loc)
    if (kblk == 128) SP_HU(128);
    else if (kblk == 64) SP_HU(64);
    else if (kblk == 32) SP_HU(32);
    else SP_HU(16);
#undef SP_HU
    c->launches += 2;
    CU(cudaGetLastError());
    return 0;
}

// Sparse P = [X H^T | H H^T]: H^T (rebuilt if H was set from outside), A panel by panel, B from H^T
static int launch_xht_sparse(pymfb_ctx* c) {
    if (c->ht_of != c->hcur) {
        sp::k_h_transpose<<<grid_for(c->n_loc * c->kp, 256, 16 * c->sm_count), 256, 0, c->stream>>>(c->st, c->H[c->hcur], c->ldh, c->n_loc, c->kp, c->Ht);
        c->launches += 1;
        c->ht_of = c->hcur;
    }
    const SparseX& s = c->sx;
    const int kblk = sparse_kblk(c->kp);
    const int rows_per_cta = sp::SP_THREADS / (kblk / 4);
    dim3 grid((unsigned)((c->d + rows_per_cta - 1) / rows_per_cta), (unsigned)(c->kp / kblk));
    for (int p = 0; p < s.npanels; ++p) {
        const int64_t* rp = s.rowptr + (int64_t)p * c->d;
#define SP_XHT(KBLK) sp::k_xht_csr<KBLK><<<grid, sp::SP_THREADS, 0, c->stream>>>(c->st, rp, s.ccol, s.cval, c->Ht, c->kp, c->P, c->d, p == 0)
        if (kblk == 128) SP_XHT(128);
        else if (kblk == 64) SP_XHT(64);
        else if (kblk == 32) SP_XHT(32);
        else SP_XHT(16);
#undef SP_XHT
    }
    dim3 gh((unsigned)((c->kp + TILE_N - 1) / TILE_N), (unsigned)(c->kp / c->kb), (unsigned)c->hh_splits);
    if (c->kb == 16)
        k_ltr_partial_simt<16><<<gh, SIMT_THREADS, 0, c->stream>>>(c->st, c->Ht, c->kp, c->Ht, c->kp, c->kp, c->n_loc,
                                                                   c->hh_rows_per_split, c->hh_part, c->kp, c->kp);
    else
        k_ltr_partial_simt<32><<<gh, SIMT_THREADS, 0, c->stream>>>(c->st, c->Ht, c->kp, c->Ht, c->kp, c->kp, c->n_loc,
                                                                   c->hh_rows_per_split, c->hh_part, c->kp, c->kp);
    const int64_t cnt = (int64_t)c->kp * c->kp;
    k_sum_partials<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>(c->st, c->hh_part, c->hh_splits, cnt, c->P + c->d * c->kp);
    c->launches += s.npanels + 2;
    CU(cudaGetLastError());
    return 0;
}

// H update pass: H[hcur] -> H[hcur^1]
static int launch_h_update(pymfb_ctx* c) {
    cudaEvent_t e0, e1;
    CK(timing_begin(c, 0, &e0, &e1));
    const bool snmf = c->variant == PYMFB_VARIANT_SNMF;
    if (c->path == PYMFB_PATH_TC) {
        c->tc.lam_h = (float)c->lam_h;
        c->tc.Dp = c->tc.Dn = nullptr;
        if (snmf) {                                // G+ H and G- H of the old H for the epilogue
            dim3 grid((unsigned)((c->n_loc + TILE_N - 1) / TILE_N), (unsigned)(c->kp / c->kb));
            k_gh_posneg_simt<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->Gpos, c->Gneg, c->H[c->hcur], c->ldh,
                                                                       c->n_loc, c->kp, c->Dp, c->Dn);
            c->launches += 1;
            CU(cudaGetLastError());
            c->tc.Dp = c->Dp; c->tc.Dn = c->Dn;
        }
        if (c->tc.use_ts2) {
            if (ts2_h_update(c->tc, c->st, c->H[c->hcur], c->H[c->hcur ^ 1], c->stream, &c->launches)) return fail("CTA-pair H-update launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        } else if (c->tc.use_tc2) {
            if (tc2_h_update(c->tc, c->st, c->H[c->hcur], c->H[c->hcur ^ 1], c->stream, &c->launches)) return fail("CTA-pair SS H-update launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        } else if (tc_h_update(c->tc, c->st, c->H[c->hcur], c->H[c->hcur ^ 1], c->stream, &c->launches)) return fail("tcgen05 H-update launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    } else if (c->path == PYMFB_PATH_SPARSE) {
        CK(launch_h_update_sparse(c, snmf));
    } else {
        dim3 grid((unsigned)((c->n_loc + TILE_N - 1) / TILE_N), (unsigned)(c->kp / c->kb), (unsigned)c->hsplit);
        if (c->kb == 16)
            k_h_update_simt<16><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->W[c->wcur], snmf ? c->Gpos : c->G,
                                                                      c->H[c->hcur], c->H[c->hcur ^ 1], c->ldh,
                                                                      c->d, c->n_loc, c->kp, (float)c->lam_h, snmf ? c->Gneg : nullptr,
                                                                      c->h_rows_per_split, c->h_cpart, c->h_tickets, c->P, c->ab_count, c->xps, c->xsh);
        else
            k_h_update_simt<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->W[c->wcur], snmf ? c->Gpos : c->G,
                                                                      c->H[c->hcur], c->H[c->hcur ^ 1], c->ldh,
                                                                      c->d, c->n_loc, c->kp, (float)c->lam_h, snmf ? c->Gneg : nullptr,
                                                                      c->h_rows_per_split, c->h_cpart, c->h_tickets, c->P, c->ab_count, c->xps, c->xsh);
        c->launches += 1;
        CU(cudaGetLastError());
        c->p_zeroed = true;            // the SIMT kernel cleared P (nothing reads [A | B] between here and the next X H^T pass)
    }
    CK(timing_end(c, 0, e0, e1));
    c->hcur ^= 1;
    if (c->path == PYMFB_PATH_SPARSE) c->ht_of = c->hcur;     // the sparse H update wrote H^T of the new H
    c->ab_valid = false;
    c->lam_w *= c->inc_w;      // pymf/bnmf.py:84-85: both weights grow at the end of update_h
    c->lam_h *= c->inc_h;
    return 0;
}

// One-pass iteration body (kernels_fused.cuh): H[hcur] -> H[hcur^1], P = [X H^T | H H^T], AB = allreduce(P)
static int launch_fused(pymfb_ctx* c) {
    if (c->fused.zero_p) {         // atomics flush (no room for the ordered copies): the kernel adds into a cleared P
        k_zero<<<grid_for(c->ab_count, 256, 8 * c->sm_count), 256, 0, c->stream>>>(c->st, c->P, c->ab_count);
        c->launches += 1;
    }
    cudaEvent_t e0, e1;
    CK(timing_begin(c, 0, &e0, &e1));
    if (fused_launch(c->fused, c->tc, c->st, c->H[c->hcur], c->H[c->hcur ^ 1], c->G, c->P, c->stream, &c->launches, fault_buffer()))
        return fail("fused kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    CK(timing_end(c, 0, e0, e1));
    c->hcur ^= 1;
    if (c->world > 1)
        NC(g_nccl.AllReduce(c->P, c->P, (size_t)c->ab_count, kNcclFloat32, kNcclSum, c->comm, c->stream));
    c->ab_valid = true;
    return 0;
}

static void xht_splits(pymfb_ctx* c, int64_t rows, int64_t* cols_per_split, unsigned* nsplit) {
    const int64_t rowblocks = (rows + 127) / 128, kblocks = c->kp / c->kb;
    const int64_t chunks = (c->n_loc + XHT_CK - 1) / XHT_CK;
    int64_t want = std::max<int64_t>(1, (4LL * c->sm_count) / (rowblocks * kblocks));
    want = std::min(want, chunks);
    int64_t chunks_per = (chunks + want - 1) / want;
    *cols_per_split = chunks_per * XHT_CK;
    *nsplit = (unsigned)((chunks + chunks_per - 1) / chunks_per);
}

// P = [X H^T | H H^T] for the current H, then AB = allreduce(P)
static int launch_xht(pymfb_ctx* c) {
    const float* Hc = c->H[c->hcur];
    // deterministic combine (partial copies + ordered sum) overwrites P: nothing to clear
    const bool overwrite = (c->path == PYMFB_PATH_SPARSE) ||
                           ((c->path == PYMFB_PATH_TC) ? (c->tc.xpart != nullptr) : (c->xpart_simt != nullptr));
    if (!c->p_zeroed && !overwrite) {
        k_zero<<<grid_for(c->ab_count, 256, 8 * c->sm_count), 256, 0, c->stream>>>(c->st, c->P, c->ab_count);
        c->launches += 1;
    }
    c->p_zeroed = false;
    cudaEvent_t e0, e1;
    CK(timing_begin(c, 1, &e0, &e1));
    if (c->path == PYMFB_PATH_TC) {
        if (tc_xht(c->tc, c->st, Hc, c->P, c->stream, &c->launches)) return fail("tcgen05 X.H^T launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    } else if (c->path == PYMFB_PATH_SPARSE) {
        CK(launch_xht_sparse(c));
    } else {
        // X H^T and H H^T in ONE launch: the row blocks beyond those of X stream H itself
        int64_t cps; unsigned ns;
        xht_splits(c, c->d, &cps, &ns);
        if (!c->xpart_simt && c->deterministic_simt && ns > 1)        // ns copies of the [A | B] layout
            CU(cudaMalloc(&c->xpart_simt, (size_t)ns * c->ab_count * sizeof(float)));
        const int nrb_x = (int)((c->d + 127) / 128), nrb_h = (c->kp + 127) / 128;
        dim3 grid((unsigned)(nrb_x + nrb_h), ns, (unsigned)(c->kp / c->kb));
        float* PB = c->P + c->d * c->kp;
        if (c->kb == 16)
            k_xht_simt<16><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->d, Hc, c->ldh, c->n_loc, cps, c->P, c->kp,
                                                                 nrb_x, (int64_t)c->kp, PB, c->xpart_simt, c->ab_count, c->xps, c->xsh);
        else
            k_xht_simt<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->d, Hc, c->ldh, c->n_loc, cps, c->P, c->kp,
                                                                 nrb_x, (int64_t)c->kp, PB, c->xpart_simt, c->ab_count, c->xps, c->xsh);
        c->launches += 1;
        if (c->xpart_simt && ns > 1) {              // deterministic combine of the column splits
            tc::k_sum_copies<<<grid_for(c->ab_count / 4, 256, 4 * c->sm_count), 256, 0, c->stream>>>(
                c->st, c->xpart_simt, (int)ns, c->ab_count, c->P, nullptr, 0, 0, nullptr);
            c->launches += 1;
        }
        CU(cudaGetLastError());
    }
    CK(timing_end(c, 1, e0, e1));
    if (c->world > 1)
        NC(g_nccl.AllReduce(c->P, c->P, (size_t)c->ab_count, kNcclFloat32, kNcclSum, c->comm, c->stream));
    c->ab_valid = true;
    return 0;
}

static int launch_xx(pymfb_ctx* c) {
    if (c->sparse)        // the value array as a 1 x nnz row (zero-padded to a multiple of 4)
        k_xx<<<XX_BLOCKS, 256, 0, c->stream>>>(c->st, c->sx.vals, round_up(c->sx.nnz, 4), 1, c->sx.nnz, c->red_scratch, 0, kNoPanelShift);
    else
        k_xx<<<XX_BLOCKS, 256, 0, c->stream>>>(c->st, c->X, c->ldx, c->d, c->n_loc, c->red_scratch, c->xps, c->xsh);
    c->launches += 1;
    CU(cudaGetLastError());
    if (c->world > 1)
        NC(g_nccl.AllReduce(&c->st->xx_local, &c->st->xx, 1, kNcclFloat64, kNcclSum, c->comm, c->stream));
    c->xx_valid = true;
    return 0;
}

static int launch_err(pymfb_ctx* c, bool store, bool early_stop) {
    const float* A = c->AB;
    const float* B = c->AB + c->d * c->kp;
    if (c->err_direct) {
        const int64_t cnt = c->d * c->kp;
        k_transpose_w<<<(unsigned)((cnt + 255) / 256), 256, 0, c->stream>>>(c->st, c->W[c->wcur], c->d, c->kp, c->Wt, c->ldwt);
        dim3 grid((unsigned)((c->n_loc + TILE_N - 1) / TILE_N), (unsigned)((c->d + c->kb - 1) / c->kb));
        const SparseX& s = c->sx;
        if (c->sparse && c->kb == 16)
            sp::k_resid_csc<16><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, s.colptr, s.rowidx, s.vals, c->Wt, c->ldwt, c->H[c->hcur], c->ldh, c->d, c->n_loc, c->kp, c->resid_part);
        else if (c->sparse)
            sp::k_resid_csc<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, s.colptr, s.rowidx, s.vals, c->Wt, c->ldwt, c->H[c->hcur], c->ldh, c->d, c->n_loc, c->kp, c->resid_part);
        else if (c->kb == 16)
            k_resid_simt<16><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->Wt, c->ldwt, c->H[c->hcur], c->ldh, c->d, c->n_loc, c->kp, c->resid_part, c->xps, c->xsh);
        else
            k_resid_simt<32><<<grid, SIMT_THREADS, 0, c->stream>>>(c->st, c->X, c->ldx, c->Wt, c->ldwt, c->H[c->hcur], c->ldh, c->d, c->n_loc, c->kp, c->resid_part, c->xps, c->xsh);
        c->launches += 2;
        CU(cudaGetLastError());
        if (c->world > 1)
            NC(g_nccl.AllReduce(&c->st->resid_local, &c->st->resid, 1, kNcclFloat64, kNcclSum, c->comm, c->stream));
        k_err<<<1, 256, 0, c->stream>>>(c->st, nullptr, nullptr, 0, nullptr, nullptr, 0, c->red_scratch,
                                        store ? c->ferr_dev : nullptr, (double)c->n_glob, early_stop ? 1 : 0, 1);
    } else {
        k_err<<<ERR_BLOCKS, 256, 0, c->stream>>>(c->st, c->W[c->wcur], A, c->d * c->kp, c->G, B, (int64_t)c->kp * c->kp,
                                                 c->red_scratch, store ? c->ferr_dev : nullptr,
                                                 (double)c->n_glob, early_stop ? 1 : 0, 0);
    }
    c->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

static void graph_drop(pymfb_ctx* c);

// Direct-residual buffers (W^T and the per-block partial sums), allocated on first use.
static int ensure_direct_buffers(pymfb_ctx* c) {
    if (c->Wt) return 0;
    c->ldwt = round_up(c->d, 32);
    CU(cudaMalloc(&c->Wt, (size_t)c->kp * c->ldwt * sizeof(float)));
    CU(cudaMemsetAsync(c->Wt, 0, (size_t)c->kp * c->ldwt * sizeof(float), c->stream));
    const int64_t nb = ((c->n_loc + TILE_N - 1) / TILE_N) * ((c->d + c->kb - 1) / c->kb);
    CU(cudaMalloc(&c->resid_part, sizeof(double) * nb));
    return 0;
}

// The trace identity reported a cancelled value (DevState::cancel): from now on this context measures the error
// as the reference writes it, ||X - W H|| by a direct pass (pymf/nmf.py:110), until the data changes.
static int note_cancellation(pymfb_ctx* c, DevState& hs) {
    if (!hs.cancel) return 0;
    CU(cudaMemsetAsync(&c->st->cancel, 0, sizeof(int), c->stream));
    if (c->err_mode_opt == PYMFB_ERR_TRACE || c->err_direct) return 0;      // forced identity: the caller's choice
    CK(ensure_direct_buffers(c));
    c->err_direct = true;
    c->err_auto_switched = true;
    graph_drop(c); c->graph_key = 0;
    return 0;
}

static int check_ready(pymfb_ctx* c) {
    if (!c) return fail("null context");
    if (!c->X && !c->sparse) return fail("no data bound: call pymfb_bind_x / pymfb_upload_x / pymfb_upload_x_csc / pymfb_upload_x_sparse_device / pymfb_gen_x first");
    if (!c->w_set || !c->h_set) return fail("W and H must be set (pymfb_set_w/h or pymfb_gen_w/h) before running");
    return 0;
}

// One iteration of the factorize() loop (pymf/nmf.py:182-190): W update, H update, error.
// more_after: another iteration follows (its W update needs A, B of the new H).
static int enqueue_one(pymfb_ctx* c, bool do_w, bool do_h, bool do_e, bool trace, bool early, bool more_after) {
    if (do_w) {
        if (!c->ab_valid) CK(launch_xht(c));      // bootstrap: A, B of the current H
        CK(launch_update_w(c));
    }
    if (do_h) {
        if (!c->g_valid) CK(launch_gram_w(c));
        // A, B of the new H feed the next W update and this iteration's error
        const bool need_ab = trace || (do_w && more_after);
        if (need_ab && c->path == PYMFB_PATH_TC && c->fused.ready && c->lam_h == 0.0 && c->variant == PYMFB_VARIANT_NMF) {
            CK(launch_fused(c));
        } else {
            CK(launch_h_update(c));
            if (need_ab) CK(launch_xht(c));
        }
    }
    if (do_e) {
        if (trace && !c->g_valid) CK(launch_gram_w(c));
        if (trace && !c->ab_valid) CK(launch_xht(c));
        CK(launch_err(c, true, early));
    }
    return 0;
}

static LoopState loop_state(const pymfb_ctx* c) {
    return LoopState{c->wcur, c->hcur, c->ab_valid, c->g_valid, c->xx_valid, c->tc.hs_valid[0], c->tc.hs_valid[1], c->ht_of};
}

static void graph_drop(pymfb_ctx* c) {
    if (c->graph_exec) { cudaGraphExecDestroy(c->graph_exec); c->graph_exec = nullptr; }
}

// Launch-bound problems (an iteration is ~10 kernels of a few microseconds each: cfg1 1000 x 500 ran 108 us per
// iteration, almost all of it launch gaps) replay TWO iterations - one full ping-pong period of the W / H buffers -
// as one CUDA graph.  Eligible: plain NMF (the BNMF weight changes every iteration), no per-kernel timing, small X;
// any number of ranks - the in-place ncclAllReduce of [X H^T | H H^T] is captured with the kernels (every rank
// replays the same sequence of collectives; the plain warm-up iterations before the capture have already set up
// NCCL's connections).  The graph is captured from the steady state (after two plain iterations) and cached.
static bool graph_eligible(const pymfb_ctx* c, int niter) {
    if (c->graph_opt == PYMFB_GRAPH_OFF) return false;
    if (c->timing || c->lam_w != 0.0 || c->lam_h != 0.0 || niter < 5) return false;
    if (c->path == PYMFB_PATH_TC && c->fused.ready) return false;
    if (c->graph_opt == PYMFB_GRAPH_ON) return true;
    return (double)c->d * (double)c->n_loc <= 16777216.0;
}

static int graph_build(pymfb_ctx* c, unsigned key, bool do_w, bool do_h, bool do_e, bool trace, bool early) {
    graph_drop(c);
    const LoopState s0 = loop_state(c);
    const int64_t l0 = c->launches;
    cudaGraph_t g = nullptr;
    CU(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue_one(c, do_w, do_h, do_e, trace, early, true);
    if (!rc) rc = enqueue_one(c, do_w, do_h, do_e, trace, early, true);
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    const int64_t per = c->launches - l0;
    c->launches = l0;                              // nothing ran yet
    const bool periodic = loop_state(c) == s0;
    // capture only recorded the launches: put the scheduling state back to where the stream really is
    c->wcur = s0.wcur; c->hcur = s0.hcur; c->ab_valid = s0.ab; c->g_valid = s0.g; c->xx_valid = s0.xx;
    c->tc.hs_valid[0] = s0.hs0; c->tc.hs_valid[1] = s0.hs1; c->ht_of = s0.ht;
    if (rc || e != cudaSuccess || !g || !periodic) {
        if (g) cudaGraphDestroy(g);
        cudaGetLastError();
        c->graph_key = 0xFFFFFFFFu;                // do not retry for this flag set / state
        c->graph_state = s0;
        return 0;                                  // not an error: the caller falls back to plain launches
    }
    e = cudaGraphInstantiate(&c->graph_exec, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) { c->graph_exec = nullptr; cudaGetLastError(); return 0; }
    c->graph_key = key; c->graph_state = s0; c->graph_launches = per;
    return 0;
}

static int enqueue_iterations(pymfb_ctx* c, int niter, unsigned flags) {
    CK(check_ready(c));
    CU(cudaSetDevice(c->device));
    const bool do_w = flags & PYMFB_COMPUTE_W, do_h = flags & PYMFB_COMPUTE_H, do_e = flags & PYMFB_COMPUTE_ERR;
    const bool early = (flags & PYMFB_EARLY_STOP) && do_e;
    const bool trace = do_e && !c->err_direct;   // the trace identity needs ||X||^2, A, B, G
    if (do_e) CU(cudaMemsetAsync(&c->st->it, 0, sizeof(int), c->stream));
    if (trace && !c->xx_valid) CK(launch_xx(c));
    int i = 0;
    if (graph_eligible(c, niter)) {
        for (; i < 2; ++i) CK(enqueue_one(c, do_w, do_h, do_e, trace, early, true));   // reach the steady state (both ping-pong halves)
        const unsigned key = (do_w ? 1u : 0u) | (do_h ? 2u : 0u) | (do_e ? 4u : 0u) | (early ? 8u : 0u) | (trace ? 16u : 0u);
        if (!(c->graph_exec && c->graph_key == key && c->graph_state == loop_state(c)) &&
            !(c->graph_key == 0xFFFFFFFFu && c->graph_state == loop_state(c)))
            CK(graph_build(c, key, do_w, do_h, do_e, trace, early));
        if (c->graph_exec && c->graph_key == key && c->graph_state == loop_state(c)) {
            for (; i + 2 < niter; i += 2) {        // the last iteration stays outside (more_after = false)
                CU(cudaGraphLaunch(c->graph_exec, c->stream));
                c->launches += c->graph_launches;
                c->graph_replays += 1;
            }
        }
    }
    for (; i < niter; ++i) CK(enqueue_one(c, do_w, do_h, do_e, trace, early, i + 1 < niter));
    return 0;
}

// stage (rows x cols of T, leading dimension lds) -> X_own rows [r0, r0 + rows), columns [dcol0, dcol0 + cols)
template <typename T>
static void launch_place_x(pymfb_ctx* c, const T* stage, int64_t lds, int64_t r0, int64_t rows, int64_t cols, int64_t dcol0) {
    dim3 grid((unsigned)((cols + 1023) / 1024), (unsigned)std::min<int64_t>(rows, 4096));
    k_place_x<T><<<grid, 256, 0, c->stream>>>(stage, lds, c->X_own + r0 * c->ldx, c->ldx, rows, cols, dcol0, c->xps, c->xsh);
    c->launches += 1;
}

static int p_unregister(pymfb_ctx* c) {
    if (c->p_reg && c->comm && g_nccl.CommDeregister) g_nccl.CommDeregister(c->comm, c->p_reg);
    c->p_reg = nullptr;
    return 0;
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

int pymfb_version(void) { return 1002; }
const char* pymfb_last_error(void) { return g_err; }

int pymfb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int pymfb_create(pymfb_ctx** out, int device, int64_t d, int64_t n_local, int64_t n_global, int64_t col0, int k) {
    if (!out) return fail("out is null");
    *out = nullptr;
    if (d <= 0 || n_local <= 0 || k <= 0 || n_global < n_local) return fail("bad shape d=%lld n_local=%lld n_global=%lld k=%d", (long long)d, (long long)n_local, (long long)n_global, k);
    int ndev = pymfb_device_count();
    if (ndev <= 0) return fail("no CUDA device available: libpymfb has no CPU fallback");
    if (device < 0 || device >= ndev) return fail("device %d out of range (have %d)", device, ndev);
    CU(cudaSetDevice(device));
    // single attributes, not cudaGetDeviceProperties (which queries everything and costs milliseconds per call)
    int cc_major = 0, cc_minor = 0, sm_count = 0;
    CU(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    CU(cudaDeviceGetAttribute(&cc_minor, cudaDevAttrComputeCapabilityMinor, device));
    CU(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    if (cc_major != 10) return fail("device %d is sm_%d%d; libpymfb is built for sm_100a (B200) only", device, cc_major, cc_minor);
    {   // the W-update kernels stage UW_ROWS rows of A (UW_ROWS x kp fp32) in dynamic shared memory
        const int64_t kp_max = (int64_t)(227 * 1024) / (UW_ROWS * (int64_t)sizeof(float)) / 32 * 32;
        if ((int64_t)k > kp_max) return fail("k = %d is beyond the supported bound (k <= %lld: one row block of the W update must fit shared memory)", k, (long long)kp_max);
    }
    pymfb_ctx* c = new pymfb_ctx();
    c->device = device; c->d = d; c->n_loc = n_local; c->n_glob = n_global; c->col0 = col0; c->k = k;
    // k is zero-padded to kp (exact: padded rows / columns of W and H stay 0 under the updates).  Small k on a
    // small problem keeps the 16-wide SIMT kernels; on a streaming-sized problem it is padded to 32 so that the
    // tcgen05 path (kp % 32 == 0) serves it: 8192 x 524288, k = 16 ran 15.2 ms / iteration on SIMT vs 6.1 ms padded.
    const bool streaming_size = (double)d * (double)n_local >= 16777216.0 && d >= 64 && n_local >= 128;
    c->kp = (int)((k <= 16 && !streaming_size) ? 16 : round_up(k, 32));
    // 128 < k <= 512 on a streaming-sized problem: blocks of 128 bases on the tensor path (kernels_tc.cuh)
    if (k > 128 && k <= 512 && streaming_size) c->kp = (int)round_up(k, 128);
    c->kb = std::min(c->kp, 32);
    c->sm_count = sm_count;
    { const char* e = getenv("PYMFB_DETERMINISTIC"); c->deterministic_simt = !(e && e[0] == '0'); }
    c->ldh = padded_ld(n_local);
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    const size_t wbytes = (size_t)d * c->kp * sizeof(float), hbytes = (size_t)c->kp * c->ldh * sizeof(float);
    for (int i = 0; i < 2; ++i) {
        CU(cudaMalloc(&c->W[i], wbytes)); CU(cudaMemsetAsync(c->W[i], 0, wbytes, c->stream));
        CU(cudaMalloc(&c->H[i], hbytes)); CU(cudaMemsetAsync(c->H[i], 0, hbytes, c->stream));
    }
    c->ab_count = d * c->kp + (int64_t)c->kp * c->kp;
    CU(cudaMalloc(&c->P, c->ab_count * sizeof(float)));
    CU(cudaMemsetAsync(c->P, 0, c->ab_count * sizeof(float), c->stream));
    c->AB = c->P;   // reduced in place (comm_bind may move it into NCCL-registered memory)
    CU(cudaMalloc(&c->G, (size_t)c->kp * c->kp * sizeof(float)));
    // row splits of the W^T W reduction: enough CTAs to cover the SMs, >= 64 rows each
    {
        int64_t tiles = ((c->kp + TILE_N - 1) / TILE_N) * (c->kp / c->kb);
        int64_t want = std::max<int64_t>(1, (2LL * c->sm_count) / tiles);
        int64_t max_by_rows = std::max<int64_t>(1, d / 64);
        c->g_splits = (int)std::min(want, max_by_rows);
        c->g_rows_per_split = round_up((d + c->g_splits - 1) / c->g_splits, TILE_DK);
        c->g_splits = (int)((d + c->g_rows_per_split - 1) / c->g_rows_per_split);
    }
    CU(cudaMalloc(&c->Gpart, (size_t)c->g_splits * c->kp * c->kp * sizeof(float)));
    CU(cudaMalloc(&c->red_scratch, sizeof(double) * std::max(2 * ERR_BLOCKS, XX_BLOCKS)));
    // error mode (see k_resid_simt): direct residual while the extra pass is cheap
    c->err_direct = (double)d * (double)n_local * (double)c->kp <= kDirectErrMaxWork;
    if (c->err_direct) {
        c->ldwt = round_up(d, 32);
        CU(cudaMalloc(&c->Wt, (size_t)c->kp * c->ldwt * sizeof(float)));
        CU(cudaMemsetAsync(c->Wt, 0, (size_t)c->kp * c->ldwt * sizeof(float), c->stream));
        const int64_t nb = ((n_local + TILE_N - 1) / TILE_N) * ((d + c->kb - 1) / c->kb);
        CU(cudaMalloc(&c->resid_part, sizeof(double) * nb));
    }
    {   // SIMT H-update: enough CTAs to cover the SMs, >= 64 rows of X per split
        const int64_t tiles = ((n_local + TILE_N - 1) / TILE_N) * (c->kp / c->kb);
        int64_t want = std::max<int64_t>(1, (2LL * c->sm_count) / tiles);
        want = std::min<int64_t>(want, std::max<int64_t>(1, d / 64));
        c->h_rows_per_split = round_up((d + want - 1) / want, TILE_DK);
        c->hsplit = (int)((d + c->h_rows_per_split - 1) / c->h_rows_per_split);
        if (c->hsplit > 1) {
            CU(cudaMalloc(&c->h_cpart, (size_t)tiles * c->hsplit * c->kb * TILE_N * sizeof(float)));
            CU(cudaMalloc(&c->h_tickets, (size_t)tiles * sizeof(unsigned)));
            CU(cudaMemsetAsync(c->h_tickets, 0, (size_t)tiles * sizeof(unsigned), c->stream));
        }
    }
    CU(cudaMalloc(&c->st, sizeof(DevState)));
    CU(cudaMemsetAsync(c->st, 0, sizeof(DevState), c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *out = c;
    return 0;
}

int pymfb_destroy(pymfb_ctx* c) {
    if (!c) return 0;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    graph_drop(c);
    p_unregister(c);
    if (c->comm && c->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    tc_release(c->tc);
    fused_release(c->fused);
    sparse_free(c->sx); cudaFree(c->Ht); cudaFree(c->GH); cudaFree(c->hh_part);
    for (int w = 0; w < 2; ++w)
        for (auto& p : c->ev[w]) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
    if (c->p_nccl && g_nccl.MemFree) g_nccl.MemFree(c->P); else cudaFree(c->P);
    cudaFree(c->G); cudaFree(c->Gpart); cudaFree(c->red_scratch); cudaFree(c->st);
    cudaFree(c->h_cpart); cudaFree(c->h_tickets); cudaFree(c->xpart_simt);
    cudaFree(c->Gpos); cudaFree(c->Gneg); cudaFree(c->Dp); cudaFree(c->Dn); cudaFree(c->inv_work); cudaFree(c->Binv);
    for (int s_ = 0; s_ < 2; ++s_) { if (c->panel_ev[s_]) cudaEventDestroy(c->panel_ev[s_]); cudaFree(c->panel_stage[s_]); }
    cudaFree(c->stage); cudaFree(c->ferr_dev); cudaFree(c->flush_buf); cudaFree(c->X_own); cudaFree(c->Wt); cudaFree(c->resid_part);
    for (int i = 0; i < 2; ++i) { cudaFree(c->W[i]); cudaFree(c->H[i]); }
    cudaStreamDestroy(c->stream);
    delete c;
    return 0;
}

int pymfb_set_option(pymfb_ctx* c, int option, int64_t value) {
    if (!c) return fail("null context");
    graph_drop(c); c->graph_key = 0;          // every option changes which kernels an iteration launches
    if (option == PYMFB_OPT_GRAPH) {
        if (value < 0 || value > 2) return fail("bad graph option %lld", (long long)value);
        c->graph_opt = (int)value;
        return 0;
    }
    if (option == PYMFB_OPT_PATH) {
        if (value < 0 || value > 2) return fail("bad path option %lld", (long long)value);
        if (c->sparse && value != PYMFB_PATH_AUTO)
            return fail("sparse data runs on its own passes: the dense kernel families (path simt / tc) do not apply");
        c->path_opt = (int)value;
        if (c->X) { CK(resolve_path(c)); if (c->path == PYMFB_PATH_TC) CK(plan_tc(c)); c->g_valid = false; }
        return 0;
    }
    if (option == PYMFB_OPT_NNDSVD_PATH) {
        if (value < 0 || value > 2) return fail("bad NNDSVD path option %lld", (long long)value);
        c->nndsvd_path_opt = (int)value;
        return 0;
    }
    if (option == PYMFB_OPT_ERR_MODE) {
        if (value < 0 || value > 2) return fail("bad error mode %lld", (long long)value);
        CU(cudaSetDevice(c->device));
        bool direct = value == PYMFB_ERR_DIRECT ||
                      (value == PYMFB_ERR_AUTO && (double)c->d * (double)c->n_loc * (double)c->kp <= kDirectErrMaxWork);
        if (direct) CK(ensure_direct_buffers(c));
        c->err_direct = direct;
        c->err_mode_opt = (int)value;
        c->err_auto_switched = false;
        return 0;
    }
    return fail("unknown option %d", option);
}

int pymfb_set_penalty(pymfb_ctx* c, double lamb_w, double lamb_h, double increase_w, double increase_h) {
    if (!c) return fail("null context");
    if (!(lamb_w >= 0.0) || !(lamb_h >= 0.0) || !(increase_w > 0.0) || !(increase_h > 0.0))
        return fail("bad penalty lamb_w=%g lamb_h=%g increase_w=%g increase_h=%g", lamb_w, lamb_h, increase_w, increase_h);
    c->lam_w = lamb_w; c->lam_h = lamb_h; c->inc_w = increase_w; c->inc_h = increase_h;
    return 0;
}
int pymfb_set_variant(pymfb_ctx* c, int variant) {
    if (!c) return fail("null context");
    if (variant != PYMFB_VARIANT_NMF && variant != PYMFB_VARIANT_SNMF) return fail("unknown variant %d", variant);
    CU(cudaSetDevice(c->device));
    graph_drop(c); c->graph_key = 0;
    if (variant == PYMFB_VARIANT_SNMF) {
        if (c->k > 512) return fail("Semi-NMF supports k <= 512 (the k x k inverse runs in one CTA); got k = %d", c->k);
        if (!c->Gpos) {
            const size_t gb = (size_t)c->kp * c->kp * sizeof(float), hb = (size_t)c->kp * c->ldh * sizeof(float);
            CU(cudaMalloc(&c->Gpos, gb)); CU(cudaMalloc(&c->Gneg, gb));
            CU(cudaMalloc(&c->Dp, hb)); CU(cudaMalloc(&c->Dn, hb));
            CU(cudaMemsetAsync(c->Dp, 0, hb, c->stream)); CU(cudaMemsetAsync(c->Dn, 0, hb, c->stream));
            CU(cudaMalloc(&c->inv_work, sizeof(double) * 2 * c->k * c->k));
            CU(cudaMalloc(&c->Binv, sizeof(double) * c->k * c->k));
        }
    }
    if (variant != c->variant) c->g_valid = false;   // G+ / G- follow the Gram kernel
    c->variant = variant;
    return 0;
}

int pymfb_get_penalty(pymfb_ctx* c, double* lamb_w, double* lamb_h) {
    if (!c) return fail("null context");
    if (lamb_w) *lamb_w = c->lam_w;
    if (lamb_h) *lamb_h = c->lam_h;
    return 0;
}

int pymfb_comm_unique_id(void* out128) {
    CK(nccl_load());
    NC(g_nccl.GetUniqueId(out128));
    return 0;
}

static int comm_bind(pymfb_ctx* c, void* comm, bool owned, int world, int rank) {
    CK(p_unregister(c));                      // from the previous communicator, while it still exists
    if (c->comm && c->comm_owned && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    c->comm = comm; c->comm_owned = owned;
    c->world = world; c->rank = rank;
    // [X H^T | H H^T] lives in ONE buffer that the pass epilogues write and ncclAllReduce reduces in place.  With
    // a registration-capable NCCL the buffer comes from ncclMemAlloc and is registered with the communicator
    // (PYMFB_NCCL_REG=0 keeps the plain cudaMalloc buffer).
    const char* e = getenv("PYMFB_NCCL_REG");
    const bool want_reg = !(e && e[0] == '0') && g_nccl.MemAlloc && g_nccl.MemFree && g_nccl.CommRegister && g_nccl.CommDeregister;
    if (want_reg) {
        void* np = nullptr;
        if (!c->p_nccl && g_nccl.MemAlloc(&np, c->ab_count * sizeof(float)) == 0 && np) {
            CU(cudaStreamSynchronize(c->stream));
            CU(cudaFree(c->P));
            c->P = c->AB = (float*)np;
            c->p_nccl = true;
            CU(cudaMemset(c->P, 0, c->ab_count * sizeof(float)));
        }
        if (c->p_nccl && g_nccl.CommRegister(comm, c->P, c->ab_count * sizeof(float), &c->p_reg) != 0) c->p_reg = nullptr;
    }
    c->p_zeroed = false;
    graph_drop(c); c->graph_key = 0;
    c->ab_valid = false; c->xx_valid = false;
    return 0;
}

int pymfb_comm_init(pymfb_ctx* c, const void* uid128, int world, int rank) {
    if (!c) return fail("null context");
    if (world < 1 || rank < 0 || rank >= world) return fail("bad world/rank %d/%d", world, rank);
    if (world == 1) return 0;
    CK(nccl_load());
    CU(cudaSetDevice(c->device));
    Uid128 uid;
    memcpy(&uid, uid128, sizeof(uid));
    void* comm = nullptr;
    NC(g_nccl.CommInitRank(&comm, world, uid, rank));
    return comm_bind(c, comm, true, world, rank);
}

int pymfb_comm_create(void** comm_out, int device, const void* uid128, int world, int rank) {
    if (!comm_out) return fail("comm_out is null");
    *comm_out = nullptr;
    if (world < 2 || rank < 0 || rank >= world) return fail("bad world/rank %d/%d", world, rank);
    CK(nccl_load());
    CU(cudaSetDevice(device));
    Uid128 uid;
    memcpy(&uid, uid128, sizeof(uid));
    NC(g_nccl.CommInitRank(comm_out, world, uid, rank));
    return 0;
}

int pymfb_comm_attach(pymfb_ctx* c, void* comm, int world, int rank) {
    if (!c) return fail("null context");
    if (!comm) return fail("comm is null");
    if (world < 2 || rank < 0 || rank >= world) return fail("bad world/rank %d/%d", world, rank);
    CU(cudaSetDevice(c->device));
    return comm_bind(c, comm, false, world, rank);
}

int pymfb_comm_destroy(void* comm) {
    if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
    return 0;
}

// A dense upload, bind or generator call makes the dense X current again: the sparse buffers go.
static void sparse_drop(pymfb_ctx* c) {
    if (!c->sparse) return;
    cudaStreamSynchronize(c->stream);
    sparse_free(c->sx);
    cudaFree(c->Ht); cudaFree(c->GH); cudaFree(c->hh_part);
    c->Ht = c->GH = c->hh_part = nullptr;
    c->ht_of = -1;
    c->sparse = false;
}

static int data_changed(pymfb_ctx* c) {
    graph_drop(c); c->graph_key = 0;
    if (c->err_auto_switched) { c->err_direct = false; c->err_auto_switched = false; }   // new data: try the identity again
    c->p_zeroed = false;
    c->ab_valid = false; c->xx_valid = false;
    CK(resolve_path(c));
    if (c->path == PYMFB_PATH_TC) CK(plan_tc(c));
    c->g_valid = false;
    return 0;
}

// Context-owned copy of X.  Streaming-sized matrices on tensor-path shapes are stored panel-major (common.cuh): column
// panels of 128 columns, each a dense d x 128 block.  A column tile of the H-update pass is then ONE contiguous
// d x 512 B region, and the 128-row boxes of the X H^T pass sit 512 B apart instead of a whole row (4 MB at
// n = 2^20: 128 pages of 2 MB per box).  Same-box A/B against row-major (ms per iteration): cfg3 53.5 -> 50.4,
// cfg4 k=64 8.44 -> 7.83, cfg5 33.7 -> 31.4, cfg2 1.443 -> 1.405; wider panels (512 .. 16384 columns) gave less.
// PYMFB_XPANEL=0 keeps everything row-major, =<log2 width> picks another width.
static int ensure_own_x(pymfb_ctx* c) {
    sparse_drop(c);
    if (!c->X_own) {
        int sh = 7;
        bool want = (double)c->d * (double)c->n_loc >= 16777216.0 && c->d >= 64 && c->n_loc >= 128 && c->kp % 32 == 0 && c->kp <= 512;
        if (const char* e = getenv("PYMFB_XPANEL")) {     // 0: never; 7..20: panels of 2^v columns whatever n is (tests)
            const int v = atoi(e);
            if (v <= 0) want = false;
            else if (v >= 7 && v <= 20) { sh = v; want = c->d >= 64 && c->n_loc >= 128 && c->kp % 32 == 0 && c->kp <= 512; }
        }
        if (want) {
            const int64_t pw = (int64_t)1 << sh, npan = (c->n_loc + pw - 1) / pw;
            c->own_ldx = pw; c->own_xps = c->d * pw; c->own_xsh = sh;
            c->own_bytes = (size_t)npan * c->d * pw * sizeof(float);
        } else {
            c->own_ldx = padded_ld(c->n_loc); c->own_xps = 0; c->own_xsh = kNoPanelShift;
            c->own_bytes = (size_t)c->d * c->own_ldx * sizeof(float);
        }
        CU(cudaMalloc(&c->X_own, c->own_bytes));
        CU(cudaMemsetAsync(c->X_own, 0, c->own_bytes, c->stream));
    }
    c->ldx = c->own_ldx; c->xps = c->own_xps; c->xsh = c->own_xsh;
    c->X = c->X_own;
    return 0;
}

int pymfb_bind_x(pymfb_ctx* c, const float* x_dev, int64_t ld) {
    if (!c) return fail("null context");
    if (!x_dev) return fail("x_dev is null");
    if (ld < c->n_loc || (ld % 4) != 0) return fail("leading dimension %lld must be >= n_local and a multiple of 4", (long long)ld);
    if (((uintptr_t)x_dev & 15) != 0) return fail("x_dev must be 16-byte aligned");
    CU(cudaSetDevice(c->device));
    sparse_drop(c);
    c->X = x_dev; c->ldx = ld; c->xps = 0; c->xsh = kNoPanelShift;
    return data_changed(c);
}

// Pageable -> pinned copy of the staging ring.  The destination is written once and then only read by the DMA
// engine, so it is stored with NON-TEMPORAL stores: a plain memcpy first reads every destination line into the
// cache (read-for-ownership), i.e. 3 bytes of memory traffic per byte copied instead of 2 (measured with 8 threads
// on the build box: 25.9 -> 34.7 GB/s).
__attribute__((target("avx2"))) static void stream_copy_avx2(char* dst, const char* src, size_t n) {
    size_t head = (32 - ((uintptr_t)dst & 31)) & 31;
    if (head > n) head = n;
    if (head) { memcpy(dst, src, head); dst += head; src += head; n -= head; }
    const size_t v = n / 32;
    const __m256i* s = (const __m256i*)src;
    __m256i* d = (__m256i*)dst;
    size_t i = 0;
    for (; i + 4 <= v; i += 4) {
        const __m256i a = _mm256_loadu_si256(s + i), b = _mm256_loadu_si256(s + i + 1);
        const __m256i c = _mm256_loadu_si256(s + i + 2), e = _mm256_loadu_si256(s + i + 3);
        _mm256_stream_si256(d + i, a); _mm256_stream_si256(d + i + 1, b);
        _mm256_stream_si256(d + i + 2, c); _mm256_stream_si256(d + i + 3, e);
    }
    for (; i < v; ++i) _mm256_stream_si256(d + i, _mm256_loadu_si256(s + i));
    _mm_sfence();
    if (n - v * 32) memcpy(dst + v * 32, src + v * 32, n - v * 32);
}
static void stream_copy(void* dst, const void* src, size_t n) {
    static const bool avx2 = __builtin_cpu_supports("avx2") && getenv("PYMFB_NO_NT_COPY") == nullptr;
    if (avx2 && n >= 4096) stream_copy_avx2((char*)dst, (const char*)src, n);
    else memcpy(dst, src, n);
}

// Host -> device ingest of X (SURVEY 8f rank 2): a ring of pinned staging buffers is filled by a
// few host threads (pageable user memory -> pinned) while the previous chunk's H2D copy (and the
// fp64 -> fp32 cast kernel) run on the context's stream.
// The pinned staging ring is kept by the PROCESS between uploads (3 x 64 MiB): allocating and page-locking it costs
// ~50 ms, which on a 4 GiB upload was a fifth of the whole ingest.  One upload at a time uses it; a concurrent
// second upload (another context on another thread) allocates its own.
static std::mutex g_ring_mu;
static void* g_ring[3] = {nullptr, nullptr, nullptr};
static size_t g_ring_bytes = 0;
static bool g_ring_busy = false;

static int staged_upload(pymfb_ctx* c, const void* host, int dtype, int64_t ld) {
    const size_t esz = dtype == PYMFB_F32 ? 4 : 8;
    const int64_t row_bytes = c->n_loc * (int64_t)esz;
    const int NB = 3;
    int64_t rows_per = std::max<int64_t>(1, (64LL << 20) / row_bytes);
    rows_per = std::min(rows_per, c->d);
    const size_t buf_bytes = (size_t)rows_per * row_bytes;
    void* pinned[NB] = {nullptr, nullptr, nullptr};
    void* dstage[NB] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev[NB] = {nullptr, nullptr, nullptr};
    int rc = 0;
    bool own_ring = false;                      // this call took the process ring (give it back, do not free it)
    auto cleanup = [&]() {
        cudaStreamSynchronize(c->stream);
        for (int b = 0; b < NB; ++b) {
            if (pinned[b] && !own_ring) pymfb_host_free(pinned[b]);
            if (dstage[b]) cudaFree(dstage[b]);
            if (ev[b]) cudaEventDestroy(ev[b]);
        }
        if (own_ring) { std::lock_guard<std::mutex> lk(g_ring_mu); g_ring_busy = false; }
    };
#define UP(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    {
        std::lock_guard<std::mutex> lk(g_ring_mu);
        if (!g_ring_busy) {
            if (g_ring_bytes < buf_bytes) {
                for (int b = 0; b < NB; ++b) { if (g_ring[b]) pymfb_host_free(g_ring[b]); g_ring[b] = nullptr; }
                g_ring_bytes = 0;
                bool ok = true;
                for (int b = 0; b < NB && ok; ++b) ok = pymfb_host_alloc(&g_ring[b], buf_bytes) == 0;
                if (ok) g_ring_bytes = buf_bytes;
                else for (int b = 0; b < NB; ++b) { if (g_ring[b]) pymfb_host_free(g_ring[b]); g_ring[b] = nullptr; }
            }
            if (g_ring_bytes >= buf_bytes) {
                for (int b = 0; b < NB; ++b) pinned[b] = g_ring[b];
                g_ring_busy = true;
                own_ring = true;
            }
        }
    }
    for (int b = 0; b < NB; ++b) {
        if (!own_ring && pymfb_host_alloc(&pinned[b], buf_bytes)) { cleanup(); return 1; }
        if (dtype == PYMFB_F64 || c->xps != 0) UP(cudaMalloc(&dstage[b], buf_bytes));   // cast and / or panel scatter on the device
        UP(cudaEventCreateWithFlags(&ev[b], cudaEventDisableTiming));
    }
    // copy threads: the pageable -> pinned copy is the slow leg (DMA: 50 GB/s).  Up to 16, but the host's cores are
    // shared by the ranks of this box (torchrun exports LOCAL_WORLD_SIZE): 8 ranks x 16 threads on 32 cores measured
    // 0.48 of the pinned e2e rate.
    unsigned hw = std::thread::hardware_concurrency();
    unsigned local_ranks = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) local_ranks = (unsigned)std::max(1, atoi(e));
    else if (c->world > 1) local_ranks = (unsigned)c->world;
    const int nthr = (int)std::max(2u, std::min(16u, (hw ? hw : 1u) / local_ranks));
    int64_t chunk = 0;
    for (int64_t r0 = 0; r0 < c->d; r0 += rows_per, ++chunk) {
        const int b = (int)(chunk % NB);
        const int64_t nr = std::min(rows_per, c->d - r0);
        if (chunk >= NB) UP(cudaEventSynchronize(ev[b]));
        {   // pageable -> pinned, rows split over threads
            std::vector<std::thread> th;
            const int64_t per = (nr + nthr - 1) / nthr;
            for (int t = 0; t < nthr; ++t) {
                const int64_t a = t * per, e = std::min(nr, a + per);
                if (a >= e) break;
                th.emplace_back([=]() {
                    const char* src = (const char*)host + (size_t)(r0 + a) * ld * esz;
                    char* dst = (char*)pinned[b] + (size_t)a * row_bytes;
                    if (ld == c->n_loc) stream_copy(dst, src, (size_t)(e - a) * row_bytes);
                    else for (int64_t r = a; r < e; ++r, src += (size_t)ld * esz, dst += row_bytes) stream_copy(dst, src, row_bytes);
                });
            }
            for (auto& t : th) t.join();
        }
        if (dtype == PYMFB_F32 && c->xps == 0) {
            UP(cudaMemcpy2DAsync(c->X_own + r0 * c->ldx, c->ldx * sizeof(float), pinned[b], row_bytes, row_bytes, nr,
                                 cudaMemcpyHostToDevice, c->stream));
        } else {
            UP(cudaMemcpyAsync(dstage[b], pinned[b], (size_t)nr * row_bytes, cudaMemcpyHostToDevice, c->stream));
            if (dtype == PYMFB_F32) launch_place_x<float>(c, (const float*)dstage[b], c->n_loc, r0, nr, c->n_loc, 0);
            else launch_place_x<double>(c, (const double*)dstage[b], c->n_loc, r0, nr, c->n_loc, 0);
            UP(cudaGetLastError());
        }
        UP(cudaEventRecord(ev[b], c->stream));
    }
#undef UP
    cleanup();
    return 0;
}

// True when `p` is page-locked host memory the DMA engines can read directly (cudaHostAlloc,
// cudaHostRegister, pymfb_host_alloc, torch pin_memory).
static bool host_is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

// Page-locked source: no host-side copy at all.  fp32 goes straight into X with one strided DMA;
// fp64 is DMA'd in row chunks into two device staging buffers and cast to fp32 by k_cast_in while
// the next chunk is in flight.
static int pinned_upload(pymfb_ctx* c, const void* host, int dtype, int64_t ld) {
    if (dtype == PYMFB_F32 && c->xps == 0) {
        if (ld == c->n_loc && c->ldx == c->n_loc)
            CU(cudaMemcpyAsync(c->X_own, host, (size_t)c->d * c->n_loc * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        else
            CU(cudaMemcpy2DAsync(c->X_own, c->ldx * sizeof(float), host, (size_t)ld * sizeof(float),
                                 (size_t)c->n_loc * sizeof(float), (size_t)c->d, cudaMemcpyHostToDevice, c->stream));
        return 0;
    }
    // fp64 (cast) and / or panel-major X (scatter): whole rows travel by DMA into a device staging pair - long
    // contiguous transfers whatever the device layout is - and one kernel casts / places them
    const int NB = 2;
    const size_t esz = dtype == PYMFB_F32 ? 4 : 8;
    const int64_t row_bytes = c->n_loc * (int64_t)esz;
    int64_t rows_per = std::min<int64_t>(c->d, std::max<int64_t>(1, (64LL << 20) / row_bytes));
    void* dstage[NB] = {nullptr, nullptr};
    cudaEvent_t cast_done[NB] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t copied = nullptr;
    int rc = 0;
    auto cleanup = [&]() {
        cudaStreamSynchronize(c->stream);
        if (copy_stream) { cudaStreamSynchronize(copy_stream); cudaStreamDestroy(copy_stream); }
        for (int b = 0; b < NB; ++b) { if (dstage[b]) cudaFree(dstage[b]); if (cast_done[b]) cudaEventDestroy(cast_done[b]); }
        if (copied) cudaEventDestroy(copied);
    };
#define UP(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    UP(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    UP(cudaEventCreateWithFlags(&copied, cudaEventDisableTiming));
    for (int b = 0; b < NB; ++b) {
        UP(cudaMalloc(&dstage[b], (size_t)rows_per * row_bytes));
        UP(cudaEventCreateWithFlags(&cast_done[b], cudaEventDisableTiming));
    }
    // X_own was zeroed on c->stream by ensure_own_x; the casts run on c->stream, so order holds.
    int64_t chunk = 0;
    for (int64_t r0 = 0; r0 < c->d; r0 += rows_per, ++chunk) {
        const int b = (int)(chunk % NB);
        const int64_t nr = std::min(rows_per, c->d - r0);
        if (chunk >= NB) UP(cudaStreamWaitEvent(copy_stream, cast_done[b], 0));   // staging buffer free again
        UP(cudaMemcpy2DAsync(dstage[b], (size_t)row_bytes, (const char*)host + (size_t)r0 * ld * esz, (size_t)ld * esz,
                             (size_t)row_bytes, (size_t)nr, cudaMemcpyHostToDevice, copy_stream));
        UP(cudaEventRecord(copied, copy_stream));
        UP(cudaStreamWaitEvent(c->stream, copied, 0));
        if (dtype == PYMFB_F32) launch_place_x<float>(c, (const float*)dstage[b], c->n_loc, r0, nr, c->n_loc, 0);
        else launch_place_x<double>(c, (const double*)dstage[b], c->n_loc, r0, nr, c->n_loc, 0);
        UP(cudaGetLastError());
        UP(cudaEventRecord(cast_done[b], c->stream));
    }
#undef UP
    cleanup();
    return 0;
}

int pymfb_upload_x(pymfb_ctx* c, const void* x_host, int dtype, int64_t ld) {
    if (!c) return fail("null context");
    if (!x_host) return fail("x_host is null");
    if (ld < c->n_loc) return fail("leading dimension too small");
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    CU(cudaSetDevice(c->device));
    static const bool tlog = getenv("PYMFB_UPLOAD_LOG") != nullptr;      // experiment: phase times of the ingest on stderr
    const auto t0 = std::chrono::steady_clock::now();
    CK(ensure_own_x(c));
    if (tlog) CU(cudaStreamSynchronize(c->stream));
    const auto t1 = std::chrono::steady_clock::now();
    c->last_upload_pinned = host_is_pinned(x_host);
    if (c->last_upload_pinned) CK(pinned_upload(c, x_host, dtype, ld));
    else CK(staged_upload(c, x_host, dtype, ld));
    CU(cudaStreamSynchronize(c->stream));
    const auto t2 = std::chrono::steady_clock::now();
    const int rc = data_changed(c);
    if (tlog) {
        const auto t3 = std::chrono::steady_clock::now();
        auto sec = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
        fprintf(stderr, "[pymfb] upload_x: allocate + clear %.3f s, transfer %.3f s (%s), after %.3f s\n", sec(t0, t1), sec(t1, t2),
                c->last_upload_pinned ? "direct DMA" : "staged", sec(t2, t3));
    }
    return rc;
}

int pymfb_last_upload_pinned(pymfb_ctx* c) { return c && c->last_upload_pinned ? 1 : 0; }

static int factor_stage(pymfb_ctx* c, size_t bytes, void** out);

// ---- sparse X (include/pymfb.h, kernels_sparse.cuh) -----------------------------------------
// Stable radix sort of (keys[0], perm[0]) into (keys[1], perm[1]) on the bits of keys up to max_key.  Stable: equal
// keys keep their payload order, so everything built from the result is deterministic.  The CUB scratch is freed
// before returning (cudaFree waits for the sort).
static cudaError_t sort_pairs(pymfb_ctx* c, uint64_t* const keys[2], uint32_t* const perm[2], int64_t nnz, uint64_t max_key) {
    int end_bit = 1;
    while (end_bit < 64 && (max_key >> end_bit) != 0) ++end_bit;
    size_t temp_bytes = 0;
    void* temp = nullptr;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, temp_bytes, keys[0], keys[1], perm[0], perm[1], (int)nnz, 0, end_bit, c->stream);
    if (e == cudaSuccess) e = cudaMalloc(&temp, std::max<size_t>(temp_bytes, 16));
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(temp, temp_bytes, keys[0], keys[1], perm[0], perm[1], (int)nnz, 0, end_bit, c->stream);
    cudaFree(temp);
    return e;
}

// Column-panel CSR of s (CSC on the device): a stable radix sort of the entries by (panel, row) - the entry index is
// the payload, so a row keeps its column order and the build is deterministic - then the rows' offsets by binary search.
static int build_csr_panels(pymfb_ctx* c, SparseX& s) {
    const int64_t d = c->d, n = c->n_loc, nnz = s.nnz;
    // PYMFB_SPARSE_PANEL (experiment knob): panel width in columns; default: H^T rows of a panel fill ~ half the L2
    int64_t pw = (int64_t)(63 << 20) / ((int64_t)c->kp * 4);
    if (const char* e = getenv("PYMFB_SPARSE_PANEL")) { const int64_t v = atoll(e); if (v > 0) pw = v; }
    s.pw = std::max<int64_t>(1, std::min(pw, n));
    s.npanels = (int)((n + s.pw - 1) / s.pw);
    const int64_t nkeys = (int64_t)s.npanels * d;
    CU(cudaMalloc(&s.rowptr, (size_t)(nkeys + 1) * sizeof(int64_t)));
    CU(cudaMalloc(&s.ccol, (size_t)std::max<int64_t>(nnz, 1) * sizeof(int32_t)));
    CU(cudaMalloc(&s.cval, (size_t)std::max<int64_t>(nnz, 1) * sizeof(float)));
    int32_t* colof = nullptr;
    uint64_t* keys[2] = {nullptr, nullptr};
    uint32_t* perm[2] = {nullptr, nullptr};
    int rc = 0;
    auto cleanup = [&]() {
        cudaStreamSynchronize(c->stream);
        cudaFree(colof); cudaFree(keys[0]); cudaFree(keys[1]); cudaFree(perm[0]); cudaFree(perm[1]);
    };
#define SB(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    const int g = grid_for(std::max<int64_t>(nnz, 1), 256, 16 * c->sm_count);
    if (nnz > 0) {
        SB(cudaMalloc(&colof, (size_t)nnz * sizeof(int32_t)));
        for (int i = 0; i < 2; ++i) {
            SB(cudaMalloc(&keys[i], (size_t)nnz * sizeof(uint64_t)));
            SB(cudaMalloc(&perm[i], (size_t)nnz * sizeof(uint32_t)));
        }
        sp::k_csc_cols<<<grid_for(n * 32, 256, 16 * c->sm_count), 256, 0, c->stream>>>(s.colptr, n, colof);
        sp::k_csr_keys<<<g, 256, 0, c->stream>>>(s.rowidx, colof, nnz, d, s.pw, keys[0], perm[0]);
        SB(cudaGetLastError());
        SB(sort_pairs(c, keys, perm, nnz, (uint64_t)(nkeys - 1)));
        sp::k_csr_gather<<<g, 256, 0, c->stream>>>(perm[1], colof, s.vals, nnz, s.ccol, s.cval);
    }
    sp::k_csr_rowptr<<<grid_for(nkeys + 1, 256, 16 * c->sm_count), 256, 0, c->stream>>>(keys[1], nnz, nkeys, s.rowptr);
    c->launches += nnz > 0 ? 5 : 1;
    SB(cudaGetLastError());
#undef SB
    cleanup();
    return 0;
}

// Shared tail of the sparse uploads.  s holds a CSC X staged on the device (colptr, rowidx, vals, nnz); it is checked
// before any kernel indexes with it, the column-panel CSR is built from it, and it replaces whatever X was current.
// s is consumed: freed on failure (the context keeps its previous X), owned by the context on success.
static int sparse_commit(pymfb_ctx* c, SparseX& s) {
    const int64_t n = c->n_loc, nnz = s.nnz;
    int* flag = nullptr;
    int bad = 0, rc = 0;
    auto cleanup = [&]() { cudaStreamSynchronize(c->stream); cudaFree(flag); sparse_free(s); };
#define SU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    SU(cudaMalloc(&flag, sizeof(int)));
    SU(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
    // the arrays come from outside: no kernel indexes with them before this check has passed
    sp::k_csc_validate<<<grid_for(n * 32, 256, 16 * c->sm_count), 256, 0, c->stream>>>(s.colptr, s.rowidx, n, nnz, c->d, flag);
    c->launches += 1;
    SU(cudaGetLastError());
    SU(cudaMemcpyAsync(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    SU(cudaStreamSynchronize(c->stream));
    if (bad) {
        cleanup();
        return fail("malformed CSC matrix (%lld x %lld, nnz %lld):%s%s%s%s%s", (long long)c->d, (long long)n, (long long)nnz,
                    bad & sp::BAD_START ? " colptr[0] != 0;" : "", bad & sp::BAD_PTR_ORDER ? " colptr decreases;" : "",
                    bad & sp::BAD_END ? " colptr[n] != nnz;" : "", bad & sp::BAD_ROW ? " row index outside [0, d);" : "",
                    bad & sp::BAD_ROW_ORDER ? " row indices not strictly increasing within a column;" : "");
    }
    if ((rc = build_csr_panels(c, s)) != 0) { cleanup(); return rc; }
    // commit: the sparse X replaces whatever was current
    sparse_drop(c);
    if (c->X_own) { CU(cudaFree(c->X_own)); c->X_own = nullptr; }
    c->X = nullptr;
    tc_release(c->tc);
    fused_release(c->fused);
    c->sx = s;
    s = SparseX();
    cudaFree(flag); flag = nullptr;
    c->sparse = true;
    c->ht_of = -1;
    SU(cudaMalloc(&c->Ht, (size_t)n * c->kp * sizeof(float)));
    SU(cudaMalloc(&c->GH, (size_t)c->kp * c->ldh * sizeof(float)));
    {   // H H^T row splits: enough CTAs to cover the SMs, >= 64 rows of H^T each
        const int64_t tiles = ((c->kp + TILE_N - 1) / TILE_N) * (c->kp / c->kb);
        const int64_t want = std::min<int64_t>(std::max<int64_t>(1, (2LL * c->sm_count) / tiles), std::max<int64_t>(1, n / 64));
        c->hh_rows_per_split = round_up((n + want - 1) / want, TILE_DK);
        c->hh_splits = (int)((n + c->hh_rows_per_split - 1) / c->hh_rows_per_split);
        SU(cudaMalloc(&c->hh_part, (size_t)c->hh_splits * c->kp * c->kp * sizeof(float)));
    }
#undef SU
    c->last_upload_pinned = false;
    return data_changed(c);
}

int pymfb_upload_x_csc(pymfb_ctx* c, const int64_t* colptr, const int32_t* rowidx, const void* values, int dtype, int64_t nnz) {
    if (!c) return fail("null context");
    if (!colptr) return fail("colptr is null");
    if (nnz < 0 || nnz > (int64_t)INT32_MAX) return fail("nnz = %lld: 0 <= nnz < 2^31 supported", (long long)nnz);
    if (nnz > 0 && (!rowidx || !values)) return fail("rowidx / values are null");
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    if (c->path_opt != PYMFB_PATH_AUTO)
        return fail("sparse data runs on its own passes: the dense kernel families (path simt / tc) do not apply");
    CU(cudaSetDevice(c->device));
    const int64_t n = c->n_loc, nv = round_up(std::max<int64_t>(nnz, 1), 4);
    SparseX s;
    s.nnz = nnz;
    int rc = 0;
    auto cleanup = [&]() { cudaStreamSynchronize(c->stream); sparse_free(s); };
#define SU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    SU(cudaMalloc(&s.colptr, (size_t)(n + 1) * sizeof(int64_t)));
    SU(cudaMalloc(&s.rowidx, (size_t)std::max<int64_t>(nnz, 1) * sizeof(int32_t)));
    SU(cudaMalloc(&s.vals, (size_t)nv * sizeof(float)));
    SU(cudaMemsetAsync(s.vals, 0, (size_t)nv * sizeof(float), c->stream));
    SU(cudaMemcpyAsync(s.colptr, colptr, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    if (nnz > 0) {
        SU(cudaMemcpyAsync(s.rowidx, rowidx, (size_t)nnz * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        if (dtype == PYMFB_F32) {
            SU(cudaMemcpyAsync(s.vals, values, (size_t)nnz * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        } else {                                   // fp64 through the factor staging buffer, cast on the device
            void* stage = nullptr;
            if ((rc = factor_stage(c, (size_t)nnz * sizeof(double), &stage)) != 0) { cleanup(); return rc; }
            SU(cudaMemcpyAsync(stage, values, (size_t)nnz * sizeof(double), cudaMemcpyHostToDevice, c->stream));
            k_cast_in<double><<<grid_for(nnz, 256, 16 * c->sm_count), 256, 0, c->stream>>>((const double*)stage, nnz, s.vals, nnz, 1, nnz);
            c->launches += 1;
        }
    }
#undef SU
    return sparse_commit(c, s);
}

// An array pymfb_upload_x_sparse_device reads: device memory of the context's device, aligned to its elements.
static int check_device_array(const pymfb_ctx* c, const void* p, size_t elem, const char* what) {
    if (!p) return fail("%s: null pointer", what);
    if ((uintptr_t)p % elem != 0) return fail("%s: address not aligned to its %zu-byte elements", what, elem);
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return fail("%s: not a CUDA pointer", what); }
    if (at.type != cudaMemoryTypeDevice || at.device != c->device)
        return fail("%s must be device memory of device %d (memory type %d, device %d)", what, c->device, (int)at.type, at.device);
    return 0;
}

// The canonical CSC of a device COO / CSR / CSC input into s (kernels_sparse.cuh, "Device canonicalisation").
// Temporaries: sort keys and payloads (2 x 12 B per input entry), reused for the run slots and the unique keys, plus
// the CUB scratch; all freed before returning, after the stream has drained (the caller's arrays have been read).
extern "C++" {       // a template: C++ linkage inside the extern "C" block
template <typename T>
static int sparse_canonical_csc(pymfb_ctx* c, int layout, const T* a, const T* b, const void* values, int dtype,
                                int64_t nnz, SparseX& s) {
    const int64_t d = c->d, n = c->n_loc;
    const int64_t m = layout == PYMFB_LAYOUT_CSR ? d : n;          // pointer array of CSR / CSC: m + 1 entries
    int* flag = nullptr;
    uint64_t* keys[2] = {nullptr, nullptr};
    uint32_t* perm[2] = {nullptr, nullptr};
    void* temp = nullptr;
    int bad = 0, rc = 0;
    auto cleanup = [&]() {
        cudaStreamSynchronize(c->stream);
        cudaFree(flag); cudaFree(keys[0]); cudaFree(keys[1]); cudaFree(perm[0]); cudaFree(perm[1]); cudaFree(temp);
    };
#define SC(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
    const int g = grid_for(std::max<int64_t>(nnz, 1), 256, 16 * c->sm_count);
    // 1. the arrays come from outside: check them before any kernel indexes with their values
    SC(cudaMalloc(&flag, sizeof(int)));
    SC(cudaMemsetAsync(flag, 0, sizeof(int), c->stream));
    if (layout != PYMFB_LAYOUT_COO) {
        sp::k_sp_check_ptr<T><<<grid_for(m + 1, 256, 16 * c->sm_count), 256, 0, c->stream>>>(a, m, nnz, flag);
        c->launches += 1;
    }
    if (nnz > 0) {
        if (layout == PYMFB_LAYOUT_COO) {
            sp::k_sp_check_idx<T><<<g, 256, 0, c->stream>>>(a, nnz, d, sp::BAD_ROW, flag);
            c->launches += 1;
        }
        const bool rows = layout == PYMFB_LAYOUT_CSC;
        sp::k_sp_check_idx<T><<<g, 256, 0, c->stream>>>(b, nnz, rows ? d : n, rows ? sp::BAD_ROW : sp::BAD_COL, flag);
        c->launches += 1;
    }
    SC(cudaGetLastError());
    SC(cudaMemcpyAsync(&bad, flag, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    SC(cudaStreamSynchronize(c->stream));
    if (bad) {
        static const char* names[3] = {"COO", "CSR", "CSC"};
        cleanup();
        return fail("malformed %s matrix (%lld x %lld, nnz %lld):%s%s%s%s%s", names[layout], (long long)d, (long long)n,
                    (long long)nnz, bad & sp::BAD_START ? " pointers[0] != 0;" : "",
                    bad & sp::BAD_PTR_ORDER ? " pointers decrease;" : "", bad & sp::BAD_END ? " pointers[last] != nnz;" : "",
                    bad & sp::BAD_ROW ? " row index outside [0, d);" : "",
                    bad & sp::BAD_COL ? " column index outside [0, n_local);" : "");
    }
    SC(cudaMalloc(&s.colptr, (size_t)(n + 1) * sizeof(int64_t)));
    int64_t nu = 0;                                                // entries after the duplicates are summed
    if (nnz > 0) {
        // 2. (column, row) keys with the input position as payload, 3. stable sort
        for (int i = 0; i < 2; ++i) {
            SC(cudaMalloc(&keys[i], (size_t)nnz * sizeof(uint64_t)));
            SC(cudaMalloc(&perm[i], (size_t)nnz * sizeof(uint32_t)));
        }
        if (layout == PYMFB_LAYOUT_COO)
            sp::k_sp_keys_coo<T><<<g, 256, 0, c->stream>>>(a, b, nnz, d, keys[0], perm[0]);
        else
            sp::k_sp_keys_ptr<T><<<grid_for(m * 32, 256, 16 * c->sm_count), 256, 0, c->stream>>>(a, b, m, d, layout == PYMFB_LAYOUT_CSC, keys[0], perm[0]);
        SC(cudaGetLastError());
        SC(sort_pairs(c, keys, perm, nnz, (uint64_t)n * (uint64_t)d - 1));
        // 4. runs of equal keys: heads in perm[0] (free after the sort), scanned in place into 1 + each run's slot
        uint32_t* slot = perm[0];
        sp::k_sp_heads<<<g, 256, 0, c->stream>>>(keys[1], nnz, slot);
        SC(cudaGetLastError());
        size_t temp_bytes = 0;
        SC(cub::DeviceScan::InclusiveSum(nullptr, temp_bytes, slot, slot, (int)nnz, c->stream));
        SC(cudaMalloc(&temp, std::max<size_t>(temp_bytes, 16)));
        SC(cub::DeviceScan::InclusiveSum(temp, temp_bytes, slot, slot, (int)nnz, c->stream));
        uint32_t nu32 = 0;
        SC(cudaMemcpyAsync(&nu32, slot + nnz - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        SC(cudaStreamSynchronize(c->stream));
        nu = nu32;
        c->launches += 3;
    }
    const int64_t nv = round_up(std::max<int64_t>(nu, 1), 4);
    SC(cudaMalloc(&s.rowidx, (size_t)std::max<int64_t>(nu, 1) * sizeof(int32_t)));
    SC(cudaMalloc(&s.vals, (size_t)nv * sizeof(float)));
    SC(cudaMemsetAsync(s.vals, 0, (size_t)nv * sizeof(float), c->stream));
    s.nnz = nu;
    if (nnz > 0) {
        // sums into the CSC; the unique keys go to keys[0] (free after the sort), 5. column pointers from them
        if (dtype == PYMFB_F64)
            sp::k_sp_sum_runs<double><<<g, 256, 0, c->stream>>>(keys[1], perm[1], perm[0], (const double*)values, nnz, d, s.rowidx, s.vals, keys[0]);
        else
            sp::k_sp_sum_runs<float><<<g, 256, 0, c->stream>>>(keys[1], perm[1], perm[0], (const float*)values, nnz, d, s.rowidx, s.vals, keys[0]);
        sp::k_sp_colptr<<<grid_for(n + 1, 256, 16 * c->sm_count), 256, 0, c->stream>>>(keys[0], nu, n, d, s.colptr);
        c->launches += 2;
    } else {
        SC(cudaMemsetAsync(s.colptr, 0, (size_t)(n + 1) * sizeof(int64_t), c->stream));
    }
    SC(cudaGetLastError());
#undef SC
    cleanup();
    return 0;
}
}  // extern "C++"

int pymfb_upload_x_sparse_device(pymfb_ctx* c, int layout, const void* a, const void* b, int index_dtype,
                                 const void* values, int dtype, int64_t nnz) {
    if (!c) return fail("null context");
    if (layout != PYMFB_LAYOUT_COO && layout != PYMFB_LAYOUT_CSR && layout != PYMFB_LAYOUT_CSC) return fail("bad layout %d", layout);
    if (index_dtype != PYMFB_I32 && index_dtype != PYMFB_I64) return fail("bad index dtype %d", index_dtype);
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    if (nnz < 0 || nnz > (int64_t)INT32_MAX) return fail("nnz = %lld: 0 <= nnz < 2^31 supported", (long long)nnz);
    if (c->path_opt != PYMFB_PATH_AUTO)
        return fail("sparse data runs on its own passes: the dense kernel families (path simt / tc) do not apply");
    CU(cudaSetDevice(c->device));
    const size_t isz = index_dtype == PYMFB_I64 ? 8 : 4;
    if (layout != PYMFB_LAYOUT_COO) CK(check_device_array(c, a, isz, layout == PYMFB_LAYOUT_CSR ? "row pointers" : "column pointers"));
    if (nnz > 0) {
        if (layout == PYMFB_LAYOUT_COO) CK(check_device_array(c, a, isz, "row indices"));
        CK(check_device_array(c, b, isz, layout == PYMFB_LAYOUT_CSC ? "row indices" : "column indices"));
        CK(check_device_array(c, values, dtype == PYMFB_F64 ? 8 : 4, "values"));
    }
    SparseX s;
    const int rc = index_dtype == PYMFB_I64
                       ? sparse_canonical_csc<int64_t>(c, layout, (const int64_t*)a, (const int64_t*)b, values, dtype, nnz, s)
                       : sparse_canonical_csc<int32_t>(c, layout, (const int32_t*)a, (const int32_t*)b, values, dtype, nnz, s);
    if (rc != 0) { cudaStreamSynchronize(c->stream); sparse_free(s); return rc; }
    return sparse_commit(c, s);
}

// ---- panel-streamed ingest (include/pymfb.h) --------------------------------------------------
int pymfb_upload_x_begin(pymfb_ctx* c) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CK(ensure_own_x(c));
    for (int s = 0; s < 2; ++s)
        if (!c->panel_ev[s]) CU(cudaEventCreateWithFlags(&c->panel_ev[s], cudaEventDisableTiming));
    c->panel_open = true;
    c->last_upload_pinned = true;
    return 0;
}
int pymfb_upload_x_panel(pymfb_ctx* c, const void* host, int dtype, int64_t ld, int64_t col0, int64_t ncols, int slot) {
    if (!c) return fail("null context");
    if (!c->panel_open) return fail("pymfb_upload_x_panel without pymfb_upload_x_begin");
    if (!host) return fail("panel_host is null");
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    if (slot < 0 || slot > 1) return fail("slot must be 0 or 1");
    if (col0 < 0 || ncols <= 0 || col0 + ncols > c->n_loc || ld < ncols) return fail("bad panel: col0=%lld ncols=%lld ld=%lld n_local=%lld", (long long)col0, (long long)ncols, (long long)ld, (long long)c->n_loc);
    CU(cudaSetDevice(c->device));
    if (!host_is_pinned(host)) c->last_upload_pinned = false;      // the runtime stages pageable panels itself (synchronous)
    if (dtype == PYMFB_F32 && c->xps == 0) {
        CU(cudaMemcpy2DAsync(c->X_own + col0, c->ldx * sizeof(float), host, (size_t)ld * sizeof(float), (size_t)ncols * sizeof(float),
                             (size_t)c->d, cudaMemcpyHostToDevice, c->stream));
    } else {                                   // cast (fp64) and / or scatter into the panel-major layout on the device
        const size_t esz = dtype == PYMFB_F32 ? 4 : 8;
        const size_t need = (size_t)c->d * ncols * esz;
        if (need > c->panel_stage_bytes[slot]) {
            CU(cudaStreamSynchronize(c->stream));
            if (c->panel_stage[slot]) CU(cudaFree(c->panel_stage[slot]));
            c->panel_stage[slot] = nullptr; c->panel_stage_bytes[slot] = 0;
            CU(cudaMalloc(&c->panel_stage[slot], need));
            c->panel_stage_bytes[slot] = need;
        }
        CU(cudaMemcpy2DAsync(c->panel_stage[slot], (size_t)ncols * esz, host, (size_t)ld * esz,
                             (size_t)ncols * esz, (size_t)c->d, cudaMemcpyHostToDevice, c->stream));
        if (dtype == PYMFB_F32) launch_place_x<float>(c, (const float*)c->panel_stage[slot], ncols, 0, c->d, ncols, col0);
        else launch_place_x<double>(c, (const double*)c->panel_stage[slot], ncols, 0, c->d, ncols, col0);
        CU(cudaGetLastError());
    }
    CU(cudaEventRecord(c->panel_ev[slot], c->stream));
    return 0;
}
int pymfb_upload_x_wait(pymfb_ctx* c, int slot) {
    if (!c) return fail("null context");
    if (slot < 0 || slot > 1) return fail("slot must be 0 or 1");
    if (c->panel_ev[slot]) CU(cudaEventSynchronize(c->panel_ev[slot]));
    return 0;
}
int pymfb_upload_x_end(pymfb_ctx* c) {
    if (!c) return fail("null context");
    if (!c->panel_open) return fail("pymfb_upload_x_end without pymfb_upload_x_begin");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    for (int s = 0; s < 2; ++s) { if (c->panel_stage[s]) cudaFree(c->panel_stage[s]); c->panel_stage[s] = nullptr; c->panel_stage_bytes[s] = 0; }
    c->panel_open = false;
    return data_changed(c);
}

// ---- NUMA-aware page-locked host memory ---------------------------------------------------
// Page-locked buffers are placed on the GPU's own NUMA node when the OS exposes one: mmap + mbind(preferred node)
// + cudaHostRegister (DMA across sockets is typically 2-3x slower).  The GPU boxes of this project are single-node
// VMs (numa_node = -1), where this degrades to plain cudaHostAlloc; the H2D rate there varied between 20 and
// 53 GB/s from box to box with identical code (VM placement), see DESIGN.md 5.3.
int pymfb_device_numa_node(int device) {
    char bus[64] = "";
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* q = bus; *q; ++q) *q = (char)tolower((unsigned char)*q);
    char path[160];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

int pymfb_host_node_of(const void* p) {
    if (!p) return -1;
    void* page = (void*)((uintptr_t)p & ~(uintptr_t)4095);
    int status = -1;
    long rc = syscall(SYS_move_pages, 0, 1UL, &page, (const int*)nullptr, &status, 0);
    return rc == 0 ? status : -1;
}

static std::mutex g_host_mu;
static std::map<void*, size_t> g_host_mapped;      // buffers made by mmap + cudaHostRegister

static void* numa_pinned_alloc(size_t bytes, int node) {
    if (node < 0 || node >= 1024) return nullptr;
    const size_t len = (bytes + 4095) & ~(size_t)4095;
    void* p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return nullptr;
    unsigned long mask[16] = {0};
    mask[node / 64] = 1UL << (node % 64);
    // MPOL_PREFERRED = 1: falls back to other nodes instead of failing when the node is full or not allowed
    if (syscall(SYS_mbind, p, len, 1, mask, 1025UL, 0) != 0) { munmap(p, len); return nullptr; }
    if (cudaHostRegister(p, len, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); munmap(p, len); return nullptr; }
    std::lock_guard<std::mutex> lk(g_host_mu);
    g_host_mapped[p] = len;
    return p;
}

int pymfb_host_alloc(void** out, size_t bytes) {
    if (!out) return fail("out is null");
    *out = nullptr;
    if (pymfb_device_count() <= 0) return fail("no CUDA device available: page-locked memory needs the driver");
    if (!bytes) bytes = 1;
    int dev = 0;
    CU(cudaGetDevice(&dev));
    static const bool numa_off = getenv("PYMFB_NO_NUMA") != nullptr;
    if (!numa_off) {
        void* p = numa_pinned_alloc(bytes, pymfb_device_numa_node(dev));
        if (p) { *out = p; return 0; }
    }
    CU(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
    return 0;
}
int pymfb_host_free(void* p) {
    if (!p) return 0;
    size_t len = 0;
    {
        std::lock_guard<std::mutex> lk(g_host_mu);
        auto it = g_host_mapped.find(p);
        if (it != g_host_mapped.end()) { len = it->second; g_host_mapped.erase(it); }
    }
    if (len) {
        cudaHostUnregister(p);
        cudaGetLastError();
        munmap(p, len);
        return 0;
    }
    CU(cudaFreeHost(p));
    return 0;
}

int pymfb_gen_x(pymfb_ctx* c, uint64_t seed) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CK(ensure_own_x(c));
    k_gen_uniform<<<grid_for(c->d * c->n_loc, 256, 32 * c->sm_count), 256, 0, c->stream>>>(
        c->X_own, c->ldx, c->d, c->n_loc, seed, c->n_glob, c->col0, c->xps, c->xsh);
    c->launches += 1;
    CU(cudaGetLastError());
    return data_changed(c);
}

// Device staging buffer of the factor transfers (grow-only, owned by the context: a cudaMalloc / cudaFree pair
// per set/get call showed up as 10 - 1000 ms stalls next to the frees of a previous 4 GiB engine).
static int factor_stage(pymfb_ctx* c, size_t bytes, void** out) {
    if (bytes > c->stage_bytes) {
        if (c->stage) { CU(cudaStreamSynchronize(c->stream)); CU(cudaFree(c->stage)); c->stage = nullptr; c->stage_bytes = 0; }
        CU(cudaMalloc(&c->stage, bytes));
        c->stage_bytes = bytes;
    }
    *out = c->stage;
    return 0;
}

// host (rows x cols, dense, dtype) -> device fp32 (rows x ldd), padding zeroed
static int set_factor(pymfb_ctx* c, float* dst, int64_t ldd, int64_t rows_alloc, int64_t rows, int64_t cols,
                      const void* host, int dtype) {
    if (!host) return fail("host pointer is null");
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    CU(cudaSetDevice(c->device));
    const size_t esz = dtype == PYMFB_F32 ? 4 : 8;
    void* stage = nullptr;
    CK(factor_stage(c, (size_t)rows * cols * esz, &stage));
    CU(cudaMemcpyAsync(stage, host, (size_t)rows * cols * esz, cudaMemcpyHostToDevice, c->stream));
    CU(cudaMemsetAsync(dst, 0, (size_t)rows_alloc * ldd * sizeof(float), c->stream));
    const int g = grid_for(rows * cols, 256, 16 * c->sm_count);
    if (dtype == PYMFB_F32) k_cast_in<float><<<g, 256, 0, c->stream>>>((const float*)stage, cols, dst, ldd, rows, cols);
    else k_cast_in<double><<<g, 256, 0, c->stream>>>((const double*)stage, cols, dst, ldd, rows, cols);
    c->launches += 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}
static int get_factor(pymfb_ctx* c, const float* src, int64_t lds, int64_t rows, int64_t cols, void* host, int dtype) {
    if (!host) return fail("host pointer is null");
    if (dtype != PYMFB_F32 && dtype != PYMFB_F64) return fail("bad dtype %d", dtype);
    CU(cudaSetDevice(c->device));
    const size_t esz = dtype == PYMFB_F32 ? 4 : 8;
    void* stage = nullptr;
    CK(factor_stage(c, (size_t)rows * cols * esz, &stage));
    const int g = grid_for(rows * cols, 256, 16 * c->sm_count);
    if (dtype == PYMFB_F32) k_cast_out<float><<<g, 256, 0, c->stream>>>(src, lds, (float*)stage, cols, rows, cols);
    else k_cast_out<double><<<g, 256, 0, c->stream>>>(src, lds, (double*)stage, cols, rows, cols);
    c->launches += 1;
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(host, stage, (size_t)rows * cols * esz, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}

int pymfb_set_w(pymfb_ctx* c, const void* w_host, int dtype) {
    if (!c) return fail("null context");
    CK(set_factor(c, c->W[c->wcur], c->kp, c->d, c->d, c->k, w_host, dtype));
    c->w_set = true; c->g_valid = false;
    return 0;
}
int pymfb_set_h(pymfb_ctx* c, const void* h_host, int dtype) {
    if (!c) return fail("null context");
    CK(set_factor(c, c->H[c->hcur], c->ldh, c->kp, c->k, c->n_loc, h_host, dtype));
    c->h_set = true; c->ab_valid = false; c->tc.hs_valid[c->hcur] = false; c->ht_of = -1;
    return 0;
}
int pymfb_get_w(pymfb_ctx* c, void* w_host, int dtype) {
    if (!c) return fail("null context");
    if (!c->w_set) return fail("W is not set");
    return get_factor(c, c->W[c->wcur], c->kp, c->d, c->k, w_host, dtype);
}
int pymfb_get_h(pymfb_ctx* c, void* h_host, int dtype) {
    if (!c) return fail("null context");
    if (!c->h_set) return fail("H is not set");
    return get_factor(c, c->H[c->hcur], c->ldh, c->k, c->n_loc, h_host, dtype);
}
int pymfb_gen_w(pymfb_ctx* c, uint64_t seed) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CU(cudaMemsetAsync(c->W[c->wcur], 0, (size_t)c->d * c->kp * sizeof(float), c->stream));
    k_gen_uniform<<<grid_for(c->d * c->k, 256, 16 * c->sm_count), 256, 0, c->stream>>>(c->W[c->wcur], c->kp, c->d, c->k, seed, c->k, 0);
    c->launches += 1;
    CU(cudaGetLastError());
    c->w_set = true; c->g_valid = false;
    return 0;
}
int pymfb_gen_h(pymfb_ctx* c, uint64_t seed) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CU(cudaMemsetAsync(c->H[c->hcur], 0, (size_t)c->kp * c->ldh * sizeof(float), c->stream));
    k_gen_uniform<<<grid_for((int64_t)c->k * c->n_loc, 256, 16 * c->sm_count), 256, 0, c->stream>>>(c->H[c->hcur], c->ldh, c->k, c->n_loc, seed, c->n_glob, c->col0);
    c->launches += 1;
    CU(cudaGetLastError());
    c->h_set = true; c->ab_valid = false; c->tc.hs_valid[c->hcur] = false; c->ht_of = -1;
    return 0;
}

// ---- NNDSVD initialisation (pymf/nndsvd.py:79-108), kernels_svd.cuh -----------------------------
// The tensor-core passes by default only beyond the graph-replay sizes, the rule of the one-pass NMF kernel: below it the
// CUDA-core passes keep the results of the tested shapes as they were.  Where the tensor-core width enlarges the block
// (b = 160..224 -> 256, one GPU) the b x b work of the wider block outweighs the faster passes up to much larger X
// (measured, DESIGN 5.7: 16384 x 131072 k=128 0.81x, 8192 x 524288 k=128 1.22x).
static const double kNndsvdTcMinWork = 16777216.0;     // d * n_local
static const double kNndsvdTcMinWorkWider = 4294967296.0;
int pymfb_nndsvd(pymfb_ctx* c, int max_iter, double tol, int extra_iter, int* iters_done, double* sigma_out) {
    if (!c) return fail("null context");
    if (c->sparse) return fail("NNDSVD of sparse data is not supported: upload a dense X");
    if (!c->X) return fail("no data bound: call pymfb_bind_x / pymfb_upload_x / pymfb_gen_x first");
    if (c->world > 1 && !c->comm) return fail("pymfb_nndsvd: world = %d but no communicator is attached", c->world);
    if (max_iter < 1) max_iter = 100;
    if (extra_iter < 0) extra_iter = 6;
    CU(cudaSetDevice(c->device));
    const int k = c->k;
    const int b_simt = (int)round_up(k + std::max(8, k / 4), 32);     // block of the subspace iteration (oversampled)
    if (b_simt > 256) return fail("NNDSVD supports k <= 200 (subspace block %d > 256)", b_simt);
    const int b_tc = b_simt <= 128 ? b_simt : 256;                      // a width the SS kernels take (256: two 128-wide blocks)
    const int64_t d = c->d, n = c->n_loc, ldz = c->ldh;
    std::string why;
    const bool tc_ok = tc_supported(d, n, b_tc, c->ldx, c->X, &why);
    const double dn = (double)d * (double)n;
    bool use_tc = tc_ok && dn > kNndsvdTcMinWork && (b_tc == b_simt || c->world > 1 || dn >= kNndsvdTcMinWorkWider);
    if (c->nndsvd_path_opt == PYMFB_PATH_SIMT) use_tc = false;
    if (c->nndsvd_path_opt == PYMFB_PATH_TC) {
        if (!tc_ok) return fail("tcgen05 path not available for NNDSVD on this shape: %s", why.c_str());
        use_tc = true;
    }
    // Shards pick their pass family on their own (a narrow one stays on the CUDA cores), so a sharded run iterates the
    // tensor-core width on every rank: the collectives below need the same block everywhere.  Extra vectors only oversample.
    const int b = (use_tc || c->world > 1) ? b_tc : b_simt;
    if (!(tol > 0.0)) tol = 3e-7;
    const int b_real = (int)std::min<int64_t>(b, std::min(d, c->n_glob));
    cudaStream_t s = c->stream;
    float *Q = nullptr, *Y = nullptr, *Zt = nullptr, *Zt2 = nullptr, *Rm = nullptr, *Rt = nullptr, *Ct = nullptr, *Ppart = nullptr;
    double *gpart = nullptr, *Tm = nullptr, *work = nullptr, *vals = nullptr, *norms = nullptr;
    TcPlan tp;                                                  // Q^T X / X Z^T on the tensor cores (use_tc), freed below
    // X Z^T launches: column splits combined deterministically (k_xht_simt)
    const int64_t rowblocks = (d + 127) / 128, kblocks = b / 32, chunks = (n + XHT_CK - 1) / XHT_CK;
    int64_t want = std::min<int64_t>(chunks, std::max<int64_t>(1, (4LL * c->sm_count) / (rowblocks * kblocks)));
    const int64_t chunks_per = (chunks + want - 1) / want;
    const int64_t cps = chunks_per * XHT_CK;
    const unsigned ns = (unsigned)((chunks + chunks_per - 1) / chunks_per);
    const int gsplit_n = (int)std::max<int64_t>(1, std::min<int64_t>(256, n / 2048));
    const int gsplit_d = (int)std::max<int64_t>(1, std::min<int64_t>(64, d / 512));
    const int nb2 = ((b + 63) / 64) * ((b + 63) / 64);
    int rc = 0;
    auto cleanup = [&]() {
        cudaStreamSynchronize(s);
        cudaFree(Q); cudaFree(Y); cudaFree(Zt); cudaFree(Zt2); cudaFree(Rm); cudaFree(Rt); cudaFree(Ct); cudaFree(Ppart);
        cudaFree(gpart); cudaFree(Tm); cudaFree(work); cudaFree(vals); cudaFree(norms);
        tc_release(tp);
    };
#define SV(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            rc = fail("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));        \
            cleanup();                                                                             \
            return rc;                                                                             \
        }                                                                                          \
    } while (0)
#define SK(call)                                                                                   \
    do {                                                                                           \
        if ((rc = (call)) != 0) { cleanup(); return rc; }                                          \
    } while (0)
    SV(cudaMalloc(&Q, (size_t)d * b * 4)); SV(cudaMalloc(&Y, (size_t)d * b * 4));
    SV(cudaMalloc(&Zt, (size_t)b * ldz * 4)); SV(cudaMalloc(&Zt2, (size_t)b * ldz * 4));
    SV(cudaMemsetAsync(Zt, 0, (size_t)b * ldz * 4, s)); SV(cudaMemsetAsync(Zt2, 0, (size_t)b * ldz * 4, s));
    SV(cudaMalloc(&Rm, (size_t)b * b * 4)); SV(cudaMalloc(&Rt, (size_t)b * b * 4)); SV(cudaMalloc(&Ct, (size_t)b * b * 4));
    SV(cudaMalloc(&gpart, (size_t)std::max(gsplit_n, gsplit_d) * b * b * 8)); SV(cudaMalloc(&Tm, (size_t)b * b * 8));
    SV(cudaMalloc(&work, (size_t)2 * b * b * 8)); SV(cudaMalloc(&vals, (size_t)b * 8)); SV(cudaMalloc(&norms, (size_t)4 * b * 8));
    // (a non-null Ppart selects k_xht_simt's overwrite mode, also for a single split)
    SV(cudaMalloc(&Ppart, ns > 1 && !use_tc ? (size_t)ns * d * b * 4 : 16));
    if (use_tc && tc_plan(tp, c->device, c->sm_count, d, n, b, b, c->X, c->ldx, ldz, Zt, Zt2, c->xps, c->xsh, true)) {
        rc = fail("tcgen05 plan for NNDSVD failed: %s", tp.err.c_str());
        cleanup();
        return rc;
    }
    // in-place sum over the ranks on the context's stream (replicated quantities: the same on every rank afterwards)
    auto rank_sum = [&](void* buf, size_t count, int dtype) -> int {
        if (c->world == 1) return 0;
        const int r = g_nccl.AllReduce(buf, buf, count, dtype, kNcclSum, c->comm, s);
        return r ? fail("NNDSVD ncclAllReduce -> nccl error %d (%s)", r, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?") : 0;
    };
    // G = A^T A (by_rows = 0, A: len x b) or A A^T (by_rows = 1, A: b x len) in fp64 -> Tm
    auto gram = [&](const float* A, int64_t ld, int64_t len, int by_rows) {
        const int sp = by_rows ? gsplit_n : gsplit_d;
        const int64_t per = round_up((len + sp - 1) / sp, svd::GR_T);
        const int sp_eff = (int)((len + per - 1) / per);
        svd::k_gram_f64<<<dim3((unsigned)sp_eff, (unsigned)nb2), 256, 0, s>>>(A, ld, b, len, by_rows, per, gpart);
        svd::k_sum_f64<<<(unsigned)(((int64_t)b * b + 255) / 256), 256, 0, s>>>(gpart, sp_eff, (int64_t)b * b, Tm);
        c->launches += 2;
    };
    // Out (d x b) = A (d x b) * M where Mt = M^T is b x b row-major:  Out[r][i] = sum_j A[r][j] Mt[i][j]
    auto right_mul = [&](const float* A, const float* Mt, float* Out) {
        k_xht_simt<32><<<dim3((unsigned)rowblocks, 1, (unsigned)kblocks), SIMT_THREADS, 0, s>>>(
            c->st, A, b, d, Mt, b, b, b, Out, b, (int)rowblocks, 0, nullptr, Ppart, 0);
        c->launches += 1;
    };
    // Out (b x n) = L^T In with L b x b row-major (L[j][i]):  Out[i][col] = sum_j L[j][i] In[j][col]
    auto left_mul_t = [&](const float* L, int64_t ldl, int64_t rows, const float* In, int64_t ldin, float* Out) {
        const bool is_x = In == c->X;                             // the data matrix may be panel-major
        k_ltr_partial_simt<32><<<dim3((unsigned)((n + TILE_N - 1) / TILE_N), (unsigned)kblocks, 1), SIMT_THREADS, 0, s>>>(
            c->st, L, ldl, In, ldin, n, rows, rows, Out, ldz, b, is_x ? c->xps : 0, is_x ? c->xsh : kNoPanelShift);
        c->launches += 1;
    };
    auto orthonormalise = [&](const float* A, float* Out) {      // Out = A L^-T with L L^T = A^T A
        gram(A, b, d, 0);
        svd::k_chol_inv_f64<<<1, 256, 0, s>>>(Tm, b, work, Ct);
        c->launches += 1;
        right_mul(A, Ct, Out);
    };
    auto rayleigh_ritz = [&]() -> int {                          // Zt = Q^T X; eigh(sum over ranks of Zt Zt^T) -> vals, Rm, Rt
        if (use_tc) {
            if (tc_qtx(tp, c->st, Q, Zt, s, &c->launches)) return fail("tcgen05 Q^T X launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        } else {
            left_mul_t(Q, b, d, c->X, c->ldx, Zt);
        }
        gram(Zt, ldz, n, 1);
        CK(rank_sum(Tm, (size_t)b * b, kNcclFloat64));
        svd::k_jacobi_eigh_f64<<<1, 256, 0, s>>>(Tm, b, work, vals, Rm, Rt);
        c->launches += 1;
        return 0;
    };
    auto x_zt = [&]() -> int {                                   // Y = sum over ranks of X Zt2^T
        if (use_tc) {
            if (tc_xzt(tp, c->st, Y, s, &c->launches)) return fail("tcgen05 X Z^T launch failed: %s", cudaGetErrorString(cudaGetLastError()));
        } else {
            k_xht_simt<32><<<dim3((unsigned)rowblocks, ns, (unsigned)kblocks), SIMT_THREADS, 0, s>>>(
                c->st, c->X, c->ldx, d, Zt2, ldz, n, cps, Y, b, (int)rowblocks, 0, nullptr, Ppart, d * b, c->xps, c->xsh);
            if (ns > 1)
                tc::k_sum_copies<<<grid_for(d * b / 4, 256, 4 * c->sm_count), 256, 0, s>>>(c->st, Ppart, (int)ns, d * b, Y, nullptr, 0, 0, nullptr);
            c->launches += 2;
        }
        return rank_sum(Y, (size_t)d * b, kNcclFloat32);
    };
    svd::k_svd_seed<<<(unsigned)((d * b + 255) / 256), 256, 0, s>>>(Y, d, b, b_real, 0x5EEDull);
    c->launches += 1;
    orthonormalise(Y, Q);
    std::vector<double> ev(b, 0.0), prev(b, 0.0);
    int it = 0, settled = -1;
    double worst = 0.0;
    for (; it < max_iter; ++it) {
        SK(rayleigh_ritz());
        left_mul_t(Rm, b, b, Zt, ldz, Zt2);                      // rows of Zt2: (Ritz vector)^T X
        SK(x_zt());
        orthonormalise(Y, Q);                                    // Y = X X^T (Ritz vectors) -> next Q
        SV(cudaGetLastError());
        SV(cudaMemcpyAsync(ev.data(), vals, (size_t)b * 8, cudaMemcpyDeviceToHost, s));
        SV(cudaStreamSynchronize(s));
        worst = 0.0;
        for (int i = 0; i < k; ++i) worst = std::max(worst, std::fabs(ev[i] - prev[i]) / std::max(std::fabs(ev[i]), 1e-300));
        prev = ev;
        if (settled < 0 && it > 0 && worst < tol) settled = it;
        if (settled >= 0 && it >= settled + extra_iter) { ++it; break; }
    }
    // final extraction with the converged basis: U = Q R, S = sqrt(vals), S V^T = R^T Q^T X
    SK(rayleigh_ritz());
    right_mul(Q, Rt, Y);                                         // U -> Y
    left_mul_t(Rm, b, b, Zt, ldz, Zt2);                          // S V^T -> Zt2
    svd::k_posneg_norms<<<dim3((unsigned)k, 2), 256, 0, s>>>(Y, b, d, Zt2, ldz, n, vals, norms);
    c->launches += 1;
    if (c->world > 1) {
        // |u+|, |u-| (entries 0, 1 of each basis) are the same on every rank: rank 0 contributes them, the others 0 (exact),
        // so that one sum gives |v+|^2, |v-|^2 over all columns and leaves the u norms as they are
        if (c->rank != 0) SV(cudaMemset2DAsync(norms, 4 * sizeof(double), 0, 2 * sizeof(double), (size_t)k, s));
        SK(rank_sum(norms, (size_t)4 * k, kNcclFloat64));
    }
    SV(cudaMemsetAsync(c->W[c->wcur], 0, (size_t)d * c->kp * sizeof(float), s));
    SV(cudaMemsetAsync(c->H[c->hcur], 0, (size_t)c->kp * c->ldh * sizeof(float), s));
    svd::k_nndsvd_fill<<<dim3((unsigned)std::min<int64_t>((d + n + 255) / 256, 8 * c->sm_count), (unsigned)k), 256, 0, s>>>(
        Y, b, d, Zt2, ldz, n, vals, norms, k, c->W[c->wcur], c->kp, c->H[c->hcur], c->ldh);
    c->launches += 1;
    SV(cudaGetLastError());
    SV(cudaMemcpyAsync(ev.data(), vals, (size_t)b * 8, cudaMemcpyDeviceToHost, s));
    SV(cudaStreamSynchronize(s));
#undef SV
#undef SK
    cleanup();
    if (sigma_out) for (int i = 0; i < k; ++i) sigma_out[i] = std::sqrt(std::max(ev[i], 0.0));
    if (iters_done) *iters_done = it;
    c->nndsvd_path = use_tc ? PYMFB_PATH_TC : PYMFB_PATH_SIMT;
    c->nndsvd_change = worst;
    c->w_set = c->h_set = true;
    c->g_valid = false; c->ab_valid = false; c->p_zeroed = false;
    c->tc.hs_valid[0] = c->tc.hs_valid[1] = false;
    return 0;
}
int pymfb_nndsvd_info(pymfb_ctx* c, int* path, double* change) {
    if (!c) return fail("null context");
    if (path) *path = c->nndsvd_path;
    if (change) *change = c->nndsvd_change;
    return 0;
}

int pymfb_run(pymfb_ctx* c, int niter, unsigned flags, double* ferr_host, int* n_iter_done, int* n_ferr) {
    CK(check_ready(c));
    if (niter < 0) return fail("niter < 0");
    const bool do_e = flags & PYMFB_COMPUTE_ERR;
    if (do_e && niter > 0 && !ferr_host) return fail("ferr_host is null but PYMFB_COMPUTE_ERR is set");
    CU(cudaSetDevice(c->device));
    if (do_e && niter > c->ferr_cap) {
        if (c->ferr_dev) CU(cudaFree(c->ferr_dev));
        graph_drop(c); c->graph_key = 0;       // the graph holds the old ferr pointer
        c->ferr_cap = std::max(niter, 1024);
        CU(cudaMalloc(&c->ferr_dev, sizeof(double) * c->ferr_cap));
    }
    const int w0 = c->wcur, h0 = c->hcur;
    const double lw0 = c->lam_w, lh0 = c->lam_h;
    CK(enqueue_iterations(c, niter, flags));
    DevState hs;
    CU(cudaMemcpyAsync(&hs, c->st, sizeof(hs), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    CK(note_cancellation(c, hs));
    int done = niter, nf = do_e ? niter : 0;
    if (hs.stop) {
        // converged(i) fired at i = n_exec - 1: W/H keep iteration i's update, entry i of ferr
        // is dropped (pymf/nmf.py:199-202).  Kernels after the stop were no-ops, so the live
        // ping-pong buffers are the ones after n_exec swaps.
        done = hs.n_exec;
        nf = hs.n_exec - 1;
        if (flags & PYMFB_COMPUTE_W) c->wcur = w0 ^ (done & 1);
        if (flags & PYMFB_COMPUTE_H) c->hcur = h0 ^ (done & 1);
        CU(cudaMemsetAsync(&c->st->stop, 0, sizeof(int), c->stream));
        c->g_valid = false;   // recomputed lazily for the surviving W
        c->p_zeroed = false;  // kernels after the stop (incl. the one that clears P) were no-ops
        c->ab_valid = false;
        c->tc.hs_valid[0] = c->tc.hs_valid[1] = false;
        c->ht_of = -1;
        if (flags & PYMFB_COMPUTE_H) {   // the penalty weights grew once per EXECUTED update_h only
            c->lam_w = lw0; c->lam_h = lh0;
            for (int i = 0; i < done; ++i) { c->lam_w *= c->inc_w; c->lam_h *= c->inc_h; }
        }
    }
    if (do_e && nf > 0) CU(cudaMemcpyAsync(ferr_host, c->ferr_dev, sizeof(double) * nf, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (n_iter_done) *n_iter_done = done;
    if (n_ferr) *n_ferr = nf;
    return 0;
}

int pymfb_frobenius(pymfb_ctx* c, double* out) {
    CK(check_ready(c));
    if (!out) return fail("out is null");
    CU(cudaSetDevice(c->device));
    if (!c->err_direct) {
        if (!c->xx_valid) CK(launch_xx(c));
        if (!c->g_valid) CK(launch_gram_w(c));
        if (!c->ab_valid) CK(launch_xht(c));
    }
    CK(launch_err(c, false, false));
    DevState hs;
    CU(cudaMemcpyAsync(&hs, c->st, sizeof(hs), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (hs.cancel && !c->err_direct) {           // the identity cancelled: measure this value directly instead
        CK(note_cancellation(c, hs));
        if (c->err_direct) {
            CK(launch_err(c, false, false));
            CU(cudaMemcpyAsync(&hs, c->st, sizeof(hs), cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
        }
    }
    *out = hs.last_ferr;
    return 0;
}

int pymfb_enqueue(pymfb_ctx* c, int niter, unsigned flags) {
    CK(check_ready(c));
    if (niter < 0) return fail("niter < 0");
    if (flags & PYMFB_EARLY_STOP) return fail("pymfb_enqueue does not support PYMFB_EARLY_STOP (use pymfb_run)");
    if ((flags & PYMFB_COMPUTE_ERR) && niter > c->ferr_cap) {
        CU(cudaSetDevice(c->device));
        if (c->ferr_dev) CU(cudaFree(c->ferr_dev));
        graph_drop(c); c->graph_key = 0;       // the graph holds the old ferr pointer
        c->ferr_cap = std::max(niter, 1024);
        CU(cudaMalloc(&c->ferr_dev, sizeof(double) * c->ferr_cap));
    }
    return enqueue_iterations(c, niter, flags);
}
int pymfb_sync(pymfb_ctx* c) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
}
void* pymfb_stream(pymfb_ctx* c) { return c ? (void*)c->stream : nullptr; }

int pymfb_event_create(void** ev) {
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    *ev = (void*)e;
    return 0;
}
int pymfb_event_record(pymfb_ctx* c, void* ev) {
    if (!c) return fail("null context");
    CU(cudaEventRecord((cudaEvent_t)ev, c->stream));
    return 0;
}
int pymfb_event_elapsed_ms(void* a, void* b, float* ms) {
    CU(cudaEventSynchronize((cudaEvent_t)b));
    CU(cudaEventElapsedTime(ms, (cudaEvent_t)a, (cudaEvent_t)b));
    return 0;
}
int pymfb_event_destroy(void* ev) { CU(cudaEventDestroy((cudaEvent_t)ev)); return 0; }

int pymfb_kernel_timing(pymfb_ctx* c, int enable) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    for (int w = 0; w < 2; ++w) {
        for (auto& p : c->ev[w]) { cudaEventDestroy(p.first); cudaEventDestroy(p.second); }
        c->ev[w].clear();
    }
    c->timing = enable != 0;
    return 0;
}
int pymfb_kernel_timing_read(pymfb_ctx* c, int which, double* avg_ms, int64_t* launches) {
    if (!c) return fail("null context");
    if (which < 0 || which > 1) return fail("which must be 0 or 1");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    double tot = 0.0;
    for (auto& p : c->ev[which]) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, p.first, p.second));
        tot += ms;
    }
    const int64_t n = (int64_t)c->ev[which].size();
    if (avg_ms) *avg_ms = n ? tot / n : 0.0;
    if (launches) *launches = n;
    return 0;
}

int64_t pymfb_launch_count(pymfb_ctx* c) { return c ? c->launches : 0; }
int64_t pymfb_graph_replays(pymfb_ctx* c) { return c ? c->graph_replays : 0; }
int pymfb_active_path(pymfb_ctx* c) { return c ? c->path : 0; }

int pymfb_flush_l2(pymfb_ctx* c) {
    if (!c) return fail("null context");
    CU(cudaSetDevice(c->device));
    if (!c->flush_buf) {
        c->flush_bytes = 256u << 20;   // > 126 MB L2
        CU(cudaMalloc(&c->flush_buf, c->flush_bytes));
    }
    k_fill<<<8 * c->sm_count, 256, 0, c->stream>>>(c->flush_buf, (int64_t)(c->flush_bytes / sizeof(float)), 1.0f);
    c->launches += 1;
    CU(cudaGetLastError());
    return 0;
}

}  // extern "C"
