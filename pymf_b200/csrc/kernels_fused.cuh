// kernels_fused.cuh - ONE persistent kernel per iteration: H update + X H^T + H H^T with X read from
// HBM once and re-read from L2 (k <= 32 path).
//
// Ownership.  The rows of X are cut into slabs of F_SLAB = 256 rows; CTA (g, r) of the grid owns slab r
// for the whole launch, and the nslab CTAs of group g work on the SAME 128-column tile at the same time
// (tiles g, g + NG, g + 2 NG, ...; NG = #SMs / nslab groups).  Per tile every CTA runs two tasks:
//
//   A(t)  C_part = X[slab, tile]^T [W_hi|W_lo][slab]      8 stages of 32 rows, first read of X (HBM,
//         L2 evict_last); the epilogue warps add the partial into the tile's L2-resident accumulator
//         (coalesced fp32 REDs) and hand the tile to a PUBLISHER warp, which fences (cumulative over the
//         epilogue's REDs, PTX causality order) and bumps the tile's arrival counter.  The CTA whose
//         partial arrives LAST queues the tile for its UPDATE warps: Hn = H * C / (G H + 1e-9)
//         (H / (G H + 1e-9) precomputed by k_gh_ratio), Hn and its chunk-major [hi ; lo] split are published
//         and the tile's done flag is released.
//   B(t)  acc[slab rows] += X[slab, tile] [Hn_hi;Hn_lo]^T  2 row blocks x 4 stages of 32 columns, second
//         read of the SAME bytes by the SAME SM a few microseconds later (L2 hit, evict_first); the
//         128 epilogue threads keep the slab's 256 x k result in registers for the whole launch and
//         flush it to P with one atomic per element at the end.
//   HH(t) Hn Hn^T for the tile, by the CTA whose slab index equals the tile's sequence number mod nslab.
//
// Each CTA streams  A(0) .. A(D-1) | B(0) A(D) | B(1) A(D+1) | ...  (D = depth, default 3) through ONE
// TMA -> convert -> MMA ring, so B(t) normally finds its flag already set and the L2 window is about
// (D + 1) tasks x 128 KB x #CTAs (~40 MB at D = 2) instead of the hundreds of MB the first version of
// this kernel needed (task lists interleaved over the whole grid; see DESIGN.md 5.4).
//
// Warp roles: 2 TMA producers | F_NMMA MMA issuers (alternate segments) | 8 convert warps (two groups, alternate stages) |
// 4 epilogue warps (TMEM -> registers -> REDs) | 2 publisher warps (fence + arrival counter, alternate
// A tasks; the fence / atomic round trip costs microseconds under load and must not block the
// epilogue) | 4 update warps (one team: the H update of tiles whose last partial arrived here).
#pragma once
#include "kernels_tc.cuh"

namespace pymfb {
namespace tc {

constexpr int F_KP = 32;
constexpr int F_SLAB = 256;                          // rows of X owned by one CTA
constexpr int F_ASTAGES = F_SLAB / R1;               // 8 stages (32 rows each) per A task
constexpr int F_BSEG = TILE_COLS / 32;               // 4 stages (32 columns each) per row block of a B task
constexpr int F_NPROD = 2;                           // TMA producer warps
constexpr int F_CONV_GROUPS = 2;
constexpr int F_NPUB = 2;                            // publisher warps
constexpr int F_NMMA = 1;                            // MMA issuer warps (alternate accumulation segments).  One warp spends
                                                     // ~40 issue cycles per tcgen05.mma (329 cycles for the 8 MMAs + 2 commits
                                                     // of a stage whose tensor time is 192), but 2 warps measured no faster:
                                                     // the 7-slot ring (stage lifetime ~4300 cycles) is the tighter bound
constexpr int F_WARPS = F_NPROD + F_NMMA + 4 * F_CONV_GROUPS + 4 + F_NPUB + 4;
constexpr int F_THREADS = 32 * F_WARPS;
constexpr int F_CONV_WARP0 = F_NPROD + F_NMMA;
constexpr int F_EPI_WARP0 = F_CONV_WARP0 + 4 * F_CONV_GROUPS;
constexpr int F_PUB_WARP0 = F_EPI_WARP0 + 4;
constexpr int F_UPD_WARP0 = F_PUB_WARP0 + F_NPUB;
constexpr int F_RING = 4;                            // publisher -> update-team queue entries
constexpr int F_STAGES = 7;                          // TMA ring depth (24 KB stages); the rest of shared memory holds
                                                     // the slab's X Hn^T accumulators
static_assert(TsCfg<F_KP>::NT % F_CONV_GROUPS == 0, "an A-ring slot must always belong to the same convert group");
constexpr int F_PACC_FLOATS = 2 * F_KP * 128;        // [row block][k][row]: 256 rows x k, fp32, owned by the epilogue threads
constexpr int F_PHH_FLOATS = F_KP * F_KP;            // [k][row < k] of Hn Hn^T

struct FusedParams {
    const DevState* st;
    const float* Hc;        // old H (kp x ldh)
    float* Hn;              // new H
    float* Hs;              // chunk-major [Hn_hi ; Hn_lo] (hs_index)
    const float* Rg;        // H / (G H + 1e-9) of the OLD H (kp x ldh), from k_gh_ratio
    float* PA;              // d x kp   (+= X Hn^T)
    float* PB;              // kp x kp  (+= Hn Hn^T)
    float* PartA;           // deterministic flush: ngroups copies of A (d x kp each), copy g written by the CTAs of group g; null = atomics
    float* PartB;           // gridDim.x copies of B (kp x kp), one per CTA
    float* Cpart;           // [ngroups][nslot][kp][128] fp32 accumulators of the slab partials (zero between uses)
    int* tile_cnt;          // [n_tiles] slabs arrived
    int* tile_done;         // [n_tiles] 1 once Hn / Hs of the tile are visible
    int64_t ldh;
    int d, n_loc, n_tiles;
    int nslab, ngroups, depth, nslot, hint;
    int xsh;                // log2 of the panel width of X (tma_load_x)
    int pf;                 // L2 prefetch distance of the A tasks in tiles of this group (0 = off)
    const float* wmean;     // centered W (kernels_tc.cuh "centering"): column means of W and column sums of X, else null
    const float* xsum;
    int* fault;             // mapped host memory: the watchdogs note which wait timed out before they trap
    float* dbg;             // PYMFB_TRACE builds: event log
};

// PYMFB_TRACE (experiment builds): CTA `FTRACE_CTA` appends (code, value, clock) events to dbg + 2 MB.
#if defined(PYMFB_TRACE)
#ifndef FTRACE_CTA
#define FTRACE_CTA 0
#endif
#define FTRACE(code, val)                                                                                 \
    do {                                                                                                  \
        if (p.dbg != nullptr && blockIdx.x == FTRACE_CTA && lane == 0) {                                  \
            unsigned long long* ev_ = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(p.dbg) + (2 << 20)); \
            const unsigned long long i_ = atomicAdd(ev_, 1ull);                                           \
            if (i_ < 87000ull) { ev_[1 + 3 * i_] = (code); ev_[2 + 3 * i_] = (unsigned long long)(val); ev_[3 + 3 * i_] = clock64(); } \
        }                                                                                                 \
    } while (0)
#else
#define FTRACE(code, val) do { } while (0)
#endif

struct FTask {
    int type;      // 0 = A, 1 = B, 2 = HH
    int tile;
    int seq;       // index of the tile in this group's sequence
};

// The task sequence of CTA (g, r); every warp role walks it independently.
struct FSeq {
    int g, r, n_my, depth, ngroups, nslab;
    int i, phase;
    __device__ __forceinline__ void init(const FusedParams& p, int cta) {
        g = cta / p.nslab; r = cta % p.nslab;
        ngroups = p.ngroups; nslab = p.nslab; depth = p.depth;
        n_my = g < p.n_tiles ? (p.n_tiles - g + ngroups - 1) / ngroups : 0;
        i = 0; phase = 0;
    }
    __device__ __forceinline__ bool next(FTask& t) {
        while (i < n_my + depth) {
            const int sq = i - depth;
            if (phase == 0) {
                phase = 1;
                if (sq >= 0) { t.type = 1; t.seq = sq; t.tile = g + sq * ngroups; return true; }
            }
            if (phase == 1) {
                phase = 2;
                if (sq >= 0 && (sq % nslab) == r) { t.type = 2; t.seq = sq; t.tile = g + sq * ngroups; return true; }
            }
            phase = 0;
            const int ii = i++;
            if (ii < n_my) { t.type = 0; t.seq = ii; t.tile = g + ii * ngroups; return true; }
        }
        return false;
    }
};
__device__ __forceinline__ int f_stages(int type) { return type == 0 ? F_ASTAGES : (type == 1 ? 2 * F_BSEG : F_BSEG); }
// An A task drains W^T X after every stage (32 rows): the truncating C chain stays 4 MMAs long against the
// round-to-nearest G H of k_gh_ratio, which keeps the scale drift of DESIGN 5.1 ("Segments") small.  With 2-stage
// segments (8 MMAs) the 200-iteration trajectory at 256 x 65664, k = 32 ended 1.13e-4 from the oracle.
constexpr int F_ASEG = 1;
__device__ __forceinline__ int f_segs(int type) { return type == 0 ? F_ASTAGES / F_ASEG : (type == 1 ? 2 : 1); }
__device__ __forceinline__ int f_seglen(int type) { return type == 0 ? F_ASEG : F_BSEG; }

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __noinline__ void f_watchdog(int* fault, int code, int aux) {
    if (fault != nullptr && (threadIdx.x & 31) == 0) {            // plain stores: atomics on mapped host memory fault
        volatile int* f = fault;
        if (f[0] == 0) { f[1] = (int)blockIdx.x; f[2] = aux; f[3] = (int)threadIdx.x; f[0] = code; }
        __threadfence_system();
    }
    __nanosleep(1000000);
    __trap();
}
constexpr long long F_WATCHDOG_CYCLES = 2000000000LL;     // ~1 s
__device__ __forceinline__ void spin_until_ge(const int* p, int want, int* fault, int code, int aux) {
    if (ld_acquire_gpu(p) >= want) return;
    const long long t0 = clock64();
    while (ld_acquire_gpu(p) < want) {
        __nanosleep(40);
        if (clock64() - t0 > F_WATCHDOG_CYCLES) f_watchdog(fault, code, aux);
    }
}
// mbarrier wait with a watchdog note (code identifies the wait, aux the task / stage)
__device__ __forceinline__ void mbar_wait_f(uint32_t bar, uint32_t parity, int* fault, int code, int aux) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > F_WATCHDOG_CYCLES) f_watchdog(fault, code, aux);
    }
}
// L2 prefetch with an eviction-priority hint (the hinted loads are in kernels_tc.cuh)
__device__ __forceinline__ void tma_prefetch_2d_hint(const CUtensorMap* map, int c0, int c1, uint64_t policy);
__device__ __forceinline__ void tma_prefetch_x_hint(const CUtensorMap* map, int col, int row, int xsh, uint64_t policy) {
    if (xsh == kNoPanel) { tma_prefetch_2d_hint(map, col, row, policy); return; }
    const int pn = col >> xsh;
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.L2::cache_hint [%0, {%1, %2, %3}], %4;" ::"l"(map), "r"(col - (pn << xsh)), "r"(row), "r"(pn), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_prefetch_2d_hint(const CUtensorMap* map, int c0, int c1, uint64_t policy) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.L2::cache_hint [%0, {%1, %2}], %3;" ::"l"(map), "r"(c0), "r"(c1), "l"(policy) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
// 16 values -> hi at column c0.., lo at column 32 + c0.. of an A-ring slot
__device__ __forceinline__ void park_hilo16(uint32_t slot_addr, int c0, const float (&v)[16]) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        hi[i] = __float_as_uint(v[i]) & 0xFFFFE000u;
        lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
    }
    tmem_st16(slot_addr + c0, hi);
    tmem_st16(slot_addr + 32 + c0, lo);
}

// Rg = H / (G H + 1e-9): the factor that multiplies W^T X in the H update (pymf/nmf.py:124-126), G H in exact
// fp32 FMA; one thread per column.  Precomputed so that the update on the fused kernel's critical path is one
// batch of loads and a multiply.
__global__ void __launch_bounds__(128)
k_gh_ratio(const DevState* __restrict__ st, const float* __restrict__ G, const float* __restrict__ H, int64_t ldh,
           int n_loc, float* __restrict__ Rg) {
    constexpr int KP = F_KP;
    if (st->stop) return;
    __shared__ float Gs[KP * KP];
    for (int i = threadIdx.x; i < KP * KP; i += blockDim.x) Gs[i] = G[i];
    __syncthreads();
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= n_loc) return;
    float h[KP];
#pragma unroll
    for (int l = 0; l < KP; ++l) h[l] = __ldg(H + (int64_t)l * ldh + col);
#pragma unroll 4
    for (int j = 0; j < KP; ++j) {
        float dj = 0.f;
#pragma unroll
        for (int l = 0; l < KP; ++l) dj = fmaf(Gs[j * KP + l], h[l], dj);
        Rg[(int64_t)j * ldh + col] = h[j] / (dj + kEpsDenom);
    }
}

__global__ void __launch_bounds__(F_THREADS, 1)
k_fused_ts(const __grid_constant__ CUtensorMap mapXp,   // X, plain boxes 128 cols x 32 rows   (A tasks)
           const __grid_constant__ CUtensorMap mapW,    // [W_hi|W_lo], MN-major chunks        (A tasks)
           const __grid_constant__ CUtensorMap mapXx,   // X, SW128 boxes 32 cols x 128 rows   (B tasks)
           const __grid_constant__ CUtensorMap mapHs,   // [Hn_hi;Hn_lo] chunks, SW128 32 x 2kp (B / HH tasks)
           const __grid_constant__ CUtensorMap mapHa,   // Hn as the A operand of H H^T        (HH tasks)
           const FusedParams p) {
    constexpr int KP = F_KP;
    using Cfg = TsCfg<KP>;
    if (p.st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    static_assert(Cfg::NCHAIN == 1, "the fused kernel uses one accumulation chain per segment");
    // smem: ring | X Hn^T accumulators | Hn Hn^T accumulators | barriers | queues
    constexpr int RING = F_STAGES * Cfg::STAGE_BYTES;
    constexpr int PACC_OFF = RING;
    constexpr int PHH_OFF = PACC_OFF + F_PACC_FLOATS * 4;
    constexpr int BAR_OFF = PHH_OFF + F_PHH_FLOATS * 4;
    const uint32_t bar_base = smem_base + BAR_OFF;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (F_STAGES + s); };
    // afull is per (MMA warp, A slot): a stage's convert warps arrive on the barrier of the MMA warp that owns the
    // stage's segment, so each MMA warp waits on consecutive phases of its own barriers only (a parity wait that
    // skipped a phase - or fell two behind - would alias)
    auto afull_bar = [&](int mw, int t) { return bar_base + 8u * (2 * F_STAGES + mw * Cfg::NT + t); };
    auto aempty_bar = [&](int t) { return bar_base + 8u * (2 * F_STAGES + F_NMMA * Cfg::NT + t); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * F_STAGES + (F_NMMA + 1) * Cfg::NT + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * F_STAGES + (F_NMMA + 1) * Cfg::NT + 2 + a); };
    constexpr int NB0 = 2 * F_STAGES + (F_NMMA + 1) * Cfg::NT + 4;
    auto pubfull_bar = [&](int w) { return bar_base + 8u * (NB0 + w); };              // epilogue -> publisher w
    auto pubempty_bar = [&](int w) { return bar_base + 8u * (NB0 + F_NPUB + w); };    // publisher w read its tile
    constexpr int NBAR = NB0 + 2 * F_NPUB;
    const uint32_t tmem_slot = bar_base + 8u * NBAR;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + BAR_OFF + 8 * NBAR);
    volatile int* qv = reinterpret_cast<volatile int*>(smem_gen + BAR_OFF + 8 * NBAR + 16);
    volatile int* pub_tile = qv;                         // [F_NPUB] tile handed to publisher w
    volatile int* ring_tile = qv + F_NPUB;               // [F_RING] tiles waiting for the update team
    volatile int* ring_valid = qv + F_NPUB + F_RING;     // [F_RING]
    int* ring_tail = const_cast<int*>(qv) + F_NPUB + 2 * F_RING;          // tickets handed out
    volatile int* pub_exited = qv + F_NPUB + 2 * F_RING + 1;
    float* pacc = reinterpret_cast<float*>(smem_gen + PACC_OFF);
    float* phh = reinterpret_cast<float*>(smem_gen + PHH_OFF);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#if defined(PYMFB_TRACE)
    float* dbg = p.dbg;                                  // per-stage timeline (TRACE_AT, kernels_tc.cuh)
#endif
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapXp); tma_prefetch_desc(&mapW); tma_prefetch_desc(&mapXx); tma_prefetch_desc(&mapHs); tma_prefetch_desc(&mapHa);
        for (int s = 0; s < F_STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int t = 0; t < Cfg::NT; ++t) {
            for (int m = 0; m < F_NMMA; ++m) mbar_init(afull_bar(m, t), 4);
            mbar_init(aempty_bar(t), 1);
        }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
        for (int w = 0; w < F_NPUB; ++w) { mbar_init(pubfull_bar(w), 4); mbar_init(pubempty_bar(w), 1); }
        for (int i = 0; i < F_RING; ++i) { ring_tile[i] = 0; ring_valid[i] = 0; }
        *ring_tail = 0; *pub_exited = 0;
        fence_barrier_init();
    }
    if (warp == F_NPROD) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    auto xs_addr = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };
    auto bop = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + XSTAGE_BYTES; };
    FSeq seq;
    seq.init(p, blockIdx.x);
    const int row_slab = seq.r * F_SLAB;
    FTask t;

    if (warp < F_NPROD) {
        // ===== TMA producers (stage pcnt % F_NPROD == warp) =====
        uint32_t pcnt = 0;
        const uint64_t pol_keep = l2_policy_evict_last(), pol_drop = l2_policy_evict_first();
        while (seq.next(t)) {
            if (t.type != 0) {
                if (warp == 0) FTRACE(10 + t.type, t.tile);
                spin_until_ge(p.tile_done + t.tile, 1, p.fault, 1, t.tile);      // Hn / Hs of the tile are final
                fence_proxy_async_all();                     // generic-proxy stores of another CTA -> our TMA reads
                if (warp == 0) FTRACE(13, t.tile);
            } else if (warp == 0) FTRACE(10, t.tile);
            const int nst = f_stages(t.type);
            const int col0 = t.tile * TILE_COLS;
            for (int it = 0; it < nst; ++it, ++pcnt) {
                if (pcnt % F_NPROD != (uint32_t)warp) continue;
                const int s = (int)(pcnt % F_STAGES);
                const uint32_t ph = (pcnt / F_STAGES) & 1u;
                TRACE_AT(pcnt, 0);
#if defined(PYMFB_TRACE)
                if (dbg != nullptr && blockIdx.x == 0 && lane == 0 && pcnt < (uint32_t)TRACE_STAGES) reinterpret_cast<long long*>(dbg + (1 << 18))[(size_t)pcnt * 16 + 13] = 1 + t.type;
#endif
                mbar_wait_f(empty_bar(s), ph ^ 1, p.fault, 2, t.tile * 4 + t.type);
                TRACE_AT(pcnt, 1);
                if (elect_one()) {
                    mbar_expect_tx(full_bar(s), XSTAGE_BYTES + Cfg::BSTAGE_BYTES);
                    if (t.type == 0) {
                        const int r0 = row_slab + it * R1;
                        if (p.pf && t.tile + p.pf * p.ngroups < p.n_tiles)     // the same rows of the A task `pf` tiles ahead -> L2
                            tma_prefetch_x_hint(&mapXp, (t.tile + p.pf * p.ngroups) * TILE_COLS, r0, p.xsh, pol_keep);
                        if (p.hint) tma_load_x_hint(xs_addr(s), &mapXp, full_bar(s), col0, r0, p.xsh, pol_keep);
                        else tma_load_x(xs_addr(s), &mapXp, full_bar(s), col0, r0, p.xsh);
                        tma_load_2d(bop(s), &mapW, full_bar(s), 0, r0);
                        tma_load_2d(bop(s) + R1 * 128, &mapW, full_bar(s), 32, r0);
                    } else {
                        const int ch = it % F_BSEG;
                        const int c0 = col0 + 32 * ch;
                        if (t.type == 1) {
                            const int r0 = row_slab + (it / F_BSEG) * 128;
                            if (p.hint) tma_load_x_hint(xs_addr(s), &mapXx, full_bar(s), c0, r0, p.xsh, pol_drop);
                            else tma_load_x(xs_addr(s), &mapXx, full_bar(s), c0, r0, p.xsh);
                        } else {
                            tma_load_x(xs_addr(s), &mapHa, full_bar(s), c0, 0, kNoPanel);
                        }
                        tma_load_2d(bop(s), &mapHs, full_bar(s), 0, (c0 >> 5) * (2 * KP));
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp < F_CONV_WARP0) {
        // ===== MMA issuers: warp mw issues the segments g with g % F_NMMA == mw (segment g accumulates into
        // TMEM buffer g & 1, so the two warps never share an accumulator; tcgen05.commit tracks the MMAs of
        // the issuing thread, which is exactly the stage / segment that thread owns) =====
        constexpr uint32_t idA_hl = make_idesc(128, 2 * KP, 0, 1), idA_h = make_idesc(128, KP, 0, 1);
        constexpr uint32_t idB_hl = make_idesc(128, 2 * KP, 0, 0), idB_h = make_idesc(128, KP, 0, 0);
        const uint32_t mw = (uint32_t)(warp - F_NPROD);
        uint32_t c = 0, g = 0, apar = 0;                    // apar: phase parity of this warp's afull barriers, one bit per slot
        while (seq.next(t)) {
            const int nseg = f_segs(t.type), seglen = f_seglen(t.type);
            for (int sg = 0; sg < nseg; ++sg, ++g) {
                if (g % F_NMMA != mw) { c += (uint32_t)seglen; continue; }
                const uint32_t b = g & 1u;
                mbar_wait_f(tempty_bar(b), ((g >> 1) & 1u) ^ 1u, p.fault, 3, t.tile * 4 + t.type);
                tc_fence_after();
                const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                for (int it = 0; it < seglen; ++it, ++c) {
                    const int s = (int)(c % F_STAGES), ts = (int)(c % Cfg::NT);
                    // afull implies full: the convert warps waited for the stage's TMA transaction (X and the
                    // [b_hi|b_lo] operand share it) before they arrived here
#if defined(FUSED_MMA_WAIT_FULL)
                    mbar_wait_f(full_bar(s), (c / F_STAGES) & 1u, p.fault, 4, t.tile * 4 + t.type);
#endif
                    TRACE_AT(c, 5);
                    mbar_wait_f(afull_bar((int)mw, ts), (apar >> ts) & 1u, p.fault, 5, t.tile * 4 + t.type);
                    apar ^= 1u << ts;
                    TRACE_AT(c, 6);
                    tc_fence_after();
                    const uint32_t a_hi = tmem_base + Cfg::A_COL0 + ts * 64;
                    if (elect_one()) {
                        if (t.type == 0) {
#pragma unroll
                            for (int kg = 0; kg < 4; ++kg) {
                                const uint64_t bd = make_desc(bop(s) + kg * 1024, R1 * 128, 512, 1);
                                umma_tf32_ts(dcol, a_hi + kg * 8, bd, idA_hl, (it == 0 && kg == 0) ? 0u : 1u);
                                umma_tf32_ts(dcol + KP, a_hi + 32 + kg * 8, bd, idA_h, 1u);
                            }
                        } else {
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                const uint64_t bd = make_desc(bop(s) + ks * 32, 16, 1024);
                                umma_tf32_ts(dcol, a_hi + ks * 8, bd, idB_hl, (it == 0 && ks == 0) ? 0u : 1u);
                                umma_tf32_ts(dcol + KP, a_hi + 32 + ks * 8, bd, idB_h, 1u);
                            }
                        }
                        umma_commit(empty_bar(s));
                        umma_commit(aempty_bar(ts));
                    }
                    __syncwarp();
                    TRACE_AT(c, 7);
                }
                if (elect_one()) umma_commit(tfull_bar(b));
                __syncwarp();
            }
            if (mw == 0) FTRACE(20 + t.type, t.tile);
        }
    } else if (warp < F_EPI_WARP0) {
        // ===== convert warps: smem tile -> registers -> hi/lo -> TMEM A ring =====
        const int q = warp & 3;
        const int group = (warp - F_CONV_WARP0) >> 2;
        const int mylane = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::A_COL0;
        uint32_t c = 0, g = 0;
        while (seq.next(t)) {
            const int nst = f_stages(t.type), seglen = f_seglen(t.type);
            for (int it = 0; it < nst; ++it, ++c) {
                const int owner = (int)((g + (uint32_t)(it / seglen)) % F_NMMA);      // MMA warp of this stage's segment
                if (it == nst - 1) g += (uint32_t)f_segs(t.type);
                if ((int)(c % F_CONV_GROUPS) != group) continue;
                const int s = (int)(c % F_STAGES), ts = (int)(c % Cfg::NT);
                // ORDER MATTERS.  F_STAGES is odd and the two convert groups take alternate stages, so a group sees
                // only every other phase of a stage's full barrier; a parity wait two phases ahead would pass on
                // the stale phase if the stage in between (the other group's) had not landed yet.  The A-slot
                // barrier (NT is even: always the same group, consecutive phases) is therefore taken first: it
                // opens only after the MMA consumed stage c - NT, i.e. after every earlier stage has landed.
                if (q == 0) TRACE_AT(c, 2);
                mbar_wait_f(aempty_bar(ts), ((c / Cfg::NT) & 1u) ^ 1u, p.fault, 7, t.tile * 4 + t.type);
                if (q == 0) TRACE_AT(c, 9);
                mbar_wait_f(full_bar(s), (c / F_STAGES) & 1u, p.fault, 6, t.tile * 4 + t.type);
                if (q == 0) TRACE_AT(c, 3);
                tc_fence_after();
                const uint8_t* stage = smem_gen + s * Cfg::STAGE_BYTES;
                const uint32_t slot = lane_addr + ts * 64;
                if (t.type == 0) {
                    // plain [32 rows][128 cols]: lane = column, TMEM column = row
                    const float* xs = reinterpret_cast<const float*>(stage);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        float v[16];
#pragma unroll
                        for (int r = 0; r < 16; ++r) v[r] = xs[(h * 16 + r) * TILE_COLS + mylane];
                        park_hilo16(slot, h * 16, v);
                    }
                } else {
                    // SW128 [128 rows][128 B]: lane = row, 16 B chunk j at (j ^ (row & 7))
                    const uint8_t* rowp = stage + mylane * 128;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        float v[16];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float4 f = *reinterpret_cast<const float4*>(rowp + (((h * 4 + j) ^ (mylane & 7)) << 4));
                            v[4 * j + 0] = f.x; v[4 * j + 1] = f.y; v[4 * j + 2] = f.z; v[4 * j + 3] = f.w;
                        }
                        park_hilo16(slot, h * 16, v);
                    }
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(c, 4);
                if (lane == 0) mbar_arrive(afull_bar(owner, ts));
            }
        }
    } else if (warp < F_PUB_WARP0) {
        // ===== epilogue warps: drain segments; A -> staging for the update warps; B / HH -> registers =====
        const int q = warp & 3;
        const int et = q * 32 + lane;                            // TMEM lane of this thread (= column / row of the tile)
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0, uq = 0;
        // thread et owns rows et and 128 + et of the slab (and row et of Hn Hn^T when et < k)
        for (int j = 0; j < 2 * KP; ++j) pacc[j * 128 + et] = 0.f;
        if (et < KP) for (int j = 0; j < KP; ++j) phh[j * KP + et] = 0.f;
        while (seq.next(t)) {
            const int nseg = f_segs(t.type);
#pragma unroll 1
            for (int sg = 0; sg < nseg; ++sg, ++g) {
                const uint32_t b = g & 1u;
                mbar_wait_f(tfull_bar(b), (g >> 1) & 1u, p.fault, 8, t.tile * 4 + t.type);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
                float v[KP];
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
                    float hi[16], sm[16];
                    tmem_ld16(taddr + j0, hi);
                    tmem_ld16(taddr + KP + j0, sm);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j0 + j] = hi[j] + sm[j];
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(b));
                if (q == 0) FTRACE(30 + t.type, t.tile);
                if (t.type == 0) {
                    // each segment's partial C -> the tile's accumulator [k][128 columns] (lane = column: coalesced
                    // REDs); the tile is published after the slab's last segment
                    float* cp = p.Cpart + ((size_t)(seq.g * p.nslot + t.seq % p.nslot) * KP) * TILE_COLS + et;
#pragma unroll
                    for (int j = 0; j < KP; ++j) atomicAdd(cp + j * TILE_COLS, v[j]);
                    if (sg + 1 < nseg) continue;
                    const uint32_t w = uq % F_NPUB;
                    mbar_wait_f(pubempty_bar(w), ((uq / F_NPUB) & 1u) ^ 1u, p.fault, 9, t.tile);
                    if (et == 0) pub_tile[w] = t.tile;
                    __syncwarp();
                    if (lane == 0) mbar_arrive(pubfull_bar(w));          // release: our REDs precede the publisher's fence
                    if (q == 0) FTRACE(33, t.tile);
                    ++uq;
                } else if (t.type == 1) {
                    float* acc = pacc + sg * (KP * 128) + et;
#pragma unroll
                    for (int j = 0; j < KP; ++j) acc[j * 128] += v[j];
                } else if (et < KP) {
#pragma unroll
                    for (int j = 0; j < KP; ++j) phh[j * KP + et] += v[j];
                }
            }
        }
        for (int e = 0; e < F_NPUB; ++e, ++uq) {   // tell the publishers to exit
            const uint32_t w = uq % F_NPUB;
            mbar_wait_f(pubempty_bar(w), ((uq / F_NPUB) & 1u) ^ 1u, p.fault, 10, (int)uq);
            if (et == 0) pub_tile[w] = -1;
            __syncwarp();
            if (lane == 0) mbar_arrive(pubfull_bar(w));
        }
        // flush the slab's rows of X Hn^T (and this CTA's share of Hn Hn^T)
#pragma unroll 1
        for (int rb = 0; rb < 2; ++rb) {
            const int row = row_slab + rb * 128 + et;
            if (row < p.d) {
                const float* acc = pacc + rb * (KP * 128) + et;
                if (p.PartA != nullptr) {              // this group's copy of A: k_sum_copies adds the copies in group order
                    float* dst = p.PartA + (size_t)seq.g * p.d * KP + (int64_t)row * KP;
#pragma unroll
                    for (int j = 0; j < KP; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(acc[j * 128], acc[(j + 1) * 128], acc[(j + 2) * 128], acc[(j + 3) * 128]);
                } else {
                    float* dst = p.PA + (int64_t)row * KP;
#pragma unroll
                    for (int j = 0; j < KP; ++j) atomicAdd(dst + j, acc[j * 128]);
                }
            }
        }
        if (et < KP) {
            if (p.PartB != nullptr) {
                float* dst = p.PartB + (size_t)blockIdx.x * KP * KP + (int64_t)et * KP;
#pragma unroll
                for (int j = 0; j < KP; ++j) dst[j] = phh[j * KP + et];
            } else {
                float* dst = p.PB + (int64_t)et * KP;
#pragma unroll
                for (int j = 0; j < KP; ++j) atomicAdd(dst + j, phh[j * KP + et]);
            }
        }
    } else if (warp < F_UPD_WARP0) {
        // ===== publisher warps: fence (covers the epilogue warps' REDs: they happen-before through the
        // mbarrier), bump the tile's arrival counter; the last arrival queues the tile for the update team =====
        const int pw = warp - F_PUB_WARP0;
        for (uint32_t n = 0;; ++n) {
            mbar_wait_f(pubfull_bar(pw), n & 1u, p.fault, 11, (int)n);
            const int tile = pub_tile[pw];
            __syncwarp();
            if (lane == 0) mbar_arrive(pubempty_bar(pw));
            if (tile < 0) break;
            FTRACE(40, tile);
            __threadfence();
            FTRACE(41, tile);
            if (lane == 0) {
                const int old = atomicAdd(p.tile_cnt + tile, 1);
                FTRACE(42, tile * 64 + old);
                if (old == p.nslab - 1) {                              // (the update team fences before it reads the partials)
#if defined(FUSED_PUB_ACQ_FENCE)
                    __threadfence();
#endif
                    const int tk = atomicAdd(ring_tail, 1);
                    const int e = tk % F_RING;
                    while (ring_valid[e] != 0) __nanosleep(50);        // entry still unread (never in practice)
                    ring_tile[e] = tile;
                    __threadfence_block();
                    ring_valid[e] = 1;
                }
            }
            __syncwarp();
        }
        __threadfence_block();
        if (lane == 0) atomicAdd(const_cast<int*>(pub_exited), 1);
    } else {
        // ===== update warps (one team, thread = column of the tile): Hn = H * C / (G H + 1e-9) =====
        const int ut = threadIdx.x - 32 * F_UPD_WARP0;          // 0..127
        for (int head = 0;; ++head) {
            const int e = head % F_RING;
            int tile = -1;
            if (lane == 0) {
                const long long t0 = clock64();
                while (true) {
                    if (ring_valid[e] != 0) { tile = ring_tile[e]; break; }
                    if (*pub_exited == F_NPUB && *reinterpret_cast<volatile int*>(ring_tail) == head) break;
                    __nanosleep(20);
                    if (clock64() - t0 > 4 * F_WATCHDOG_CYCLES) f_watchdog(p.fault, 12, head);
                }
            }
            tile = __shfl_sync(0xffffffffu, tile, 0);
            named_bar_sync(2, 128);                              // every warp has read the entry
            if (tile < 0) break;
            if (ut == 0) ring_valid[e] = 0;
            if (ut == 0) FTRACE(50, tile);
            __threadfence();
            const int sq = (tile - seq.g) / seq.ngroups;
            float* cp = p.Cpart + ((size_t)(seq.g * p.nslot + sq % p.nslot) * KP) * TILE_COLS + ut;
            const int col = tile * TILE_COLS + ut;
            {
                float cs[KP], rg[KP];
                const bool live = col < p.n_loc;
#pragma unroll
                for (int j = 0; j < KP; ++j) cs[j] = __ldcg(cp + j * TILE_COLS);
#pragma unroll
                for (int j = 0; j < KP; ++j) rg[j] = live ? __ldg(p.Rg + (int64_t)j * p.ldh + col) : 0.f;
#pragma unroll
                for (int j = 0; j < KP; ++j) __stcg(cp + j * TILE_COLS, 0.f);                    // ready for tile seq + nslot
                if (live) {
                    const float xs = (p.wmean != nullptr) ? __ldg(p.xsum + col) : 0.f;
#pragma unroll
                    for (int j = 0; j < KP; ++j) {
                        const float cj = (p.wmean != nullptr) ? fmaf(__ldg(p.wmean + j), xs, cs[j]) : cs[j];
                        const float hn = rg[j] * cj;
                        const float hh = __uint_as_float(__float_as_uint(hn) & 0xFFFFE000u);
                        p.Hn[(int64_t)j * p.ldh + col] = hn;
                        p.Hs[hs_index(j, col, 2 * KP)] = hh;
                        p.Hs[hs_index(KP + j, col, 2 * KP)] = hn - hh;
                    }
                }
            }
            if (ut == 0) FTRACE(51, tile);
            __threadfence();
            fence_proxy_async_all();
            named_bar_sync(2, 128);
            if (ut == 0) st_release_gpu(p.tile_done + tile, 1);
            if (ut == 0) FTRACE(52, tile);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == F_NPROD) tmem_dealloc(tmem_base, 512);
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct FusedPlan {
    bool ready = false;
    float* Cpart = nullptr;
    float* Part = nullptr;       // deterministic flush: ngroups copies of A, then one copy of B per CTA
    bool zero_p = true;          // atomics flush: P must be cleared before the launch
    float* Rg = nullptr;         // kp x ldh
    int* cnt = nullptr;          // [n_tiles] arrival counters, [n_tiles] done flags
    int n_tiles = 0, nslab = 0, ngroups = 0, depth = 2, nslot = 4, hint = 1, pf = 1;
    int smem = 0;
};

inline void fused_release(FusedPlan& f) {
    if (f.Cpart) cudaFree(f.Cpart);
    if (f.Part) cudaFree(f.Part);
    f.Part = nullptr;
    if (f.Rg) cudaFree(f.Rg);
    if (f.cnt) cudaFree(f.cnt);
    f.Cpart = nullptr; f.Rg = nullptr; f.cnt = nullptr; f.ready = false;
}

// The one-pass kernel serves k <= 32 shapes whose row slabs fit the grid (d <= 256 x #SMs).  It is the DEFAULT where it
// wins: d <= 256, i.e. one row slab - a column tile is then owned by ONE CTA, nothing is reduced across CTAs, and the
// kernel beats the two passes (256 x 4M, k = 32: 2.49 vs 2.91 ms per iteration; at d = 512 they tie, above the two passes
// win, DESIGN.md 5.4).  PYMFB_FUSED=1 forces it for every eligible shape, =0 disables it; PYMFB_FUSED_DEPTH (default 3)
// and PYMFB_FUSED_HINT (default 1) tune it.
inline bool fused_wanted(const TcPlan& p) {
    if (!p.ready || !p.use_ts || p.kp != tc::F_KP) return false;
    const int nslab = (int)((p.d + tc::F_SLAB - 1) / tc::F_SLAB);
    if (nslab > p.sm_count) return false;
    const char* e = getenv("PYMFB_FUSED");
    if (e) return e[0] == '1';
    // smaller problems are launch-bound and replay the two-pass iteration as a CUDA graph, which wins there (256 x 65536: 0.121 vs 0.136 ms)
    return nslab == 1 && p.h_tiles >= 2 * p.sm_count && (double)p.d * (double)p.n_loc > 16777216.0;
}

inline int fused_plan(FusedPlan& f, const TcPlan& p) {
    fused_release(f);
    auto env_int = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
    f.n_tiles = p.h_tiles;
    f.nslab = (int)((p.d + tc::F_SLAB - 1) / tc::F_SLAB);
    f.ngroups = std::max(1, std::min(p.sm_count / f.nslab, f.n_tiles));
    f.depth = std::max(1, env_int("PYMFB_FUSED_DEPTH", 3));
    f.nslot = f.depth + 2;
    f.hint = env_int("PYMFB_FUSED_HINT", 1);
    f.pf = std::max(0, env_int("PYMFB_FUSED_PF", 1));
    const size_t cbytes = (size_t)f.ngroups * f.nslot * tc::F_KP * tc::TILE_COLS * sizeof(float);
    if (cudaMalloc(&f.Cpart, cbytes) != cudaSuccess) return 1;
    if (cudaMemset(f.Cpart, 0, cbytes) != cudaSuccess) return 1;
    if (cudaMalloc(&f.Rg, (size_t)p.kp * p.ldh * sizeof(float)) != cudaSuccess) return 1;
    if (cudaMalloc(&f.cnt, (size_t)2 * f.n_tiles * sizeof(int)) != cudaSuccess) return 1;
    {   // deterministic flush (bit-reproducible W, as on the two-pass kernels) while the copies stay small
        const size_t pbytes = ((size_t)f.ngroups * p.d * p.kp + (size_t)f.ngroups * f.nslab * p.kp * p.kp) * sizeof(float);
        const char* e = getenv("PYMFB_DETERMINISTIC");
        const bool want = e ? e[0] == '1' : pbytes <= ((size_t)1 << 30);
        if (want) { if (cudaMalloc(&f.Part, pbytes) != cudaSuccess) return 1; }
        f.zero_p = f.Part == nullptr;
    }
    using Cfg = tc::TsCfg<tc::F_KP>;
    f.smem = tc::F_STAGES * Cfg::STAGE_BYTES + (tc::F_PACC_FLOATS + tc::F_PHH_FLOATS) * 4 +
             1024 /*barriers, queue*/ + 1024 /*align*/;
    if (f.smem > tc::SMEM_LIMIT) return 1;
    if (cudaFuncSetAttribute(tc::k_fused_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, f.smem) != cudaSuccess) return 1;
    f.ready = true;
    return 0;
}

// H[hsrc] -> H[hsrc^1] (and its [hi;lo] companion), P += [X Hn^T | Hn Hn^T].  P must be zero on entry.
inline int fused_launch(FusedPlan& f, TcPlan& p, const DevState* st, const float* Hc, float* Hn, const float* G, float* P,
                        cudaStream_t stream, int64_t* launches, int* fault) {
    const int hsrc = (Hc == p.Hbuf[0]) ? 0 : 1, hdst = hsrc ^ 1;
    if (cudaMemsetAsync(f.cnt, 0, (size_t)2 * f.n_tiles * sizeof(int), stream) != cudaSuccess) return 1;
    tc::k_gh_ratio<<<(unsigned)((p.n_loc + 127) / 128), 128, 0, stream>>>(st, G, Hc, p.ldh, (int)p.n_loc, f.Rg);
    tc::FusedParams fp;
    fp.st = st; fp.Hc = Hc; fp.Hn = Hn; fp.Hs = p.Hs[hdst]; fp.Rg = f.Rg; fp.PA = P; fp.PB = P + p.d * p.kp;
    fp.PartA = f.Part; fp.PartB = f.Part ? f.Part + (size_t)f.ngroups * p.d * p.kp : nullptr;
    fp.Cpart = f.Cpart; fp.tile_cnt = f.cnt; fp.tile_done = f.cnt + f.n_tiles;
    fp.ldh = p.ldh; fp.d = (int)p.d; fp.n_loc = (int)p.n_loc; fp.n_tiles = f.n_tiles;
    fp.nslab = f.nslab; fp.ngroups = f.ngroups; fp.depth = f.depth; fp.nslot = f.nslot; fp.hint = f.hint;
    fp.pf = f.pf; fp.xsh = p.xsh;
    fp.wmean = p.center ? p.wmean : nullptr; fp.xsum = p.xsum;
    fp.fault = fault;
    fp.dbg = p.dbg;
#if defined(PYMFB_TRACE)
    if (p.dbg) cudaMemsetAsync(reinterpret_cast<char*>(p.dbg) + (2 << 20), 0, 8, stream);   // event counter
#endif
    const int grid = f.ngroups * f.nslab;
    tc::k_fused_ts<<<grid, tc::F_THREADS, f.smem, stream>>>(p.mapX_p, p.mapW, p.mapX_x, p.mapH_x[hdst], p.mapH_a[hdst], fp);
    *launches += 2;
    if (f.Part) {                  // P = sum of the copies, in group / CTA order
        const int64_t na = p.d * p.kp, nb = (int64_t)p.kp * p.kp;
        tc::k_sum_copies<<<(unsigned)std::min<int64_t>(((na + nb) / 4 + 255) / 256, 8 * p.sm_count), 256, 0, stream>>>(
            st, fp.PartA, f.ngroups, na, P, fp.PartB, grid, nb, P + na);
        *launches += 1;
    }
    p.hs_valid[hdst] = true;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace pymfb
