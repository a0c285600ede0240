// kernels_tc.cuh - tcgen05 / TMEM / TMA kernels (sm_100a) of the two streaming passes.
//
//   k_h_update_tc : H <- H * (W^T X) / ((W^T W) H + 1e-9)        pymf/nmf.py:122-126
//   k_xht_tc      : P_A += X H^T  (feeds the W update, :128-132, and the error, :110)
//
// Arithmetic: fp32 storage, every product is a 3xTF32 split  a*b ~= a_hi*b_hi + a_hi*b_lo +
// a_lo*b_hi  (a_hi = a with the low 13 mantissa bits cleared, a_lo = a - a_hi, exact in fp32),
// accumulated in fp32 in TMEM.  The two a_hi terms are ONE MMA of width N = 2k against the
// concatenated operand [b_hi | b_lo]; the a_lo term is a second MMA of width k that accumulates
// into the "small terms" half, so every element of X crosses shared memory -> tensor core twice
// per pass instead of three times.  hi + small halves are added in the epilogue.
//
// Data movement: X (and H) tiles arrive by TMA (cp.async.bulk.tensor, 128B swizzle) into a
// multi-stage mbarrier ring; 4 "split" warps derive the lo tiles in shared memory; one thread
// issues tcgen05.mma; 4 epilogue warps read the accumulators with tcgen05.ld.  Persistent CTAs
// (one per SM) loop over column tiles / (row block, column range) tasks.
//
// Layout facts used below (sm_100 UMMA canonical layouts, fp32/tf32 elements, 128B swizzle):
//   MN-major operand: smem = [k rows][32 elements = 128 B], "128B swizzle with 32B atoms" (the only
//                     MN-major layout tf32 supports): 4 rows = one 512 B swizzle atom; SBO = byte
//                     stride between 4-row groups, LBO = byte stride between 32-element chunks
//                     along M/N.  One MMA (K = 8) consumes two 4-row groups.
//   K-major operand : smem = [m rows][32 elements along K = 128 B]; SBO = stride between 8-row
//                     groups (1024 B); one MMA consumes 32 B of each row (start address + 32 B).
//   Both are exactly what a TMA box of 32 fp32 x R rows writes (SWIZZLE_128B_ATOM_32B resp. SWIZZLE_128B).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <string>
#include <vector>
#include <cstdio>

#include "common.cuh"

#ifndef PYMFB_TC_RAW_HI
#define PYMFB_TC_RAW_HI 1   // 1: feed the raw fp32 tile as the hi operand - tcgen05.mma.kind::tf32 ignores the low 13
                            //    mantissa bits, bit-identical to the masked tile (tests/_rawhi_check.py) and 16 KB less
                            //    shared-memory traffic per stage: cfg3 49.99 -> 48.85 ms per iteration, same box;
                            //    0: write the masked hi tile back explicitly
#endif

namespace pymfb {
namespace tc {

constexpr int NPROD = 3;              // TMA producer warps (stages round-robin): ONE issuing thread sustains only
                                      // ~58 GB/s of TMA traffic (measured, tests/tc_probe l2bw), 4 reach 130-190 GB/s per SM
constexpr int R1 = 32;                // rows (contraction) per stage of the H-update pass
constexpr int TILE_COLS = 128;        // columns per tile = UMMA M of the H-update pass
constexpr int XSTAGE_BYTES = 128 * 32 * 4;   // 16 KB: 128 x 32 fp32 in either orientation
constexpr int SMEM_LIMIT = 227 * 1024;

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug traps (launch failure) instead of hanging the GPU.
__device__ __noinline__ void mbar_watchdog(long long t0) {
    if (clock64() - t0 > 8000000000LL) __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        // the watchdog (out of line) runs only every 256th retry: the retry loop itself stays a handful of
        // instructions, so a waiter reacts to the phase flip without a clock read + 64-bit compare in between
        if (((++spins) & 0xFFu) == 0u) mbar_watchdog(t0);
    }
}
// Wait of a warp that has slack (epilogue warps between segments, TMA producers behind a full ring): back off between
// polls instead of re-issuing try_wait back to back - fewer issue slots and less power for the warps on the critical path.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
#if defined(PYMFB_RELAXED_WAIT)
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    uint32_t spins = 0;
    while (!mbar_try_wait(bar, parity)) {
        __nanosleep(PYMFB_RELAXED_WAIT);
        if (((++spins) & 0xFFu) == 0u) mbar_watchdog(t0);
    }
#else
    mbar_wait(bar, parity);
#endif
}
// One elected lane of a CONVERGED warp.  The producer and MMA warps run their loops with all 32 lanes
// (warp-uniform control flow lets the compiler keep descriptors / addresses in uniform registers; a
// lane-0-only branch made every tcgen05.mma cost ~90 issue cycles) and elect one lane per issue.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void named_barrier(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// Box of the data matrix X (or of H through a one-panel map): X maps are 3-D (column inside the panel, row, panel),
// see "Layout of the data matrix" in common.cuh; xsh = log2(panel width), kNoPanel for a single panel.
constexpr int kNoPanel = 31;
__device__ __forceinline__ void tma_load_x(uint32_t dst, const CUtensorMap* map, uint32_t bar, int col, int row, int xsh) {
    if (xsh == kNoPanel) { tma_load_2d(dst, map, bar, col, row); return; }    // row-major matrices keep 2-D maps (make_map3)
    const int p = col >> xsh;
    tma_load_3d(dst, map, bar, col - (p << xsh), row, p);
}
// L2 prefetch of a box of X (no shared-memory destination, no barrier)
__device__ __forceinline__ void tma_prefetch_x(const CUtensorMap* map, int col, int row, int xsh) {
    if (xsh == kNoPanel) { asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(map), "r"(col), "r"(row) : "memory"); return; }
    const int p = col >> xsh;
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];" ::"l"(map), "r"(col - (p << xsh)), "r"(row), "r"(p) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// TMA loads with an L2 eviction-priority hint (createpolicy.fractional.L2::evict_*)
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_load_x_hint(uint32_t dst, const CUtensorMap* map, uint32_t bar, int col, int row, int xsh, uint64_t policy) {
    if (xsh == kNoPanel) { tma_load_2d_hint(dst, map, bar, col, row, policy); return; }
    const int pn = col >> xsh;
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(dst), "l"(map), "r"(bar), "r"(col - (pn << xsh)), "r"(row), "r"(pn), "l"(policy) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], tf32 inputs, fp32 accumulate, issued by one thread
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Same with both descriptors passed as 32-bit halves (see umma_tf32_ts_lh): the high halves are loop invariant.
__device__ __forceinline__ void umma_tf32_lh(uint32_t d_tmem, uint32_t ad_lo, uint32_t ad_hi, uint32_t bd_lo, uint32_t bd_hi,
                                             uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 ad, bd;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "mov.b64 ad, {%1, %2};\n\t"
        "mov.b64 bd, {%3, %4};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], ad, bd, %5, p;\n\t}"
        ::"r"(d_tmem), "r"(ad_lo), "r"(ad_hi), "r"(bd_lo), "r"(bd_hi), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once all previously issued MMAs of this thread have completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------------------------------------
// descriptors
// ---------------------------------------------------------------------------------------------
// shared-memory matrix descriptor, 128B swizzle (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [61,64) layout=2 (SW128)
// layout: 2 = SWIZZLE_128B (K-major operands), 1 = SWIZZLE_128B_BASE32B - the only layout the hardware
// accepts for MN-major tf32 operands (128 B rows whose four 32 B chunks are XOR-permuted by row % 4;
// TMA writes it with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; swizzle atom = 4 rows = 512 B).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = 2) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): c=F32 (1<<4), a=b=TF32 (2<<7, 2<<10),
// a_major bit 15, b_major bit 16 (1 = MN-major), N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// hi/lo split of a float4 (hi = low 13 mantissa bits cleared; lo = exact remainder)
__device__ __forceinline__ void split4(const float4 v, float4& hi, float4& lo) {
    hi.x = __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
    hi.y = __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
    hi.z = __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
    hi.w = __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
    lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
}
// split `nvec` float4 of a stage buffer: raw -> (hi in place unless RAW_HI) + lo buffer
// One element group at a time (load, split, store).  Issuing all eight loads of a thread before its first store
// (-DPYMFB_SPLIT_BATCHED: the split warps then no longer expose a shared-memory round trip per group) was measured
// SLOWER on the k = 128 kernels, cfg3 49.9 -> 51.8 ms per iteration on the same box: the bursts of loads compete
// with the MMA's operand reads for the shared-memory port, which is what bounds these kernels (DESIGN.md 5.1).
#ifndef PYMFB_SPLIT_UNROLL
#define PYMFB_SPLIT_UNROLL 4
#endif
__device__ __forceinline__ void split_buffer(float4* raw, float4* lo, int nvec, int tid, int nthreads) {
#if defined(PYMFB_EXP_SS_SKIP_SPLIT)
    return;
#endif
    constexpr int B = PYMFB_SPLIT_UNROLL;              // loads in flight per thread (8 = the whole share of a thread)
    for (int i0 = tid; i0 < nvec; i0 += B * nthreads) {
        float4 v[B];
#pragma unroll
        for (int b = 0; b < B; ++b) if (i0 + b * nthreads < nvec) v[b] = raw[i0 + b * nthreads];
#pragma unroll
        for (int b = 0; b < B; ++b) {
            if (i0 + b * nthreads < nvec) {
                float4 h, l;
                split4(v[b], h, l);
#if !PYMFB_TC_RAW_HI
                raw[i0 + b * nthreads] = h;
#endif
                lo[i0 + b * nthreads] = l;
            }
        }
    }
}

// [H_hi ; H_lo] companion of H ("Hs", the B operand of the X.H^T pass) is stored CHUNK-MAJOR:
// element (row j of the 2KP stacked rows, column c) lives at ((c / 32) * 2KP + j) * 32 + c % 32, so one
// pipeline stage (2KP rows x 32 columns) is ONE contiguous 2KP x 128 B block.  With the row-major layout
// the 2KP rows of a stage sat ldh * 4 bytes apart - 256 different 2 MB pages per stage at k = 128,
// n = 2^20 - and the pass ran 2.2x slower on one GPU than on 8 column shards (TLB-bound TMA).
__host__ __device__ __forceinline__ int64_t hs_index(int j, int64_t col, int kp2) {
    return ((col >> 5) * kp2 + j) * 32 + (col & 31);
}

// PYMFB_TRACE (experiment builds only): CTA 0 records clock64() at the hand-over points of its first
// TRACE_STAGES pipeline stages into dbg + 1 MB; dumped by tc_release() to $PYMFB_TRACE_FILE.
#if defined(PYMFB_TRACE)
constexpr int TRACE_STAGES = 4096;
#define TRACE_AT(stage_idx, slot)                                                                           \
    do {                                                                                                    \
        if (dbg != nullptr && blockIdx.x == 0 && lane == 0 && (stage_idx) < (uint32_t)TRACE_STAGES)                   \
            reinterpret_cast<long long*>(dbg + (1 << 18))[(size_t)(stage_idx) * 16 + (slot)] = clock64();   \
    } while (0)
#else
#define TRACE_AT(stage_idx, slot) do { } while (0)
#endif

constexpr int SEG_STAGES = 8;         // stages per accumulation segment (see "segments" below)
#ifndef PYMFB_SS_SEG_X
#define PYMFB_SS_SEG_X 8               // the same for the X H^T / H H^T passes of the SS kernels (run-time: PYMFB_SEG_X)
#endif

// Segments.  tcgen05.mma adds into the fp32 TMEM accumulator with truncation, so a chain of n
// accumulating MMAs over positive data comes out LOW by ~4.2e-8 * n relative (measured: 2.7e-5 after
// the 512 MMAs of d = 4096).  Both passes therefore cut their contraction into segments: the MMA
// thread alternates between two TMEM buffers, and the epilogue warps drain each finished segment
// into fp32 registers with round-to-nearest adds while the next segment is being accumulated.
//
// The segment LENGTH matters beyond its own bias.  The update H <- H * C / D is a ratio, and W, H
// carry a neutral direction (W * s, H / s leaves W H unchanged) with no restoring force: a bias of
// delta_C - delta_D per iteration in C / D accumulates LINEARLY over the iterations.  With 32-MMA
// chains for C = W^T X against the k/8-MMA chain of D = G H the cfg2 prefix drifted 1.18e-6 per
// iteration - a pure scale, H down, W up (tests/_drift_probe.py) - i.e. 1.2e-4 after 100 iterations,
// beyond the 1e-4 tolerance, while everything except the scale stayed at 1e-6.  Hence: the C
// contraction uses segments of seg_c = (rows of H contracted for G H) / 32 stages, so that the C
// chain has exactly as many MMAs as the D chain and the two biases cancel in the ratio to first order;
// the X H^T and H H^T contractions of the W update (ratio A / (W B)) both use SEG_STAGES-stage
// segments over column ranges that are multiples of a segment, for the same reason.
// Rings of the SS kernels (round 2).  Round 1 kept ONE ring whose stage held everything a contraction step needs -
// the X box, its lo tile and the [b_hi | b_lo] operand chunk: 64 KB per 16 KB of X at k = 128, i.e. 3 stages = 48 KB
// of X in flight per SM, every byte of it parked for the whole TMA -> split -> MMA lifetime (~4 500 cycles).  Ablation
// builds (build_exp/ablate.sh: no operand loads / no split / half-width MMAs) each took ~10 % off the pass and all
// three together 29 %: the pass was bound by bytes in flight / slot lifetime, not by the tensor pipe.  The three
// buffers have very different lifetimes, so they now live in three rings:
//   X ring   NX x 16 KB   HBM latency + split + MMA      (the long one: gets the most slots)
//   lo ring  NL x 16 KB   split + MMA                    (allocated by the split warps, not at TMA issue)
//   B ring   NW x 2KP x 128 B   L2 latency + MMA         (operand chunk, same for every CTA: an L2 hit)
#ifndef PYMFB_SS_MMA_ORDER
#define PYMFB_SS_MMA_ORDER 0   // experiment: 0 = hi (N = 2k) / lo (N = k) MMAs interleaved per k-step, 1 = the stage's hi MMAs first, then its
                               // lo MMAs, 2 = three N = k MMAs per k-step (no accumulator range shared by MMAs of different width)
#endif
#ifndef PYMFB_SS_NW
#define PYMFB_SS_NW 3
#endif
#ifndef PYMFB_SS_NL
#define PYMFB_SS_NL 0      // 0: 2 slots for k > 96, else 3
#endif
template <int KP>
struct SsRings {
    static constexpr int BSTAGE_BYTES = 2 * KP * 128;               // [b_hi | b_lo]: 2KP x 32 fp32
    static constexpr int NW = PYMFB_SS_NW;
    static constexpr int NL = PYMFB_SS_NL > 0 ? PYMFB_SS_NL : (KP > 96 ? 2 : 3);
    static constexpr int NX_RAW = (SMEM_LIMIT - 2048 - NW * BSTAGE_BYTES - NL * XSTAGE_BYTES) / XSTAGE_BYTES;
    static constexpr int NX = NX_RAW > 8 ? 8 : NX_RAW;
    static constexpr int LO_OFF = NX * XSTAGE_BYTES;
    static constexpr int B_OFF = LO_OFF + NL * XSTAGE_BYTES;
    static constexpr int BAR_OFF = B_OFF + NW * BSTAGE_BYTES;
    static constexpr int NR = NW;                                   // "stage ready" barriers (see SsBars); must be >= NL and >= NW
    static constexpr int NBAR = 2 * NX + NR + 4;                    // fullx, done, ready, tfull[2], tempty[2]
    static constexpr int SMEM_BYTES = BAR_OFF + 1024 /*align*/ + 512 /*barriers*/;
    static_assert(NX >= 2 && NL >= 2 && NW >= 2, "not enough shared memory for the three rings");
    static_assert(NR >= NL && NR >= NW && NX >= NR, "barrier ring depths");
    static_assert(NBAR * 8 + 8 <= 512, "barrier area too small");
    static_assert(SMEM_BYTES <= SMEM_LIMIT, "rings do not fit");
};

template <int KP>
struct HCfg : SsRings<KP> {   // H-update pass
    static constexpr int NCH = 2 * KP / 32;                         // 32-column chunks of [hi | lo]
    static constexpr int WSTAGE_BYTES = NCH * R1 * 128;             // R1 rows x 2KP fp32 (= BSTAGE_BYTES)
    static constexpr int SEG_COLS = 2 * KP;                         // [hi | small] per segment buffer
    static constexpr int EPI_WARPS = KP > 64 ? 8 : 4;               // 2 warps per TMEM lane quarter for wide k
    static constexpr int NJ = KP / (EPI_WARPS / 4);                 // basis columns per epilogue thread
    static constexpr int THREADS = 32 * (NPROD + 5 + EPI_WARPS);
    static_assert(KP % 32 == 0 && KP >= 32 && KP <= 128, "KP must be 32, 64, 96 or 128");
    static_assert(NJ % 16 == 0, "epilogue column split must be a multiple of 16");
    static_assert(WSTAGE_BYTES == SsRings<KP>::BSTAGE_BYTES, "operand stage size");
};

// Barriers of the SS kernels.  The MMA warp is the serial resource of these kernels: a PYMFB_TRACE run of the first
// three-ring version (three waits - operand chunk, X box, lo tile - and three tcgen05.commit per stage, one per ring)
// showed it spending ~1 250 cycles per stage - 230 waiting, 230 issuing the 8 MMAs, 500 in the three commits and 290
// in loop bookkeeping - against 768 cycles of tensor work.  Hence ONE wait and ONE commit per stage:
//   ready[i % NR]  the stage's operands are in place: 4 arrivals of the split warps (lo tile written; they waited for
//                  the X box, so it implies fullx) + the arrive.expect_tx of the operand-chunk producer + its bytes;
//   done[i % NX]   tcgen05.commit of the stage's MMAs.  It frees the X slot (the X producer waits NX stages back),
//                  the lo slot (the split warps wait NL stages back) and the chunk slot (NW stages back) alike: MMAs
//                  complete in order, and a waiter that lags L <= NX stages behind sees at most one completion it does
//                  not expect on its barrier, so the parity wait cannot alias.
template <class Cfg>
struct SsBars {
    uint32_t base;
    __device__ __forceinline__ uint32_t fullx(int s) const { return base + 8u * s; }
    __device__ __forceinline__ uint32_t done(int s) const { return base + 8u * (Cfg::NX + s); }
    __device__ __forceinline__ uint32_t ready(int s) const { return base + 8u * (2 * Cfg::NX + s); }
    __device__ __forceinline__ uint32_t tfull(int a) const { return base + 8u * (2 * Cfg::NX + Cfg::NR + a); }
    __device__ __forceinline__ uint32_t tempty(int a) const { return base + 8u * (2 * Cfg::NX + Cfg::NR + 2 + a); }
    __device__ __forceinline__ uint32_t tmem_slot() const { return base + 8u * Cfg::NBAR; }
    __device__ __forceinline__ void init(int epi_warps) const {
        for (int s = 0; s < Cfg::NX; ++s) { mbar_init(fullx(s), 1); mbar_init(done(s), 1); }
        for (int s = 0; s < Cfg::NR; ++s) mbar_init(ready(s), 5);
        for (int a = 0; a < 2; ++a) { mbar_init(tfull(a), 1); mbar_init(tempty(a), epi_warps); }
    }
};
// slot index + phase of one ring
template <int N>
struct RingPos {
    int s = 0; uint32_t ph = 0;
    __device__ __forceinline__ void next() { if (++s == N) { s = 0; ph ^= 1u; } }
};
// position in the done[] ring that trails the caller by LAG stages: wait() returns once the MMAs of stage i - LAG have
// completed (no-op for the first LAG stages); call it once per stage
template <int NX, int LAG>
struct DoneLag {
    RingPos<NX> p; int skip = LAG;
    template <class Bars>
    __device__ __forceinline__ void wait(const Bars& bar, bool mine = true) {
        if (skip > 0) { --skip; return; }
        if (mine) mbar_wait(bar.done(p.s), p.ph);
        p.next();
    }
};

// ---------------------------------------------------------------------------------------------
// H-update pass.  Per 128-column tile (TMEM lanes = columns of the tile, TMEM columns = basis index):
//   C segments:  [ X^T W_hi | X^T W_lo + X_lo^T W_hi ]  over 256-row slices of X  -> summed in registers
//   D segment :  [ H^T G_hi | H^T G_lo + H_lo^T G_hi ]  over the kp rows of H
//   epilogue  :  Hn = H * C / (D + 1e-9)
// X/W and H/G stages travel through the same TMA -> split -> MMA rings.
// warp 0: TMA producer of X, warps 1-2: TMA producers of the operand chunks, warp 3: MMA issuer,
// warps 4-7: lo split, warps 8..: epilogue.
// PROD = true (NNDSVD's Z^T = Q^T X, W := Q): the plain product - no G H stages, the epilogue stores C into Hn;
// Hc, Hs, mapH, mapG, kh_rows, lam, Dp, Dn are not read.
// ---------------------------------------------------------------------------------------------
template <int KP, bool PROD = false>
__global__ void __launch_bounds__(HCfg<KP>::THREADS, 1)
k_h_update_tc(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
              const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapG,
              const DevState* __restrict__ st, const float* __restrict__ Hc, float* __restrict__ Hn,
              float* __restrict__ Hs, int64_t ldh, int d, int n_loc, int num_tiles, float* __restrict__ dbg,
              int kh_rows, int seg_c, float lam, const float* __restrict__ Dp, const float* __restrict__ Dn, int xsh, int pf) {
    // pf: L2 prefetch distance of X in stages (0 = off)
    // xsh: log2 of the panel width of X (tma_load_x)
    // seg_c: stages per accumulation segment of the W^T X contraction (see "Segments" above)
    // kh_rows: rows of H contracted for G H (= the padded k of the whole problem).  For k <= 128 it equals KP;
    // for k > 128 the launch handles one 128-wide block of bases: mapH spans all kh_rows rows of H, mapG is the
    // block's [G_hi | G_lo] column slice, and Hc / Hn / Hs point at the block's rows.
    using Cfg = HCfg<KP>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const SsBars<Cfg> bar{smem_base + Cfg::BAR_OFF};
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::BAR_OFF + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapW); tma_prefetch_desc(&mapH); tma_prefetch_desc(&mapG);
        bar.init(Cfg::EPI_WARPS);
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(bar.tmem_slot(), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    const int nd = (d + R1 - 1) / R1;            // stages over the rows of X
    const int nit = nd + (PROD ? 0 : kh_rows / R1);   // + stages over the rows of H (for G H)
    auto xraw = [&](int s) { return smem_base + s * XSTAGE_BYTES; };
    auto xlo = [&](int s) { return smem_base + Cfg::LO_OFF + s * XSTAGE_BYTES; };
    auto wch = [&](int s) { return smem_base + Cfg::B_OFF + s * Cfg::WSTAGE_BYTES; };

    if (warp == 0) {
        // ===== TMA producer of the X / H boxes =====
        RingPos<Cfg::NX> rx;
        uint32_t tc_ = 0; (void)tc_;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int col0 = tile * TILE_COLS;
            for (int it = 0; it < nit; ++it, ++tc_) {
                TRACE_AT(tc_, 0);
                mbar_wait_relaxed(bar.done(rx.s), rx.ph ^ 1);
                TRACE_AT(tc_, 1);
                if (elect_one()) {
                    mbar_expect_tx(bar.fullx(rx.s), XSTAGE_BYTES);
                    const bool xphase = it < nd;
                    const int r0 = (xphase ? it : it - nd) * R1;
                    const CUtensorMap* ma = xphase ? &mapX : &mapH;
#pragma unroll
                    for (int c = 0; c < 4; ++c) tma_load_x(xraw(rx.s) + c * (R1 * 128), ma, bar.fullx(rx.s), col0 + 32 * c, r0, xphase ? xsh : kNoPanel);
                    if (pf > 0 && it + pf < nd) {      // pull the rows this tile needs pf stages from now into L2
#pragma unroll
                        for (int c = 0; c < 4; ++c) tma_prefetch_x(&mapX, col0 + 32 * c, (it + pf) * R1, xsh);
                    }
                }
                __syncwarp();
                rx.next();
            }
        }
    } else if (warp < NPROD) {
        // ===== TMA producers of the [W_hi|W_lo] / [G_hi|G_lo] chunks (stages alternate between the warps) =====
        RingPos<Cfg::NW> rw;                        // chunk slot = ready barrier of the stage (NR == NW)
        DoneLag<Cfg::NX, Cfg::NW> lag;
        uint32_t cnt = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int it = 0; it < nit; ++it) {
                const bool mine = cnt++ % (NPROD - 1) == (uint32_t)(warp - 1);
                if (mine) TRACE_AT(cnt - 1, 10);
                lag.wait(bar, mine);
                if (mine) {
                    TRACE_AT(cnt - 1, 11);
                    if (elect_one()) {
#if defined(PYMFB_EXP_SS_SKIP_B)
                        mbar_arrive(bar.ready(rw.s));
#else
                        mbar_expect_tx(bar.ready(rw.s), Cfg::WSTAGE_BYTES);
                        const bool xphase = it < nd;
                        const int r0 = (xphase ? it : it - nd) * R1;
                        const CUtensorMap* mb = xphase ? &mapW : &mapG;
#pragma unroll
                        for (int c = 0; c < Cfg::NCH; ++c) tma_load_2d(wch(rw.s) + c * (R1 * 128), mb, bar.ready(rw.s), 32 * c, r0);
#endif
                    }
                    __syncwarp();
                }
                rw.next();
            }
        }
    } else if (warp == NPROD) {
        // ===== MMA issuer =====
        {
#if defined(PYMFB_EXP_SS_HALF_N)
            constexpr uint32_t idesc_hl = make_idesc(128, KP, 1, 1);
            constexpr uint32_t idesc_h = make_idesc(128, KP / 2, 1, 1);
#else
            constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 1, 1);
            constexpr uint32_t idesc_h = make_idesc(128, KP, 1, 1);
#endif
            RingPos<Cfg::NX> rx; RingPos<Cfg::NL> rl; RingPos<Cfg::NW> rw;
            uint32_t g = 0, mc = 0; (void)mc;
            // descriptors of slot 0 of each ring (one MMA, K = 8, = two 4-row swizzle atoms, SBO = 512 B; 32-column chunks LBO
            // apart); slot s / k-group kg add (s * slot bytes + kg * 1024) >> 4 to the low words, the high words never change
            // (shared-memory addresses are < 2^18, so the 14-bit address field never carries)
            const uint64_t d_hi0 = make_desc(xraw(0), R1 * 128, 512, 1), d_lo0 = make_desc(xlo(0), R1 * 128, 512, 1);
            const uint64_t d_b0 = make_desc(wch(0), R1 * 128, 512, 1);
            const uint32_t dh = (uint32_t)(d_hi0 >> 32);      // identical for the three operands (same LBO / SBO / layout)
            const uint32_t ahi0 = (uint32_t)d_hi0, alo0 = (uint32_t)d_lo0, b0 = (uint32_t)d_b0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                int it = 0;
                while (it < nit) {
                    const int seg_end = (it < nd) ? min(it + seg_c, nd) : nit;
                    const uint32_t b = g & 1u;
                    mbar_wait(bar.tempty(b), ((g >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                    bool first = true;
                    for (; it < seg_end; ++it, ++mc) {
                        TRACE_AT(mc, 5);
                        mbar_wait(bar.ready(rw.s), rw.ph);
                        TRACE_AT(mc, 6);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t ox = ahi0 + rx.s * (XSTAGE_BYTES >> 4), ol = alo0 + rl.s * (XSTAGE_BYTES >> 4);
                            const uint32_t ob = b0 + rw.s * (Cfg::WSTAGE_BYTES >> 4);
#if PYMFB_SS_MMA_ORDER == 0
#pragma unroll
                            for (int kg = 0; kg < R1 / 8; ++kg) {
                                const uint32_t o = kg * (1024 >> 4);
                                umma_tf32_lh(dcol, ox + o, dh, ob + o, dh, idesc_hl, (first && kg == 0) ? 0u : 1u);
                                umma_tf32_lh(dcol + KP, ol + o, dh, ob + o, dh, idesc_h, 1u);
                            }
#elif PYMFB_SS_MMA_ORDER == 1
#pragma unroll
                            for (int kg = 0; kg < R1 / 8; ++kg)
                                umma_tf32_lh(dcol, ox + kg * (1024 >> 4), dh, ob + kg * (1024 >> 4), dh, idesc_hl, (first && kg == 0) ? 0u : 1u);
#pragma unroll
                            for (int kg = 0; kg < R1 / 8; ++kg)
                                umma_tf32_lh(dcol + KP, ol + kg * (1024 >> 4), dh, ob + kg * (1024 >> 4), dh, idesc_h, 1u);
#else
#pragma unroll
                            for (int kg = 0; kg < R1 / 8; ++kg) {
                                const uint32_t o = kg * (1024 >> 4);
                                const uint32_t acc = (first && kg == 0) ? 0u : 1u;
                                umma_tf32_lh(dcol, ox + o, dh, ob + o, dh, idesc_h, acc);
                                umma_tf32_lh(dcol + KP, ox + o, dh, ob + o + ((KP / 32) * R1 * 128 >> 4), dh, idesc_h, acc);
                                umma_tf32_lh(dcol + KP, ol + o, dh, ob + o, dh, idesc_h, 1u);
                            }
#endif
                            TRACE_AT(mc, 14);
                            umma_commit(bar.done(rx.s));
                            if (it + 1 == seg_end) umma_commit(bar.tfull(b));     // last stage of the segment: hand it to the epilogue
                        }
                        __syncwarp();
                        TRACE_AT(mc, 7);
                        first = false;
                        rx.next(); rl.next(); rw.next();
                    }
                    ++g;
                }
            }
        }
    } else if (warp < NPROD + 5) {
        // ===== split warps: lo tiles (and masked hi) of the X / H operand =====
        const int tid_s = threadIdx.x - 32 * (NPROD + 1);
        RingPos<Cfg::NX> rx; RingPos<Cfg::NL> rl; RingPos<Cfg::NR> rr;
        DoneLag<Cfg::NX, Cfg::NL> lag;
        uint32_t sc = 0; (void)sc;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int it = 0; it < nit; ++it, ++sc) {
                if (warp == NPROD + 1) TRACE_AT(sc, 2);
                mbar_wait(bar.fullx(rx.s), rx.ph);
                if (warp == NPROD + 1) TRACE_AT(sc, 9);
                lag.wait(bar);
                if (warp == NPROD + 1) TRACE_AT(sc, 3);
                float4* raw = reinterpret_cast<float4*>(smem_gen + rx.s * XSTAGE_BYTES);
                float4* lo = reinterpret_cast<float4*>(smem_gen + Cfg::LO_OFF + rl.s * XSTAGE_BYTES);
                split_buffer(raw, lo, XSTAGE_BYTES / 16, tid_s, 128);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar.ready(rr.s));
                if (warp == NPROD + 1) TRACE_AT(sc, 4);
                rx.next(); rl.next(); rr.next();
            }
        }
    } else {
        // ===== epilogue warps: drain segments into registers, then the H update =====
        const int q = warp & 3;                       // TMEM lane quarter this warp may access
        const int jbase = ((warp - (NPROD + 5)) >> 2) * Cfg::NJ;   // basis columns [jbase, jbase + NJ) of this warp
        const int nsegC = (nd + seg_c - 1) / seg_c;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            float creg[Cfg::NJ];
#pragma unroll
            for (int j = 0; j < Cfg::NJ; ++j) creg[j] = 0.f;
            for (int seg = 0; seg < nsegC; ++seg, ++g) {
                const uint32_t b = g & 1u;
                mbar_wait_relaxed(bar.tfull(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS + jbase;
#if !defined(PYMFB_EXP_SS_SKIP_DRAIN)
#pragma unroll
                for (int j0 = 0; j0 < Cfg::NJ; j0 += 16) {
                    float hi[16], sm[16];
                    tmem_ld16(taddr + j0, hi);
                    tmem_ld16(taddr + KP + j0, sm);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) creg[j0 + j] += hi[j] + sm[j];
                }
#else
                (void)taddr;
#endif
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar.tempty(b));
            }
            if constexpr (PROD) {
                const int col = tile * TILE_COLS + q * 32 + lane;
                if (col < n_loc) {
#pragma unroll
                    for (int j = 0; j < Cfg::NJ; ++j) Hn[(int64_t)(jbase + j) * ldh + col] = creg[j];
                }
            } else {   // D segment + H update
                const uint32_t b = g & 1u;
                mbar_wait_relaxed(bar.tfull(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS + jbase;
                const int col = tile * TILE_COLS + q * 32 + lane;
#pragma unroll
                for (int j0 = 0; j0 < Cfg::NJ; j0 += 16) {
                    float dh[16], dl[16];
                    tmem_ld16(taddr + j0, dh);
                    tmem_ld16(taddr + KP + j0, dl);
                    tmem_ld_wait();
                    if (dbg != nullptr && tile == 0) {   // raw sums of tile 0 (tests/tc_probe.cu)
                        float* o = dbg + (size_t)(q * 32 + lane) * (2 * KP) + jbase + j0;
#pragma unroll
                        for (int j = 0; j < 16; ++j) { o[j] = creg[j0 + j]; o[KP + j] = dh[j] + dl[j]; }
                    }
                    if (col < n_loc) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int64_t o = (int64_t)(jbase + j0 + j) * ldh + col;
                            const float h = Hc[o];
                            const float hn = (Dp != nullptr) ? snmf_ratio(h, creg[j0 + j], Dp[o], Dn[o]) : mu_ratio(h, creg[j0 + j], dh[j] + dl[j], lam);
                            const float hh = __uint_as_float(__float_as_uint(hn) & 0xFFFFE000u);
                            Hn[o] = hn;                                  // new H
                            Hs[hs_index((jbase + j0 + j), col, 2 * KP)] = hh;        // [H_hi ; H_lo] rows for the X.H^T pass
                            Hs[hs_index(KP + (jbase + j0 + j), col, 2 * KP)] = hn - hh;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar.tempty(b));
                ++g;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}

template <int KP>
struct XCfg : SsRings<KP> {   // X H^T pass
    static constexpr int HSTAGE_BYTES = 2 * KP * 128;               // [H hi rows | H lo rows] x 32 cols (= BSTAGE_BYTES)
    static constexpr int SEG_COLS = 2 * KP;                         // [hi | small]
    static constexpr int EPI_WARPS = KP > 64 ? 8 : 4;
    static constexpr int NJ = KP / (EPI_WARPS / 4);
    static constexpr int THREADS = 32 * (NPROD + 5 + EPI_WARPS);
    static_assert(KP % 32 == 0 && KP >= 32 && KP <= 128, "KP must be 32, 64, 96 or 128");
    static_assert(NJ % 16 == 0, "epilogue column split must be a multiple of 16");
};

// ---------------------------------------------------------------------------------------------
// X H^T pass.  Task = (block of 128 rows of X, range of columns).  TMEM lanes = rows of X, TMEM
// columns = basis index; segments [ X H_hi^T | X H_lo^T + X_lo H_hi^T ] over 256 columns each are
// summed in registers and flushed once per task into this split's copy of P (or with fp32 atomics).
// Same three rings as the H-update pass: warp 0 loads the X boxes, warps 1-2 the [H_hi ; H_lo] chunks.
// ---------------------------------------------------------------------------------------------
template <int KP>
__global__ void __launch_bounds__(XCfg<KP>::THREADS, 1)
k_xht_tc(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapH,
         const DevState* __restrict__ st, float* __restrict__ P, int d, int n_loc,
         int cols_per_task, int num_rb, int num_tasks, float* __restrict__ dbg, int ldp,
         float* __restrict__ Ppart, int64_t part_stride, int xsh, int xrev, int pf, int seg_x) {
    // seg_x: stages per accumulation segment (X H^T and H H^T launches must use the same value, see "Segments")
    // ldp: row stride of P (= padded k of the whole problem; P points at this launch's block of columns)
    // Ppart != nullptr: deterministic combine of the column splits - every task stores its sums in copy (task / num_rb)
    // of P's layout (part_stride floats apart) and k_sum_copies adds the copies in split order into P afterwards.
    // Ppart == nullptr: fp32 atomics into a cleared P.
    using Cfg = XCfg<KP>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const SsBars<Cfg> bar{smem_base + Cfg::BAR_OFF};
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::BAR_OFF + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapH);
        bar.init(Cfg::EPI_WARPS);
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(bar.tmem_slot(), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    auto xraw = [&](int s) { return smem_base + s * XSTAGE_BYTES; };
    auto xlo = [&](int s) { return smem_base + Cfg::LO_OFF + s * XSTAGE_BYTES; };
    auto hch = [&](int s) { return smem_base + Cfg::B_OFF + s * Cfg::HSTAGE_BYTES; };
    auto task_chunks = [&](int task, int& c_begin) {     // number of 32-column stages of a task
        // xrev: walk the column ranges from the END of the matrix - the H-update pass that ran just before finished
        // there, so the first tasks find their X columns still in L2 (and this pass ends where the next H-update starts)
        const int cs = xrev ? (num_tasks / num_rb - 1 - task / num_rb) : task / num_rb;
        c_begin = cs * cols_per_task;
        const int c_end = min(n_loc, c_begin + cols_per_task);
        return (c_end - c_begin + 31) / 32;
    };

    // L2 priorities: a box of X is read once per pass (evict_first); the [H_hi ; H_lo] chunks of a column range are
    // re-read by every row-block CTA of that range (evict_last), so streaming X does not push them out of L2.  Against
    // the default priority for H, evict_last measured equal on cfg3 and 0.5-1 % faster on cfg4 k = 128 / 512.
    if (warp == 0) {
        const uint64_t pol_x = l2_policy_evict_first();
        RingPos<Cfg::NX> rx;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin;
            const int nch = task_chunks(task, c_begin);
            const int row0 = (task % num_rb) * 128;
            for (int ch = 0; ch < nch; ++ch) {
                mbar_wait_relaxed(bar.done(rx.s), rx.ph ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(bar.fullx(rx.s), XSTAGE_BYTES);
                    tma_load_x_hint(xraw(rx.s), &mapX, bar.fullx(rx.s), c_begin + 32 * ch, row0, xsh, pol_x);
                    if (pf > 0 && ch + pf < nch) tma_prefetch_x(&mapX, c_begin + 32 * (ch + pf), row0, xsh);
                }
                __syncwarp();
                rx.next();
            }
        }
    } else if (warp < NPROD) {
        const uint64_t pol_h = l2_policy_evict_last();
        RingPos<Cfg::NW> rw;
        DoneLag<Cfg::NX, Cfg::NW> lag;
        uint32_t cnt = 0;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin;
            const int nch = task_chunks(task, c_begin);
            for (int ch = 0; ch < nch; ++ch) {
                const bool mine = cnt++ % (NPROD - 1) == (uint32_t)(warp - 1);
                lag.wait(bar, mine);
                if (mine) {
                    if (elect_one()) {
#if defined(PYMFB_EXP_SS_SKIP_B)
                        mbar_arrive(bar.ready(rw.s));
#else
                        mbar_expect_tx(bar.ready(rw.s), Cfg::HSTAGE_BYTES);
                        tma_load_2d_hint(hch(rw.s), &mapH, bar.ready(rw.s), 0, ((c_begin >> 5) + ch) * (2 * KP), pol_h);   // [H_hi ; H_lo] chunk
#endif
                    }
                    __syncwarp();
                }
                rw.next();
            }
        }
    } else if (warp == NPROD) {
        {
#if defined(PYMFB_EXP_SS_HALF_N)
            constexpr uint32_t idesc_hl = make_idesc(128, KP, 0, 0);
            constexpr uint32_t idesc_h = make_idesc(128, KP / 2, 0, 0);
#else
            constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 0, 0);
            constexpr uint32_t idesc_h = make_idesc(128, KP, 0, 0);
#endif
            RingPos<Cfg::NX> rx; RingPos<Cfg::NL> rl; RingPos<Cfg::NW> rw;
            uint32_t g = 0;
            // K-major SW128 descriptors of slot 0 of each ring; slot s / k-step ks add (s * slot bytes + ks * 32) >> 4 to the low words
            const uint64_t xd_hi0 = make_desc(xraw(0), 16, 1024), xd_lo0 = make_desc(xlo(0), 16, 1024), xd_b0 = make_desc(hch(0), 16, 1024);
            const uint32_t xdh = (uint32_t)(xd_hi0 >> 32);
            const uint32_t xahi0 = (uint32_t)xd_hi0, xalo0 = (uint32_t)xd_lo0, xb0 = (uint32_t)xd_b0;
            for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
                int c_begin;
                const int nch = task_chunks(task, c_begin);
                int ch = 0;
                while (ch < nch) {
                    const int seg_end = min(ch + seg_x, nch);
                    const uint32_t b = g & 1u;
                    mbar_wait(bar.tempty(b), ((g >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                    bool first = true;
                    for (; ch < seg_end; ++ch) {
                        mbar_wait(bar.ready(rw.s), rw.ph);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t ox = xahi0 + rx.s * (XSTAGE_BYTES >> 4), ol = xalo0 + rl.s * (XSTAGE_BYTES >> 4);
                            const uint32_t ob = xb0 + rw.s * (Cfg::HSTAGE_BYTES >> 4);
#if PYMFB_SS_MMA_ORDER == 0
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                const uint32_t o = ks * (32 >> 4);
                                umma_tf32_lh(dcol, ox + o, xdh, ob + o, xdh, idesc_hl, (first && ks == 0) ? 0u : 1u);
                                umma_tf32_lh(dcol + KP, ol + o, xdh, ob + o, xdh, idesc_h, 1u);
                            }
#elif PYMFB_SS_MMA_ORDER == 1
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                umma_tf32_lh(dcol, ox + ks * (32 >> 4), xdh, ob + ks * (32 >> 4), xdh, idesc_hl, (first && ks == 0) ? 0u : 1u);
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks)
                                umma_tf32_lh(dcol + KP, ol + ks * (32 >> 4), xdh, ob + ks * (32 >> 4), xdh, idesc_h, 1u);
#else
#pragma unroll
                            for (int ks = 0; ks < 4; ++ks) {
                                const uint32_t o = ks * (32 >> 4);
                                const uint32_t acc = (first && ks == 0) ? 0u : 1u;
                                umma_tf32_lh(dcol, ox + o, xdh, ob + o, xdh, idesc_h, acc);
                                umma_tf32_lh(dcol + KP, ox + o, xdh, ob + o + (KP * 128 >> 4), xdh, idesc_h, acc);
                                umma_tf32_lh(dcol + KP, ol + o, xdh, ob + o, xdh, idesc_h, 1u);
                            }
#endif
                            umma_commit(bar.done(rx.s));
                            if (ch + 1 == seg_end) umma_commit(bar.tfull(b));     // last stage of the segment: hand it to the epilogue
                        }
                        __syncwarp();
                        first = false;
                        rx.next(); rl.next(); rw.next();
                    }
                    ++g;
                }
            }
        }
    } else if (warp < NPROD + 5) {
        const int tid_s = threadIdx.x - 32 * (NPROD + 1);
        RingPos<Cfg::NX> rx; RingPos<Cfg::NL> rl; RingPos<Cfg::NR> rr;
        DoneLag<Cfg::NX, Cfg::NL> lag;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin;
            const int nch = task_chunks(task, c_begin);
            for (int ch = 0; ch < nch; ++ch) {
                mbar_wait(bar.fullx(rx.s), rx.ph);
                lag.wait(bar);
                split_buffer(reinterpret_cast<float4*>(smem_gen + rx.s * XSTAGE_BYTES),
                             reinterpret_cast<float4*>(smem_gen + Cfg::LO_OFF + rl.s * XSTAGE_BYTES), XSTAGE_BYTES / 16, tid_s, 128);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar.ready(rr.s));
                rx.next(); rl.next(); rr.next();
            }
        }
    } else {
        const int q = warp & 3;
        const int jbase = ((warp - (NPROD + 5)) >> 2) * Cfg::NJ;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin;
            const int nch = task_chunks(task, c_begin);
            const int nseg = (nch + seg_x - 1) / seg_x;
            float areg[Cfg::NJ];
#pragma unroll
            for (int j = 0; j < Cfg::NJ; ++j) areg[j] = 0.f;
            for (int seg = 0; seg < nseg; ++seg, ++g) {
                const uint32_t b = g & 1u;
                mbar_wait_relaxed(bar.tfull(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS + jbase;
#pragma unroll
                for (int j0 = 0; j0 < Cfg::NJ; j0 += 16) {
                    float hi[16], sm[16];
                    tmem_ld16(taddr + j0, hi);
                    tmem_ld16(taddr + KP + j0, sm);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) areg[j0 + j] += hi[j] + sm[j];
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar.tempty(b));
            }
            const int row = (task % num_rb) * 128 + q * 32 + lane;
            if (dbg != nullptr && task == 0) {
                float* o = dbg + (size_t)(q * 32 + lane) * KP + jbase;
#pragma unroll
                for (int j = 0; j < Cfg::NJ; ++j) o[j] = areg[j];
            }
            if (row < d) {
                if (Ppart == nullptr) {
                    float* dst = P + (int64_t)row * ldp + jbase;
#pragma unroll
                    for (int j = 0; j < Cfg::NJ; ++j) atomicAdd(dst + j, areg[j]);
                } else {                               // this split's copy of P; k_sum_copies adds the copies in order
                    float* dst = Ppart + (int64_t)(task / num_rb) * part_stride + (int64_t)row * ldp + jbase;
#pragma unroll
                    for (int j = 0; j < Cfg::NJ; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(areg[j], areg[j + 1], areg[j + 2], areg[j + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}

// =============================================================================================
// TS variants (k <= 64): the X operand is fed to the tensor core from TENSOR MEMORY.
//
// With both operands in shared memory every byte of X crosses the 128 B/clk shared-memory port
// ~7 times per pass (TMA write, split read, hi/lo writes, two MMA operand reads) and the pass is
// shared-memory-bound at ~70 % of HBM speed (measured).  Here the 4 convert warps read each X
// element from shared memory ONCE, split it in registers and park hi/lo in TMEM with tcgen05.st;
// tcgen05.mma then takes A from TMEM and only the small [W_hi|W_lo] / [H_hi|H_lo] operand from
// shared memory: ~3 B of shared-memory traffic per byte of X.
//   TMEM columns: [0, 4KP) two segment accumulators, then NT x 64 columns of A ring (32 hi + 32 lo).
// =============================================================================================
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// Same, with the shared-memory descriptor passed as two 32-bit halves: the high half (LBO/SBO/layout bits) is loop
// invariant and the low half only advances by (byte offset >> 4), so the issue loop does one 32-bit add per
// descriptor instead of rebuilding it (shift, mask, or) on the uniform datapath for every k-step.
__device__ __forceinline__ void umma_tf32_ts_lh(uint32_t d_tmem, uint32_t a_tmem, uint32_t bd_lo, uint32_t bd_hi, uint32_t idesc,
                                                uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 bd;\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "mov.b64 bd, {%2, %3};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], bd, %4, p;\n\t}"
        ::"r"(d_tmem), "r"(a_tmem), "r"(bd_lo), "r"(bd_hi), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
          "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
          "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
          "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

#ifndef PYMFB_NCHAIN
#define PYMFB_NCHAIN 1   // 2 was measured: no change (316 vs 309 us on the per-SM-bound probe), so the default stays 1
#endif
#ifndef PYMFB_H_CONV_GROUPS
#define PYMFB_H_CONV_GROUPS 1   // convert-warp groups of the TS H-update kernel (2 = alternate stages, 16 warps per CTA)
#endif
template <int KP>
struct TsCfg {
    static constexpr int CONV_GROUPS = PYMFB_H_CONV_GROUPS;
    static constexpr int NCH = 2 * KP / 32;
    static constexpr int BSTAGE_BYTES = NCH * R1 * 128;             // [b_hi | b_lo] operand per stage (= 2*KP*128)
    static constexpr int STAGE_BYTES = XSTAGE_BYTES + BSTAGE_BYTES;
    static constexpr int STAGES_RAW = (SMEM_LIMIT - 2048) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    // Accumulation chains per segment buffer.  Back-to-back tcgen05.mma into the SAME accumulator are
    // latency-bound when N is small (a K = 8, N = 64 MMA is 32 tensor cycles but the dependent issue
    // distance is far longer), so for KP = 32 consecutive K steps alternate between NCHAIN accumulator
    // sets that the epilogue sums.
    static constexpr int NCHAIN = (KP == 32) ? PYMFB_NCHAIN : 1;
    static constexpr int CHAIN_COLS = 2 * KP;                       // [hi | small] of one chain
    static constexpr int SEG_COLS = CHAIN_COLS * NCHAIN;
    static constexpr int A_COL0 = 2 * SEG_COLS;                     // first TMEM column of the A ring
    static constexpr int NT_RAW = (512 - A_COL0) / 64;
    static constexpr int NT = NT_RAW > 6 ? 6 : NT_RAW;
    static constexpr int EPI_WARPS = 4;
    static constexpr int NJ = KP;
    static constexpr int THREADS = 32 * (NPROD + 1 + 4 * CONV_GROUPS + EPI_WARPS);
    static constexpr int NBAR = 2 * STAGES + 2 * NT + 4;
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 512;
    static_assert(KP == 32 || KP == 64, "TS kernels serve KP = 32 and 64");
    static_assert(NT >= 2, "need at least two A buffers");
    static_assert(NBAR * 8 + 8 <= 512, "barrier area too small");
};

// hi/lo of 32 values -> TMEM A ring slot (this thread's lane, 32 hi columns then 32 lo columns)
__device__ __forceinline__ void park_hilo(uint32_t taddr, const float (&v)[32]) {
    uint32_t hi[32], lo[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        hi[i] = __float_as_uint(v[i]) & 0xFFFFE000u;
        lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
    }
    tmem_st32(taddr, hi);
    tmem_st32(taddr + 32, lo);
}

template <int KP>
__global__ void __launch_bounds__(TsCfg<KP>::THREADS, 1)
k_h_update_ts(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
              const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapG,
              const DevState* __restrict__ st, const float* __restrict__ Hc, float* __restrict__ Hn,
              float* __restrict__ Hs, int64_t ldh, int d, int n_loc, int num_tiles, float* __restrict__ dbg,
              int seg_c, float lam, const float* __restrict__ Dp, const float* __restrict__ Dn,
              const float* __restrict__ wmean, const float* __restrict__ gmean, const float* __restrict__ xsum, int xsh) {
    // wmean != nullptr: the B operands are the CENTERED W / G (k_split_hilo_centered); the epilogue adds
    // wmean[j] * (column sum of X) to W^T X and gmean[j] * (column sum of the H tile) to G H
    // Dp != nullptr: Semi-NMF (pymf/snmf.py:72-90) - the epilogue takes G+ H and G- H from Dp / Dn (same layout
    // as H, written by k_gh_posneg_simt) instead of the G H accumulator
#if !defined(PYMFB_TS_NO_CENTER)
    __shared__ float s_mean[2 * KP];          // [w_mean | g_mean]: read on the critical tail of every tile, so not from global
    if (threadIdx.x < 2 * KP)
        s_mean[threadIdx.x] = (wmean == nullptr) ? 0.f : (threadIdx.x < KP ? wmean[threadIdx.x] : gmean[threadIdx.x - KP]);
#endif
#if defined(PYMFB_TS_SEG_CONST)
    constexpr int segc = SEG_STAGES;          // A/B builds: compile-time segment length as in round 1
#else
    const int segc = seg_c;
#endif
    using Cfg = TsCfg<KP>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::STAGES + s); };
    auto afull_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + t); };
    auto aempty_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + Cfg::NT + t); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + 2 + a); };
    const uint32_t tmem_slot = bar_base + 8u * Cfg::NBAR;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::STAGES * Cfg::STAGE_BYTES + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapW); tma_prefetch_desc(&mapH); tma_prefetch_desc(&mapG);
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int t = 0; t < Cfg::NT; ++t) { mbar_init(afull_bar(t), 4); mbar_init(aempty_bar(t), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), Cfg::EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    const int nd = (d + R1 - 1) / R1;
    const int nit = nd + KP / R1;
    auto xs_addr = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };                    // [32 rows][128 cols] plain
    auto wch = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + XSTAGE_BYTES; };        // MN-major chunks

    if (warp < NPROD) {
        {
            int s = 0; uint32_t ph = 0; uint32_t pcnt = 0;   // this warp issues stages pcnt % NPROD == warp
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int col0 = tile * TILE_COLS;
                for (int it = 0; it < nit; ++it) {
                    if (pcnt++ % NPROD == (uint32_t)warp) {
                    TRACE_AT(pcnt - 1, 0);
                    mbar_wait(empty_bar(s), ph ^ 1);
                    TRACE_AT(pcnt - 1, 1);
                    if (elect_one()) {
#if defined(PYMFB_EXP_SKIP_WLOAD)
                        mbar_expect_tx(full_bar(s), XSTAGE_BYTES);
#else
                        mbar_expect_tx(full_bar(s), XSTAGE_BYTES + Cfg::BSTAGE_BYTES);
#endif
                        const bool xphase = it < nd;
                        const int r0 = (xphase ? it : it - nd) * R1;
                        tma_load_x(xs_addr(s), xphase ? &mapX : &mapH, full_bar(s), col0, r0, xphase ? xsh : kNoPanel);
#if !defined(PYMFB_EXP_SKIP_WLOAD)
                        const CUtensorMap* mb = xphase ? &mapW : &mapG;
#pragma unroll
                        for (int c = 0; c < Cfg::NCH; ++c) tma_load_2d(wch(s) + c * (R1 * 128), mb, full_bar(s), 32 * c, r0);
#endif
                    }
                    __syncwarp();
                    }
                    if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == NPROD) {
        {
            constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 0, 1);
            constexpr uint32_t idesc_h = make_idesc(128, KP, 0, 1);
            int s = 0; uint32_t ph = 0; int t = 0; uint32_t tph = 0; uint32_t g = 0; uint32_t mc = 0;
            // [W_hi|W_lo] / [G_hi|G_lo] operand descriptor of stage 0; stage s, k-group kg add (s * STAGE_BYTES + kg * 1024) >> 4
            // to the low word (shared-memory addresses are < 2^18, so the 14-bit address field never carries)
            const uint64_t bd0 = make_desc(wch(0), R1 * 128, 512, 1);
            const uint32_t bd_hi = (uint32_t)(bd0 >> 32), bd_lo0 = (uint32_t)bd0;
            uint32_t soff = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                int it = 0;
                while (it < nit) {
                    const int seg_end = (it < nd) ? min(it + segc, nd) : nit;
                    const uint32_t b = g & 1u;
                    TRACE_AT(mc, 8);
                    mbar_wait(tempty_bar(b), ((g >> 1) & 1u) ^ 1u);
                    tc_fence_after();
                    const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                    bool first = true;
                    for (; it < seg_end; ++it, ++mc) {
                        TRACE_AT(mc, 5);
                        // afull(t) implies full(s): the convert warps waited on full(s) - the barrier that also counts the
                        // [W_hi|W_lo] bytes of the stage - before they filled A slot t and arrived on afull(t)
                        mbar_wait(afull_bar(t), tph);
                        TRACE_AT(mc, 6);
                        tc_fence_after();
                        const uint32_t a_hi = tmem_base + Cfg::A_COL0 + t * 64;
                        if (elect_one()) {
                            const uint32_t bl = bd_lo0 + soff;
#pragma unroll
                            for (int kg = 0; kg < R1 / 8; ++kg) {
                                const uint32_t dc = dcol + (kg % Cfg::NCHAIN) * Cfg::CHAIN_COLS;
#if !defined(PYMFB_EXP_SKIP_MMA)
                                umma_tf32_ts_lh(dc, a_hi + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_hl, (first && kg < Cfg::NCHAIN) ? 0u : 1u);
#if !defined(PYMFB_EXP_ONE_MMA)
                                umma_tf32_ts_lh(dc + KP, a_hi + 32 + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_h, 1u);
#endif
#endif
                            }
                            umma_commit(empty_bar(s));
                            umma_commit(aempty_bar(t));
                        }
                        __syncwarp();
                        TRACE_AT(mc, 7);
                        first = false;
                        soff += Cfg::STAGE_BYTES >> 4;
                        if (++s == Cfg::STAGES) { s = 0; ph ^= 1; soff = 0; }
                        if (++t == Cfg::NT) { t = 0; tph ^= 1; }
                    }
                    if (elect_one()) umma_commit(tfull_bar(b));
                    __syncwarp();
                    ++g;
                }
            }
        }
    } else if (warp < NPROD + 1 + 4 * Cfg::CONV_GROUPS) {
        // ===== convert warps: smem X tile -> registers -> hi/lo -> TMEM A ring =====
        // CONV_GROUPS groups of 4 warps take alternate stages (every waiter still sees consecutive phases of the
        // barriers it waits on: a slot's next use needs this group's own arrival first)
        const int q = warp & 3;
        const int group = (warp - (NPROD + 1)) >> 2;
        const int mylane = q * 32 + lane;                 // column of the tile = TMEM lane
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::A_COL0;
        int s = 0; uint32_t ph = 0; int t = 0; uint32_t tph = 0; uint32_t cc = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int it = 0; it < nit; ++it, ++cc) {
                if (Cfg::CONV_GROUPS > 1 && (int)(cc % Cfg::CONV_GROUPS) != group) {
                    if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                    if (++t == Cfg::NT) { t = 0; tph ^= 1; }
                    continue;
                }
                if (q == 0) TRACE_AT(cc, 2);
                mbar_wait(full_bar(s), ph);
                if (q == 0) TRACE_AT(cc, 9);
                mbar_wait(aempty_bar(t), tph ^ 1);
                if (q == 0) TRACE_AT(cc, 3);
                tc_fence_after();
#if !defined(PYMFB_EXP_SKIP_CONVERT)
                const float* xs = reinterpret_cast<const float*>(smem_gen + s * Cfg::STAGE_BYTES);
                float v[32];
#pragma unroll
                for (int r = 0; r < 32; ++r) v[r] = xs[r * TILE_COLS + mylane];
                park_hilo(lane_addr + t * 64, v);
                tmem_st_wait();
#endif
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(cc, 4);
                if (lane == 0) mbar_arrive(afull_bar(t));
                if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                if (++t == Cfg::NT) { t = 0; tph ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;
        const int nsegC = (nd + segc - 1) / segc;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            float creg[KP];
#pragma unroll
            for (int j = 0; j < KP; ++j) creg[j] = 0.f;
            // Old H of this lane's column, fetched NOW: under a saturated memory system a dependent
            // global load takes ~3 us, and doing it after the last segment stalled every tile by ~10 us.
            const int col = tile * TILE_COLS + q * 32 + lane;
            // KP = 64 sits at the register cap of this kernel (168): holding the old H column (64 values) next to
            // the 64 sums through the whole tile made the compiler spill and cost the pass 20 % once the centering
            // terms were added (same-box bisect).  LEAN: the column is pulled into L2 when the last W^T X segment
            // starts, summed (and thereby pulled into L1) while the G H MMAs are in flight, and re-read 16 values at a time.
            constexpr bool LEAN = (KP == 64);
            float hreg[LEAN ? 1 : KP];
            float xs = 0.f;
            if constexpr (!LEAN) {
#pragma unroll
                for (int j = 0; j < KP; ++j) hreg[j] = (col < n_loc) ? __ldg(Hc + (int64_t)j * ldh + col) : 0.f;
                xs = (wmean != nullptr && col < n_loc) ? __ldg(xsum + col) : 0.f;
            }
            for (int seg = 0; seg < nsegC; ++seg, ++g) {
                if constexpr (LEAN) {
                    if (seg == nsegC - 1 && col < n_loc) {
#pragma unroll 8
                        for (int j = 0; j < KP; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(Hc + (int64_t)j * ldh + col));
                        if (wmean != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(xsum + col));
                    }
                }
                const uint32_t b = g & 1u;
                if (q == 0) TRACE_AT(g * segc, 10);
                mbar_wait(tfull_bar(b), (g >> 1) & 1u);
                if (q == 0) TRACE_AT(g * segc, 11);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
#pragma unroll
                    for (int ch = 0; ch < Cfg::NCHAIN; ++ch) {
                        float hi[16], sm[16];
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + j0, hi);
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + KP + j0, sm);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) creg[j0 + j] += hi[j] + sm[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(g * segc, 12);
                if (lane == 0) mbar_arrive(tempty_bar(b));
            }
            {
                float hsum = 0.f;                     // column sum of the old H tile (for the centered G H)
                if constexpr (LEAN) {
                    if (col < n_loc) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += __ldg(Hc + (int64_t)j * ldh + col);
                        if (wmean != nullptr) xs = __ldg(xsum + col);
                    }
                } else {
                    if (wmean != nullptr) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += hreg[j];
                    }
                }
                const uint32_t b = g & 1u;
                mbar_wait(tfull_bar(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
                    float dh[16], dl[16];
                    tmem_ld16(taddr + j0, dh);
                    tmem_ld16(taddr + KP + j0, dl);
                    tmem_ld_wait();
                    if (Cfg::NCHAIN > 1) {
                        float eh[16], el[16];
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + j0, eh);
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + KP + j0, el);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) { dh[j] += eh[j]; dl[j] += el[j]; }
                    }
                    if (dbg != nullptr && tile == 0) {
                        float* o = dbg + (size_t)(q * 32 + lane) * (2 * KP) + j0;
#pragma unroll
                        for (int j = 0; j < 16; ++j) { o[j] = creg[j0 + j]; o[KP + j] = dh[j] + dl[j]; }
                    }
#if defined(PYMFB_EXP_SKIP_EPI_GLOBAL)
                    if (col < -1) {
#else
                    if (col < n_loc) {
#endif
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int64_t o = (int64_t)(j0 + j) * ldh + col;
                            float h;
                            if constexpr (LEAN) h = __ldg(Hc + o); else h = hreg[j0 + j];
                            float cj = creg[j0 + j], dj = dh[j] + dl[j];
#if !defined(PYMFB_TS_NO_CENTER)
                            if (wmean != nullptr) {
#if defined(PYMFB_MEAN_LDG)
                                cj = fmaf(__ldg(wmean + j0 + j), xs, cj);
                                dj = fmaf(__ldg(gmean + j0 + j), hsum, dj);
#else
                                cj = fmaf(s_mean[j0 + j], xs, cj);
                                dj = fmaf(s_mean[KP + j0 + j], hsum, dj);
#endif
                            }
#endif
                            const float hn = (Dp != nullptr) ? snmf_ratio(h, cj, Dp[o], Dn[o]) : mu_ratio(h, cj, dj, lam);
                            const float hh = __uint_as_float(__float_as_uint(hn) & 0xFFFFE000u);
                            Hn[o] = hn;                                  // new H
                            Hs[hs_index((j0 + j), col, 2 * KP)] = hh;        // [H_hi ; H_lo] rows for the X.H^T pass
                            Hs[hs_index(KP + (j0 + j), col, 2 * KP)] = hn - hh;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(b));
                ++g;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}

// k_h_update_ts with two producer warps and TWO MMA-issuing warps (see the comment in the MMA branch).
template <int KP>
__global__ void __launch_bounds__(TsCfg<KP>::THREADS, 1)
k_h_update_ts2w(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
              const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapG,
              const DevState* __restrict__ st, const float* __restrict__ Hc, float* __restrict__ Hn,
              float* __restrict__ Hs, int64_t ldh, int d, int n_loc, int num_tiles, float* __restrict__ dbg,
              int seg_c, float lam, const float* __restrict__ Dp, const float* __restrict__ Dn,
              const float* __restrict__ wmean, const float* __restrict__ gmean, const float* __restrict__ xsum, int xsh) {
    // wmean != nullptr: the B operands are the CENTERED W / G (k_split_hilo_centered); the epilogue adds
    // wmean[j] * (column sum of X) to W^T X and gmean[j] * (column sum of the H tile) to G H
    // Dp != nullptr: Semi-NMF (pymf/snmf.py:72-90) - the epilogue takes G+ H and G- H from Dp / Dn (same layout
    // as H, written by k_gh_posneg_simt) instead of the G H accumulator
#if !defined(PYMFB_TS_NO_CENTER)
    __shared__ float s_mean[2 * KP];          // [w_mean | g_mean]: read on the critical tail of every tile, so not from global
    if (threadIdx.x < 2 * KP)
        s_mean[threadIdx.x] = (wmean == nullptr) ? 0.f : (threadIdx.x < KP ? wmean[threadIdx.x] : gmean[threadIdx.x - KP]);
#endif
#if defined(PYMFB_TS_SEG_CONST)
    constexpr int segc = SEG_STAGES;          // A/B builds: compile-time segment length as in round 1
#else
    const int segc = seg_c;
#endif
    using Cfg = TsCfg<KP>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::STAGES + s); };
    auto afull_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + t); };
    auto aempty_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + Cfg::NT + t); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + 2 + a); };
    const uint32_t tmem_slot = bar_base + 8u * Cfg::NBAR;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::STAGES * Cfg::STAGE_BYTES + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapW); tma_prefetch_desc(&mapH); tma_prefetch_desc(&mapG);
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int t = 0; t < Cfg::NT; ++t) { mbar_init(afull_bar(t), 4); mbar_init(aempty_bar(t), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), Cfg::EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    const int nd = (d + R1 - 1) / R1;
    const int nit = nd + KP / R1;
    auto xs_addr = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };                    // [32 rows][128 cols] plain
    auto wch = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + XSTAGE_BYTES; };        // MN-major chunks

    if (warp < 2) {
        {
            int s = 0; uint32_t ph = 0; uint32_t pcnt = 0;   // this warp issues stages pcnt % 2 == warp
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int col0 = tile * TILE_COLS;
                for (int it = 0; it < nit; ++it) {
                    if (pcnt++ % 2 == (uint32_t)warp) {
                    TRACE_AT(pcnt - 1, 0);
                    mbar_wait(empty_bar(s), ph ^ 1);
                    TRACE_AT(pcnt - 1, 1);
                    if (elect_one()) {
#if defined(PYMFB_EXP_SKIP_WLOAD)
                        mbar_expect_tx(full_bar(s), XSTAGE_BYTES);
#else
                        mbar_expect_tx(full_bar(s), XSTAGE_BYTES + Cfg::BSTAGE_BYTES);
#endif
                        const bool xphase = it < nd;
                        const int r0 = (xphase ? it : it - nd) * R1;
                        tma_load_x(xs_addr(s), xphase ? &mapX : &mapH, full_bar(s), col0, r0, xphase ? xsh : kNoPanel);
#if !defined(PYMFB_EXP_SKIP_WLOAD)
                        const CUtensorMap* mb = xphase ? &mapW : &mapG;
#pragma unroll
                        for (int c = 0; c < Cfg::NCH; ++c) tma_load_2d(wch(s) + c * (R1 * 128), mb, full_bar(s), 32 * c, r0);
#endif
                    }
                    __syncwarp();
                    }
                    if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp < 4) {
        // ===== two MMA issuers, alternate stages.  tcgen05.mma issue blocks on the tensor pipe's short queue, so what ONE
        // issuing warp spends per stage on its barrier wait, commits and bookkeeping (~270 cycles) is a pipe bubble when
        // the MMAs are short (k = 64: 385 tensor cycles per stage, 560-650 measured).  Here warp `mw` owns the stages with
        // mc % 2 == mw and does that work while the other warp's MMAs are being issued; a named-barrier hand-over
        // (tcgen05.fence::before_thread_sync / bar.arrive -> bar.sync / tcgen05.fence::after_thread_sync) keeps the MMAs of
        // consecutive stages in order, so results stay bit-identical to the one-warp kernel.  Each commit tracks the issuing
        // thread's own MMAs; the pipe completes MMAs in issue order, so a stage's commit also covers the earlier stages.
        {
            static_assert(Cfg::NT % 2 == 0, "each A slot must always belong to the same MMA warp (consecutive barrier phases)");
            const uint32_t mw = (uint32_t)(warp - 2);
            constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 0, 1);
            constexpr uint32_t idesc_h = make_idesc(128, KP, 0, 1);
            int s = 0; uint32_t ph = 0; int t = 0; uint32_t tph = 0; uint32_t g = 0; uint32_t mc = 0;
            const uint64_t bd0 = make_desc(wch(0), R1 * 128, 512, 1);
            const uint32_t bd_hi = (uint32_t)(bd0 >> 32), bd_lo0 = (uint32_t)bd0;
            uint32_t soff = 0;
            const uint32_t my_tiles = (uint32_t)((num_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x);
            const uint32_t total = my_tiles * (uint32_t)nit;      // stages of this CTA (the last one hands over to nobody)
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                int it = 0;
                while (it < nit) {
                    const int seg_end = (it < nd) ? min(it + segc, nd) : nit;
                    const uint32_t b = g & 1u;
                    const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                    bool first = true;
                    for (; it < seg_end; ++it, ++mc) {
                        if ((mc & 1u) == mw) {
                            TRACE_AT(mc, 5);
                            if (first) mbar_wait(tempty_bar(b), ((g >> 1) & 1u) ^ 1u);     // the segment's accumulator has been drained
                            // afull(t) implies full(s) (see k_h_update_ts)
                            mbar_wait(afull_bar(t), tph);
                            TRACE_AT(mc, 6);
                            if (mc > 0) asm volatile("bar.sync %0, 64;" ::"r"(1 + (int)mw) : "memory");   // stage mc - 1 has been issued
                            tc_fence_after();
                            const uint32_t a_hi = tmem_base + Cfg::A_COL0 + t * 64;
                            if (elect_one()) {
                                const uint32_t bl = bd_lo0 + soff;
#pragma unroll
                                for (int kg = 0; kg < R1 / 8; ++kg) {
                                    const uint32_t dc = dcol + (kg % Cfg::NCHAIN) * Cfg::CHAIN_COLS;
                                    umma_tf32_ts_lh(dc, a_hi + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_hl, (first && kg < Cfg::NCHAIN) ? 0u : 1u);
                                    umma_tf32_ts_lh(dc + KP, a_hi + 32 + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_h, 1u);
                                }
                            }
                            __syncwarp();
                            tc_fence_before();
                            if (mc + 1 < total) asm volatile("bar.arrive %0, 64;" ::"r"(1 + (int)(mw ^ 1u)) : "memory");
                            if (elect_one()) {
                                umma_commit(empty_bar(s));
                                umma_commit(aempty_bar(t));
                                if (it + 1 == seg_end) umma_commit(tfull_bar(b));
                            }
                            __syncwarp();
                            TRACE_AT(mc, 7);
                        }
                        first = false;
                        soff += Cfg::STAGE_BYTES >> 4;
                        if (++s == Cfg::STAGES) { s = 0; ph ^= 1; soff = 0; }
                        if (++t == Cfg::NT) { t = 0; tph ^= 1; }
                    }
                    ++g;
                }
            }
            (void)ph;
        }
    } else if (warp < NPROD + 1 + 4 * Cfg::CONV_GROUPS) {
        // ===== convert warps: smem X tile -> registers -> hi/lo -> TMEM A ring =====
        // CONV_GROUPS groups of 4 warps take alternate stages (every waiter still sees consecutive phases of the
        // barriers it waits on: a slot's next use needs this group's own arrival first)
        const int q = warp & 3;
        const int group = (warp - (NPROD + 1)) >> 2;
        const int mylane = q * 32 + lane;                 // column of the tile = TMEM lane
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::A_COL0;
        int s = 0; uint32_t ph = 0; int t = 0; uint32_t tph = 0; uint32_t cc = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int it = 0; it < nit; ++it, ++cc) {
                if (Cfg::CONV_GROUPS > 1 && (int)(cc % Cfg::CONV_GROUPS) != group) {
                    if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                    if (++t == Cfg::NT) { t = 0; tph ^= 1; }
                    continue;
                }
                if (q == 0) TRACE_AT(cc, 2);
                mbar_wait(full_bar(s), ph);
                if (q == 0) TRACE_AT(cc, 9);
                mbar_wait(aempty_bar(t), tph ^ 1);
                if (q == 0) TRACE_AT(cc, 3);
                tc_fence_after();
#if !defined(PYMFB_EXP_SKIP_CONVERT)
                const float* xs = reinterpret_cast<const float*>(smem_gen + s * Cfg::STAGE_BYTES);
                float v[32];
#pragma unroll
                for (int r = 0; r < 32; ++r) v[r] = xs[r * TILE_COLS + mylane];
                park_hilo(lane_addr + t * 64, v);
                tmem_st_wait();
#endif
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(cc, 4);
                if (lane == 0) mbar_arrive(afull_bar(t));
                if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
                if (++t == Cfg::NT) { t = 0; tph ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;
        const int nsegC = (nd + segc - 1) / segc;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            float creg[KP];
#pragma unroll
            for (int j = 0; j < KP; ++j) creg[j] = 0.f;
            // Old H of this lane's column, fetched NOW: under a saturated memory system a dependent
            // global load takes ~3 us, and doing it after the last segment stalled every tile by ~10 us.
            const int col = tile * TILE_COLS + q * 32 + lane;
            // KP = 64 sits at the register cap of this kernel (168): holding the old H column (64 values) next to
            // the 64 sums through the whole tile made the compiler spill and cost the pass 20 % once the centering
            // terms were added (same-box bisect).  LEAN: the column is pulled into L2 when the last W^T X segment
            // starts, summed (and thereby pulled into L1) while the G H MMAs are in flight, and re-read 16 values at a time.
            constexpr bool LEAN = (KP == 64);
            float hreg[LEAN ? 1 : KP];
            float xs = 0.f;
            if constexpr (!LEAN) {
#pragma unroll
                for (int j = 0; j < KP; ++j) hreg[j] = (col < n_loc) ? __ldg(Hc + (int64_t)j * ldh + col) : 0.f;
                xs = (wmean != nullptr && col < n_loc) ? __ldg(xsum + col) : 0.f;
            }
            for (int seg = 0; seg < nsegC; ++seg, ++g) {
                if constexpr (LEAN) {
                    if (seg == nsegC - 1 && col < n_loc) {
#pragma unroll 8
                        for (int j = 0; j < KP; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(Hc + (int64_t)j * ldh + col));
                        if (wmean != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(xsum + col));
                    }
                }
                const uint32_t b = g & 1u;
                if (q == 0) TRACE_AT(g * segc, 10);
                mbar_wait(tfull_bar(b), (g >> 1) & 1u);
                if (q == 0) TRACE_AT(g * segc, 11);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
#pragma unroll
                    for (int ch = 0; ch < Cfg::NCHAIN; ++ch) {
                        float hi[16], sm[16];
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + j0, hi);
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + KP + j0, sm);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) creg[j0 + j] += hi[j] + sm[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(g * segc, 12);
                if (lane == 0) mbar_arrive(tempty_bar(b));
            }
            {
                float hsum = 0.f;                     // column sum of the old H tile (for the centered G H)
                if constexpr (LEAN) {
                    if (col < n_loc) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += __ldg(Hc + (int64_t)j * ldh + col);
                        if (wmean != nullptr) xs = __ldg(xsum + col);
                    }
                } else {
                    if (wmean != nullptr) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += hreg[j];
                    }
                }
                const uint32_t b = g & 1u;
                mbar_wait(tfull_bar(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
                    float dh[16], dl[16];
                    tmem_ld16(taddr + j0, dh);
                    tmem_ld16(taddr + KP + j0, dl);
                    tmem_ld_wait();
                    if (Cfg::NCHAIN > 1) {
                        float eh[16], el[16];
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + j0, eh);
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + KP + j0, el);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) { dh[j] += eh[j]; dl[j] += el[j]; }
                    }
                    if (dbg != nullptr && tile == 0) {
                        float* o = dbg + (size_t)(q * 32 + lane) * (2 * KP) + j0;
#pragma unroll
                        for (int j = 0; j < 16; ++j) { o[j] = creg[j0 + j]; o[KP + j] = dh[j] + dl[j]; }
                    }
#if defined(PYMFB_EXP_SKIP_EPI_GLOBAL)
                    if (col < -1) {
#else
                    if (col < n_loc) {
#endif
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int64_t o = (int64_t)(j0 + j) * ldh + col;
                            float h;
                            if constexpr (LEAN) h = __ldg(Hc + o); else h = hreg[j0 + j];
                            float cj = creg[j0 + j], dj = dh[j] + dl[j];
#if !defined(PYMFB_TS_NO_CENTER)
                            if (wmean != nullptr) {
#if defined(PYMFB_MEAN_LDG)
                                cj = fmaf(__ldg(wmean + j0 + j), xs, cj);
                                dj = fmaf(__ldg(gmean + j0 + j), hsum, dj);
#else
                                cj = fmaf(s_mean[j0 + j], xs, cj);
                                dj = fmaf(s_mean[KP + j0 + j], hsum, dj);
#endif
                            }
#endif
                            const float hn = (Dp != nullptr) ? snmf_ratio(h, cj, Dp[o], Dn[o]) : mu_ratio(h, cj, dj, lam);
                            const float hh = __uint_as_float(__float_as_uint(hn) & 0xFFFFE000u);
                            Hn[o] = hn;                                  // new H
                            Hs[hs_index((j0 + j), col, 2 * KP)] = hh;        // [H_hi ; H_lo] rows for the X.H^T pass
                            Hs[hs_index(KP + (j0 + j), col, 2 * KP)] = hn - hh;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(b));
                ++g;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}

// ---------------------------------------------------------------------------------------------
// TS H-update, RS rows per stage (round 2b).  What the commit / MMA-group probe (tests/commit_probe.cu) and the
// PYMFB_TRACE timeline say about the 32-row kernel above at k = 64: its 8 MMAs per stage are short (64 + 32 tensor
// cycles per k-step), tcgen05.mma issue blocks on a shallow queue, so the ~300 cycles the MMA warp spends per stage on
// its barrier wait, two commits and loop bookkeeping are NOT hidden behind tensor work: 560-650 cycles per stage
// against 385 of tensor time.  This variant halves that overhead per byte: a stage is RS = 64 rows (16 MMAs per wait),
// and ONE tcgen05.commit per stage (done[s]) frees the X / operand slot and - NT stages later - the TMEM A slot that
// the convert warps wait for (DoneLag), instead of separate empty / aempty commits.
// ---------------------------------------------------------------------------------------------
#ifndef PYMFB_TSR_CONV_GROUPS
#define PYMFB_TSR_CONV_GROUPS 2
#endif
template <int KP, int RS>
struct TsrCfg {
    static constexpr int NCH = 2 * KP / 32;
    static constexpr int XS_BYTES = TILE_COLS * RS * 4;             // plain [RS rows][128 cols]
    static constexpr int BSTAGE_BYTES = NCH * RS * 128;             // [b_hi | b_lo] chunks, RS rows each
    static constexpr int STAGE_BYTES = XS_BYTES + BSTAGE_BYTES;
    static constexpr int STAGES_RAW = (SMEM_LIMIT - 2048) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_RAW > 8 ? 8 : STAGES_RAW;
    static constexpr int NCHAIN = (KP == 32) ? PYMFB_NCHAIN : 1;
    static constexpr int CHAIN_COLS = 2 * KP;
    static constexpr int SEG_COLS = CHAIN_COLS * NCHAIN;
    static constexpr int A_COL0 = 2 * SEG_COLS;
    static constexpr int ASLOT_COLS = 2 * RS;                       // RS hi columns then RS lo columns
    static constexpr int NT_RAW = (512 - A_COL0) / ASLOT_COLS;
    static constexpr int NT = NT_RAW > STAGES ? STAGES : (NT_RAW > 6 ? 6 : NT_RAW);
    static constexpr int EPI_WARPS = 4;
    // Convert-warp groups (4 warps each) taking alternate stages.  PYMFB_TRACE of the one-group kernel with 64-row stages at
    // k = 32: the group needs 545 cycles per stage + ~300 of waits, the MMA warp 470 + ~180 - the converts bound the
    // per-SM rate.  A group only sees every CG-th phase of the barriers it waits on, so the ring depth must be a multiple
    // of CG (a parity wait that skips a phase can alias).
    static constexpr int CG = (RS == 64 && STAGES % 2 == 0) ? PYMFB_TSR_CONV_GROUPS : 1;
    static constexpr int THREADS = 32 * (NPROD + 1 + 4 * CG + EPI_WARPS);
    static constexpr int NBAR = 2 * STAGES + NT + 4;                // full, done, afull, tfull[2], tempty[2]
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 512;
    static_assert(KP == 32 || KP == 64, "TS kernels serve KP = 32 and 64");
    static_assert(RS == 32 || RS == 64, "32 or 64 rows per stage");
    static_assert(NT >= 2 && NT <= STAGES, "A ring depth");
    static_assert(STAGES >= 2, "stage ring depth");
    static_assert(NBAR * 8 + 8 <= 512, "barrier area too small");
    static_assert(SMEM_BYTES <= SMEM_LIMIT, "stage ring does not fit");
};

// hi/lo of 32 values -> TMEM (this thread's lane): hi at columns hi_addr.., lo at lo_addr..
__device__ __forceinline__ void park_hilo_at(uint32_t hi_addr, uint32_t lo_addr, const float (&v)[32]) {
    uint32_t hi[32], lo[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        hi[i] = __float_as_uint(v[i]) & 0xFFFFE000u;
        lo[i] = __float_as_uint(v[i] - __uint_as_float(hi[i]));
    }
    tmem_st32(hi_addr, hi);
    tmem_st32(lo_addr, lo);
}

template <int KP, int RS>
__global__ void __launch_bounds__(TsrCfg<KP, RS>::THREADS, 1)
k_h_update_tsr(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapW,
               const __grid_constant__ CUtensorMap mapH, const __grid_constant__ CUtensorMap mapG,
               const DevState* __restrict__ st, const float* __restrict__ Hc, float* __restrict__ Hn,
               float* __restrict__ Hs, int64_t ldh, int d, int n_loc, int num_tiles, float* __restrict__ dbg,
               int seg_c, float lam, const float* __restrict__ Dp, const float* __restrict__ Dn,
               const float* __restrict__ wmean, const float* __restrict__ gmean, const float* __restrict__ xsum, int xsh) {
    // same contract as k_h_update_ts; seg_c counts stages of RS rows; the boxes of mapX / mapH are 128 columns x RS
    // rows, those of mapW / mapG 32 columns x RS rows (rows beyond the matrix read as zero)
#if !defined(PYMFB_TS_NO_CENTER)
    __shared__ float s_mean[2 * KP];          // [w_mean | g_mean]: read on the critical tail of every tile, so not from global
    if (threadIdx.x < 2 * KP)
        s_mean[threadIdx.x] = (wmean == nullptr) ? 0.f : (threadIdx.x < KP ? wmean[threadIdx.x] : gmean[threadIdx.x - KP]);
#endif
    const int segc = seg_c;
    using Cfg = TsrCfg<KP, RS>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
    struct Bars {
        uint32_t base;
        __device__ __forceinline__ uint32_t full(int s) const { return base + 8u * s; }
        __device__ __forceinline__ uint32_t done(int s) const { return base + 8u * (Cfg::STAGES + s); }
        __device__ __forceinline__ uint32_t afull(int t) const { return base + 8u * (2 * Cfg::STAGES + t); }
        __device__ __forceinline__ uint32_t tfull(int a) const { return base + 8u * (2 * Cfg::STAGES + Cfg::NT + a); }
        __device__ __forceinline__ uint32_t tempty(int a) const { return base + 8u * (2 * Cfg::STAGES + Cfg::NT + 2 + a); }
    };
    const Bars bar{bar_base};
    auto bar_tfull = [&](int a) { return bar.tfull(a); };
    auto bar_tempty = [&](int a) { return bar.tempty(a); };
    const uint32_t tmem_slot = bar_base + 8u * Cfg::NBAR;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::STAGES * Cfg::STAGE_BYTES + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapW); tma_prefetch_desc(&mapH); tma_prefetch_desc(&mapG);
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(bar.full(s), 1); mbar_init(bar.done(s), 1); }
        for (int t = 0; t < Cfg::NT; ++t) mbar_init(bar.afull(t), 4);
        for (int a = 0; a < 2; ++a) { mbar_init(bar.tfull(a), 1); mbar_init(bar.tempty(a), Cfg::EPI_WARPS); }
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    const int nd = (d + RS - 1) / RS;
    const int nit = nd + (KP + RS - 1) / RS;
    auto xs_addr = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };                    // [RS rows][128 cols] plain
    auto wch = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + Cfg::XS_BYTES; };       // MN-major chunks

    if (warp < NPROD) {
        RingPos<Cfg::STAGES> rs;
        uint32_t pcnt = 0;                               // this warp issues stages pcnt % NPROD == warp
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int col0 = tile * TILE_COLS;
            for (int it = 0; it < nit; ++it) {
                if (pcnt++ % NPROD == (uint32_t)warp) {
                    TRACE_AT(pcnt - 1, 0);
                    mbar_wait(bar.done(rs.s), rs.ph ^ 1);
                    TRACE_AT(pcnt - 1, 1);
                    if (elect_one()) {
                        mbar_expect_tx(bar.full(rs.s), Cfg::XS_BYTES + Cfg::BSTAGE_BYTES);
                        const bool xphase = it < nd;
                        const int r0 = (xphase ? it : it - nd) * RS;
                        tma_load_x(xs_addr(rs.s), xphase ? &mapX : &mapH, bar.full(rs.s), col0, r0, xphase ? xsh : kNoPanel);
                        const CUtensorMap* mb = xphase ? &mapW : &mapG;
#pragma unroll
                        for (int c = 0; c < Cfg::NCH; ++c) tma_load_2d(wch(rs.s) + c * (RS * 128), mb, bar.full(rs.s), 32 * c, r0);
                    }
                    __syncwarp();
                }
                rs.next();
            }
        }
    } else if (warp == NPROD) {
        constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 0, 1);
        constexpr uint32_t idesc_h = make_idesc(128, KP, 0, 1);
        RingPos<Cfg::STAGES> rs; RingPos<Cfg::NT> rt;
        uint32_t g = 0, mc = 0; (void)mc;
        // [W_hi|W_lo] / [G_hi|G_lo] operand descriptor of stage 0; stage s, k-group kg add (s * STAGE_BYTES + kg * 1024) >> 4
        // to the low word (shared-memory addresses are < 2^18, so the 14-bit address field never carries)
        const uint64_t bd0 = make_desc(wch(0), RS * 128, 512, 1);
        const uint32_t bd_hi = (uint32_t)(bd0 >> 32), bd_lo0 = (uint32_t)bd0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            int it = 0;
            while (it < nit) {
                const int seg_end = (it < nd) ? min(it + segc, nd) : nit;
                const uint32_t b = g & 1u;
                mbar_wait(bar.tempty(b), ((g >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                bool first = true;
                for (; it < seg_end; ++it, ++mc) {
                    TRACE_AT(mc, 5);
                    // afull(t) implies full(s): the convert warps waited on full(s) - the barrier that also counts the
                    // [W_hi|W_lo] bytes of the stage - before they filled A slot t and arrived on afull(t)
                    mbar_wait(bar.afull(rt.s), rt.ph);
                    TRACE_AT(mc, 6);
                    tc_fence_after();
                    const uint32_t a_hi = tmem_base + Cfg::A_COL0 + rt.s * Cfg::ASLOT_COLS;
                    if (elect_one()) {
                        const uint32_t bl = bd_lo0 + rs.s * (Cfg::STAGE_BYTES >> 4);
#pragma unroll
                        for (int kg = 0; kg < RS / 8; ++kg) {
                            const uint32_t dc = dcol + (kg % Cfg::NCHAIN) * Cfg::CHAIN_COLS;
                            umma_tf32_ts_lh(dc, a_hi + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_hl, (first && kg < Cfg::NCHAIN) ? 0u : 1u);
                            umma_tf32_ts_lh(dc + KP, a_hi + RS + kg * 8, bl + kg * (1024 >> 4), bd_hi, idesc_h, 1u);
                        }
                        TRACE_AT(mc, 14);
                        umma_commit(bar.done(rs.s));                          // frees the stage and (NT stages on) its A slot
                        if (it + 1 == seg_end) umma_commit(bar.tfull(b));
                    }
                    __syncwarp();
                    TRACE_AT(mc, 7);
                    first = false;
                    rs.next(); rt.next();
                }
                ++g;
            }
        }
    } else if (warp < NPROD + 1 + 4 * Cfg::CG) {
        // ===== convert warps: smem X tile -> registers -> hi/lo -> TMEM A ring (CG groups take alternate stages) =====
        const int q = warp & 3;
        const int group = (warp - (NPROD + 1)) >> 2;
        const int mylane = q * 32 + lane;                 // column of the tile = TMEM lane
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::A_COL0;
        RingPos<Cfg::STAGES> rs; RingPos<Cfg::NT> rt;
        DoneLag<Cfg::STAGES, Cfg::NT> lag;
        uint32_t cc = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            for (int it = 0; it < nit; ++it, ++cc) {
                const bool mine = Cfg::CG == 1 || (int)(cc % Cfg::CG) == group;
                if (!mine) { lag.wait(bar, false); rs.next(); rt.next(); continue; }
                if (q == 0) TRACE_AT(cc, 2);
                mbar_wait(bar.full(rs.s), rs.ph);
                if (q == 0) TRACE_AT(cc, 9);
                lag.wait(bar);                            // the MMAs that read this A slot NT stages ago have completed
                if (q == 0) TRACE_AT(cc, 3);
                tc_fence_after();
                const float* xs = reinterpret_cast<const float*>(smem_gen + rs.s * Cfg::STAGE_BYTES);
                const uint32_t slot = lane_addr + rt.s * Cfg::ASLOT_COLS;
#pragma unroll
                for (int h = 0; h < RS / 32; ++h) {
                    float v[32];
#pragma unroll
                    for (int r = 0; r < 32; ++r) v[r] = xs[(h * 32 + r) * TILE_COLS + mylane];
                    park_hilo_at(slot + h * 32, slot + RS + h * 32, v);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(cc, 4);
                if (lane == 0) mbar_arrive(bar.afull(rt.s));
                rs.next(); rt.next();
            }
        }
    } else {
        const int q = warp & 3;
        const int nsegC = (nd + segc - 1) / segc;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            float creg[KP];
#pragma unroll
            for (int j = 0; j < KP; ++j) creg[j] = 0.f;
            // Old H of this lane's column, fetched NOW: under a saturated memory system a dependent
            // global load takes ~3 us, and doing it after the last segment stalled every tile by ~10 us.
            const int col = tile * TILE_COLS + q * 32 + lane;
            // KP = 64 sits at the register cap of this kernel (168): holding the old H column (64 values) next to
            // the 64 sums through the whole tile made the compiler spill and cost the pass 20 % once the centering
            // terms were added (same-box bisect).  LEAN: the column is pulled into L2 when the last W^T X segment
            // starts, summed (and thereby pulled into L1) while the G H MMAs are in flight, and re-read 16 values at a time.
            constexpr bool LEAN = (KP == 64);
            float hreg[LEAN ? 1 : KP];
            float xs = 0.f;
            if constexpr (!LEAN) {
#pragma unroll
                for (int j = 0; j < KP; ++j) hreg[j] = (col < n_loc) ? __ldg(Hc + (int64_t)j * ldh + col) : 0.f;
                xs = (wmean != nullptr && col < n_loc) ? __ldg(xsum + col) : 0.f;
            }
            for (int seg = 0; seg < nsegC; ++seg, ++g) {
                if constexpr (LEAN) {
                    if (seg == nsegC - 1 && col < n_loc) {
#pragma unroll 8
                        for (int j = 0; j < KP; ++j) asm volatile("prefetch.global.L2 [%0];" ::"l"(Hc + (int64_t)j * ldh + col));
                        if (wmean != nullptr) asm volatile("prefetch.global.L2 [%0];" ::"l"(xsum + col));
                    }
                }
                const uint32_t b = g & 1u;
                if (q == 0) TRACE_AT(g * segc, 10);
                mbar_wait(bar_tfull(b), (g >> 1) & 1u);
                if (q == 0) TRACE_AT(g * segc, 11);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
#pragma unroll
                    for (int ch = 0; ch < Cfg::NCHAIN; ++ch) {
                        float hi[16], sm[16];
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + j0, hi);
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + KP + j0, sm);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) creg[j0 + j] += hi[j] + sm[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (q == 0) TRACE_AT(g * segc, 12);
                if (lane == 0) mbar_arrive(bar_tempty(b));
            }
            {
                float hsum = 0.f;                     // column sum of the old H tile (for the centered G H)
                if constexpr (LEAN) {
                    if (col < n_loc) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += __ldg(Hc + (int64_t)j * ldh + col);
                        if (wmean != nullptr) xs = __ldg(xsum + col);
                    }
                } else {
                    if (wmean != nullptr) {
#pragma unroll
                        for (int j = 0; j < KP; ++j) hsum += hreg[j];
                    }
                }
                const uint32_t b = g & 1u;
                mbar_wait(bar_tfull(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
                    float dh[16], dl[16];
                    tmem_ld16(taddr + j0, dh);
                    tmem_ld16(taddr + KP + j0, dl);
                    tmem_ld_wait();
                    if (Cfg::NCHAIN > 1) {
                        float eh[16], el[16];
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + j0, eh);
                        tmem_ld16(taddr + Cfg::CHAIN_COLS + KP + j0, el);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) { dh[j] += eh[j]; dl[j] += el[j]; }
                    }
                    if (dbg != nullptr && tile == 0) {
                        float* o = dbg + (size_t)(q * 32 + lane) * (2 * KP) + j0;
#pragma unroll
                        for (int j = 0; j < 16; ++j) { o[j] = creg[j0 + j]; o[KP + j] = dh[j] + dl[j]; }
                    }
#if defined(PYMFB_EXP_SKIP_EPI_GLOBAL)
                    if (col < -1) {
#else
                    if (col < n_loc) {
#endif
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int64_t o = (int64_t)(j0 + j) * ldh + col;
                            float h;
                            if constexpr (LEAN) h = __ldg(Hc + o); else h = hreg[j0 + j];
                            float cj = creg[j0 + j], dj = dh[j] + dl[j];
#if !defined(PYMFB_TS_NO_CENTER)
                            if (wmean != nullptr) {
#if defined(PYMFB_MEAN_LDG)
                                cj = fmaf(__ldg(wmean + j0 + j), xs, cj);
                                dj = fmaf(__ldg(gmean + j0 + j), hsum, dj);
#else
                                cj = fmaf(s_mean[j0 + j], xs, cj);
                                dj = fmaf(s_mean[KP + j0 + j], hsum, dj);
#endif
                            }
#endif
                            const float hn = (Dp != nullptr) ? snmf_ratio(h, cj, Dp[o], Dn[o]) : mu_ratio(h, cj, dj, lam);
                            const float hh = __uint_as_float(__float_as_uint(hn) & 0xFFFFE000u);
                            Hn[o] = hn;                                  // new H
                            Hs[hs_index((j0 + j), col, 2 * KP)] = hh;        // [H_hi ; H_lo] rows for the X.H^T pass
                            Hs[hs_index(KP + (j0 + j), col, 2 * KP)] = hn - hh;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_tempty(b));
                ++g;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}


constexpr int X_CONV_GROUPS = 2;                          // convert-warp groups of the X.H^T pass (alternate stages)
constexpr int X_THREADS = 32 * (NPROD + 1 + 4 * X_CONV_GROUPS + 4);

// X H^T pass, TS variant.  Tasks [0, x_tasks): (128-row block of X, column range) -> P_A += X H^T.
// Tasks [x_tasks, num_tasks): column ranges of H itself as the A operand -> P_B += H H^T (same code,
// rows >= k are zero-filled by TMA).  B operand = [H_hi ; H_lo] rows, pre-split by the H-update
// epilogue (or k_split_rows), so the convert warps only touch X.  Two groups of 4 convert warps take
// alternate stages (the single group was ~75 % busy and the critical path of this pass).
template <int KP>
__global__ void __launch_bounds__(X_THREADS, 1)
k_xht_ts(const __grid_constant__ CUtensorMap mapX, const __grid_constant__ CUtensorMap mapHs,
         const __grid_constant__ CUtensorMap mapHA, const DevState* __restrict__ st,
         float* __restrict__ PA, float* __restrict__ PB, int d, int n_loc,
         int cols_per_task, int num_rb, int x_tasks, int hh_cols_per_task, int num_tasks,
         float* __restrict__ dbg, float* __restrict__ PpartA, float* __restrict__ PpartB, int xsh, int xrev) {
    // PpartA != nullptr: deterministic combine of the column splits (see k_xht_tc): copies of A are d * KP floats
    // apart, copies of B = H H^T (one per H H^T task) KP * KP floats; k_sum_copies then writes P.
    using Cfg = TsCfg<KP>;
    if (st->stop) return;
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
    const uint32_t bar_base = smem_base + Cfg::STAGES * Cfg::STAGE_BYTES;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::STAGES + s); };
    auto afull_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + t); };
    auto aempty_bar = [&](int t) { return bar_base + 8u * (2 * Cfg::STAGES + Cfg::NT + t); };
    auto tfull_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + a); };
    auto tempty_bar = [&](int a) { return bar_base + 8u * (2 * Cfg::STAGES + 2 * Cfg::NT + 2 + a); };
    const uint32_t tmem_slot = bar_base + 8u * Cfg::NBAR;
    volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Cfg::STAGES * Cfg::STAGE_BYTES + 8 * Cfg::NBAR);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int EPI_WARP0 = NPROD + 1 + 4 * X_CONV_GROUPS;
    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&mapX); tma_prefetch_desc(&mapHs); tma_prefetch_desc(&mapHA);
        for (int s = 0; s < Cfg::STAGES; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
        for (int t = 0; t < Cfg::NT; ++t) { mbar_init(afull_bar(t), 4); mbar_init(aempty_bar(t), 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), 4); }
        fence_barrier_init();
    }
    if (warp == NPROD) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_gen;

    auto xs_addr = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES; };                  // [128 rows][128 B] SW128
    auto hch = [&](int s) { return smem_base + s * Cfg::STAGE_BYTES + XSTAGE_BYTES; };      // [2KP rows][128 B] SW128
    // task -> (first column, number of 32-column stages, first row, is H H^T task)
    auto task_info = [&](int task, int& c_begin, int& row0, bool& hh) {
        hh = task >= x_tasks;
        int cpt, cs;
        if (hh) { cs = task - x_tasks; cpt = hh_cols_per_task; row0 = 0; }
        else { cs = xrev ? (x_tasks / num_rb - 1 - task / num_rb) : task / num_rb; cpt = cols_per_task; row0 = (task % num_rb) * 128; }   // xrev: see k_xht_tc
        c_begin = cs * cpt;
        const int c_end = min(n_loc, c_begin + cpt);
        return (c_end - c_begin + 31) / 32;
    };

    if (warp < NPROD) {
        // No L2 priorities here (unlike k_xht_tc): X evict_first measured neutral, [H_hi ; H_lo] evict_last slower
        // (cfg5 13.5 -> 13.8 ms, cfg4 k = 64 3.30 -> 3.35 ms per pass; profiles/xht_splits.json, profiles/xht_splits_ts.json)
        int s = 0; uint32_t ph = 0; uint32_t pcnt = 0;   // this warp issues stages pcnt % NPROD == warp
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin, row0; bool hh;
            const int nch = task_info(task, c_begin, row0, hh);
            const CUtensorMap* ma = hh ? &mapHA : &mapX;
            for (int ch = 0; ch < nch; ++ch) {
                if (pcnt++ % NPROD == (uint32_t)warp) {
                    mbar_wait(empty_bar(s), ph ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(full_bar(s), XSTAGE_BYTES + 2 * KP * 128);
                    tma_load_x(xs_addr(s), ma, full_bar(s), c_begin + 32 * ch, row0, hh ? kNoPanel : xsh);
                    tma_load_2d(hch(s), &mapHs, full_bar(s), 0, ((c_begin >> 5) + ch) * (2 * KP));
                }
                __syncwarp();
                    }
                if (++s == Cfg::STAGES) { s = 0; ph ^= 1; }
            }
        }
    } else if (warp == NPROD) {
        constexpr uint32_t idesc_hl = make_idesc(128, 2 * KP, 0, 0);
        constexpr uint32_t idesc_h = make_idesc(128, KP, 0, 0);
        int s = 0; uint32_t ph = 0; int t = 0; uint32_t tph = 0; uint32_t g = 0;
        // [H_hi;H_lo] operand descriptor of stage 0; stage s / k-step ks add (s * STAGE_BYTES + ks * 32) >> 4 to the low word
        const uint64_t hd0 = make_desc(hch(0), 16, 1024);
        const uint32_t hd_hi = (uint32_t)(hd0 >> 32), hd_lo0 = (uint32_t)hd0;
        uint32_t soff = 0;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin, row0; bool hh;
            const int nch = task_info(task, c_begin, row0, hh);
            int ch = 0;
            while (ch < nch) {
                const int seg_end = min(ch + SEG_STAGES, nch);
                const uint32_t b = g & 1u;
                mbar_wait(tempty_bar(b), ((g >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t dcol = tmem_base + b * Cfg::SEG_COLS;
                bool first = true;
                for (; ch < seg_end; ++ch) {
                    mbar_wait(afull_bar(t), tph);       // implies full(s), see k_h_update_ts
                    tc_fence_after();
                    const uint32_t a_hi = tmem_base + Cfg::A_COL0 + t * 64;
                    if (elect_one()) {
                        const uint32_t bl = hd_lo0 + soff;
#pragma unroll
                        for (int ks = 0; ks < 4; ++ks) {
                            const uint32_t dc = dcol + (ks % Cfg::NCHAIN) * Cfg::CHAIN_COLS;
                            umma_tf32_ts_lh(dc, a_hi + ks * 8, bl + ks * (32 >> 4), hd_hi, idesc_hl, (first && ks < Cfg::NCHAIN) ? 0u : 1u);
                            umma_tf32_ts_lh(dc + KP, a_hi + 32 + ks * 8, bl + ks * (32 >> 4), hd_hi, idesc_h, 1u);
                        }
                        umma_commit(empty_bar(s));
                        umma_commit(aempty_bar(t));
                    }
                    __syncwarp();
                    first = false;
                    soff += Cfg::STAGE_BYTES >> 4;
                    if (++s == Cfg::STAGES) { s = 0; ph ^= 1; soff = 0; }
                    if (++t == Cfg::NT) { t = 0; tph ^= 1; }
                }
                if (elect_one()) umma_commit(tfull_bar(b));
                __syncwarp();
                ++g;
            }
        }
    } else if (warp < EPI_WARP0) {
        // convert warps: thread <-> row of the X block (TMEM lane); reads its 128 B row (SW128: 16 B
        // chunk j sits at (j ^ (row & 7))), splits in registers, parks hi/lo in the TMEM A ring.
        const int q = warp & 3;
        const int group = (warp - (NPROD + 1)) >> 2;
        const int myrow = q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + Cfg::A_COL0;
        uint32_t c = 0;                                     // stage counter of this CTA
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin, row0; bool hh;
            const int nch = task_info(task, c_begin, row0, hh);
            for (int ch = 0; ch < nch; ++ch, ++c) {
                if ((int)(c % X_CONV_GROUPS) != group) continue;
                const int s = (int)(c % Cfg::STAGES), t = (int)(c % Cfg::NT);
                const uint32_t ph = (c / Cfg::STAGES) & 1u, tph = (c / Cfg::NT) & 1u;
                mbar_wait(full_bar(s), ph);
                mbar_wait(aempty_bar(t), tph ^ 1);
                tc_fence_after();
                const uint8_t* rowp = smem_gen + s * Cfg::STAGE_BYTES + myrow * 128;
                float v[32];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float4 f = *reinterpret_cast<const float4*>(rowp + ((j ^ (myrow & 7)) << 4));
                    v[4 * j + 0] = f.x; v[4 * j + 1] = f.y; v[4 * j + 2] = f.z; v[4 * j + 3] = f.w;
                }
                park_hilo(lane_addr + t * 64, v);
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(afull_bar(t));
            }
        }
    } else {
        const int q = warp & 3;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t g = 0;
        for (int task = blockIdx.x; task < num_tasks; task += gridDim.x) {
            int c_begin, row0; bool hh;
            const int nch = task_info(task, c_begin, row0, hh);
            const int nseg = (nch + SEG_STAGES - 1) / SEG_STAGES;
            float areg[KP];
#pragma unroll
            for (int j = 0; j < KP; ++j) areg[j] = 0.f;
            for (int seg = 0; seg < nseg; ++seg, ++g) {
                const uint32_t b = g & 1u;
                mbar_wait(tfull_bar(b), (g >> 1) & 1u);
                tc_fence_after();
                const uint32_t taddr = lane_addr + b * Cfg::SEG_COLS;
#pragma unroll
                for (int j0 = 0; j0 < KP; j0 += 16) {
#pragma unroll
                    for (int ch = 0; ch < Cfg::NCHAIN; ++ch) {
                        float hi[16], sm[16];
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + j0, hi);
                        tmem_ld16(taddr + ch * Cfg::CHAIN_COLS + KP + j0, sm);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; ++j) areg[j0 + j] += hi[j] + sm[j];
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty_bar(b));
            }
            const int row = row0 + q * 32 + lane;
            if (dbg != nullptr && task == 0) {
                float* o = dbg + (size_t)(q * 32 + lane) * KP;
#pragma unroll
                for (int j = 0; j < KP; ++j) o[j] = areg[j];
            }
            if (row < (hh ? KP : d)) {
                if (PpartA == nullptr) {
                    float* dst = (hh ? PB : PA) + (int64_t)row * KP;
#pragma unroll
                    for (int j = 0; j < KP; ++j) atomicAdd(dst + j, areg[j]);
                } else {
                    float* dst = hh ? PpartB + ((int64_t)(task - x_tasks) * KP + row) * KP
                                    : PpartA + ((int64_t)(task / num_rb) * d + row) * KP;
#pragma unroll
                    for (int j = 0; j < KP; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(areg[j], areg[j + 1], areg[j + 2], areg[j + 3]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == NPROD) tmem_dealloc(tmem_base, 512);
}

// outA[i] = sum over the copies of A (in copy order: fixed summation order, bit-reproducible), then the same for B;
// ONE launch for both regions.  Counts are multiples of 4 (kp % 32 == 0).
__global__ void __launch_bounds__(256)
k_sum_copies(const DevState* __restrict__ st, const float* __restrict__ copiesA, int ncopiesA, int64_t countA,
             float* __restrict__ outA, const float* __restrict__ copiesB, int ncopiesB, int64_t countB,
             float* __restrict__ outB) {
    if (st->stop) return;
    const int64_t nA4 = countA >> 2, nB4 = countB >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nA4 + nB4; i += (int64_t)gridDim.x * blockDim.x) {
        const bool isb = i >= nA4;
        const int64_t e = isb ? i - nA4 : i, count = isb ? countB : countA;
        const float* src = isb ? copiesB : copiesA;
        const int nc = isb ? ncopiesB : ncopiesA;
        float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int c = 0; c < nc; ++c) {
            const float4 v = __ldcs(reinterpret_cast<const float4*>(src + (int64_t)c * count) + e);
            a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
        }
        reinterpret_cast<float4*>(isb ? outB : outA)[e] = a;
    }
}

// Rows [row0, row0 + kpb) of H (.. x ldh) -> chunk-major Hs = [H_hi rows ; H_lo rows] of that block; used when
// the X.H^T pass runs on an H that did not come out of the H-update epilogue (bootstrap, user-assigned H).
__global__ void k_split_rows(const DevState* __restrict__ st, const float* __restrict__ H, int kpb, int64_t ldh,
                             float* __restrict__ Hs) {
    if (st->stop) return;
    const int64_t total = (int64_t)kpb * ldh;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / ldh);
        const int64_t c = i - (int64_t)r * ldh;
        const float v = H[i];
        const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
        Hs[hs_index(r, c, 2 * kpb)] = hi;
        Hs[hs_index(kpb + r, c, 2 * kpb)] = v - hi;
    }
}

// [hi | lo] split of columns [col0, col0 + kpb) of a row-major matrix (rows x ld): -> dst rows x 2 kpb   (W and G)
__global__ void k_split_hilo(const DevState* __restrict__ st, const float* __restrict__ src, int64_t rows, int ld,
                             int col0, int kpb, float* __restrict__ dst) {
    if (st->stop) return;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * kpb) return;
    const int64_t r = i / kpb;
    const int c = (int)(i % kpb);
    const float v = src[r * ld + col0 + c];
    const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
    dst[r * 2 * kpb + c] = hi;
    dst[r * 2 * kpb + kpb + c] = v - hi;
}

// ---- centering of the small operand (TS kernels, k <= 64; PYMFB_CENTER=1, experiments only) ------------------
// W^T X and G H are sums of POSITIVE products; accumulated with truncation (see "Segments") they come out low
// by an amount that grows with the chain length.  With PYMFB_CENTER=1 the TS H-update kernels contract against the
// CENTERED operand W' = W - 1 w_mean^T (column means) resp. G' = G - 1 g_mean^T: the products change sign,
// the truncation errors stop being one-sided, and the exact identity
//     W^T x_c = W'^T x_c + w_mean * sum_r x_rc ,     G h_c = G'^T h_c + g_mean * sum_i h_ic
// is restored in the epilogue with one FMA per output (column sums of X are computed once per data set, those of
// the H tile come from the registers that already hold it).  Measured on the cfg2 prefix: scale drift of W / H per
// iteration 1.2e-6 -> see DESIGN.md 5.1.  It is off by default: the error of an entry of C becomes
// eps * w_mean * sum(x) rather than eps * C, which ruins the small entries of parts-based factors.
constexpr int CM_SPLITS = 64;          // row splits of the column-sum reduction of W

// part[split][c] = sum of src[r][c] over the rows of the split (c < cols <= 64; deterministic order)
__global__ void __launch_bounds__(256)
k_colsum_partial(const DevState* __restrict__ st, const float* __restrict__ src, int64_t rows, int ld, int cols,
                 float* __restrict__ part) {
    if (st->stop) return;
    __shared__ float sh[256];
    const int lanes = 256 / cols;                 // row lanes per block (cols = 32 or 64)
    const int c = threadIdx.x % cols, rl = threadIdx.x / cols;
    const int64_t per = (rows + gridDim.x - 1) / gridDim.x;
    const int64_t r0 = (int64_t)blockIdx.x * per, r1 = min(rows, r0 + per);
    float acc = 0.f;
    for (int64_t r = r0 + rl; r < r1; r += lanes) acc += src[r * ld + c];
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (rl == 0) {
        for (int l = 1; l < lanes; ++l) acc += sh[l * cols + c];
        part[blockIdx.x * cols + c] = acc;
    }
}

// [hi | lo] split of (src - column mean): mean[c] = (sum over the `nsplit` partials) / rows_real, also written to
// mean_out by block 0; rows >= rows_real and columns >= cols_real stay 0 (zero padding must stay exact).
__global__ void __launch_bounds__(256)
k_split_hilo_centered(const DevState* __restrict__ st, const float* __restrict__ src, int64_t rows, int ld, int kpb,
                      const float* __restrict__ part, int nsplit, int64_t rows_real, int cols_real,
                      float* __restrict__ dst, float* __restrict__ mean_out) {
    if (st->stop) return;
    __shared__ float mean[64];
    if (threadIdx.x < kpb) {
        float a = 0.f;
        for (int sp = 0; sp < nsplit; ++sp) a += part[sp * kpb + threadIdx.x];
        a = (threadIdx.x < cols_real) ? a / (float)rows_real : 0.f;
        mean[threadIdx.x] = a;
        if (blockIdx.x == 0) mean_out[threadIdx.x] = a;
    }
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < rows * kpb; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / kpb;
        const int c = (int)(i % kpb);
        const float v = (r < rows_real && c < cols_real) ? src[r * ld + c] - mean[c] : 0.f;
        const float hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
        dst[r * 2 * kpb + c] = hi;
        dst[r * 2 * kpb + kpb + c] = v - hi;
    }
}

// xsum[c] = sum over the rows of X of column c (fp64 accumulation, stored fp32); once per data set
__global__ void __launch_bounds__(256)
k_colsum_x(const float* __restrict__ X, int64_t ldx, int64_t d, int64_t n_loc, float* __restrict__ xsum, int64_t xps, int xsh) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_loc) return;
    X += xpanel_off(c, xps, xsh);
    double a0 = 0.0, a1 = 0.0;
    int64_t r = 0;
    for (; r + 1 < d; r += 2) { a0 += (double)X[r * ldx + c]; a1 += (double)X[(r + 1) * ldx + c]; }
    if (r < d) a0 += (double)X[r * ldx + c];
    xsum[c] = (float)(a0 + a1);
}

}  // namespace tc

// ---------------------------------------------------------------------------------------------
// host side: plan (tensor maps, split buffers) and launchers
// ---------------------------------------------------------------------------------------------
struct TcPlan {
    bool ready = false;
    int device = 0, sm_count = 148;
    int64_t d = 0, n_loc = 0, ldx = 0, ldh = 0;
    int64_t xps = 0;           // layout of X (common.cuh): floats between panels, 0 = row-major
    int xsh64 = kNoPanelShift; // log2(panel width) for 64-bit column arithmetic (SIMT helpers)
    int xsh = tc::kNoPanel;    // the same for the TMA coordinates of the tensor-core kernels
    int k = 0, kp = 0;
    const float* X = nullptr;
    const float* Hbuf[2] = {nullptr, nullptr};
    float* Hs[2] = {nullptr, nullptr};        // [H_hi ; H_lo] companion of each H buffer, chunk-major (hs_index)
    bool hs_valid[2] = {false, false};
    // k > 128 runs as nblk = kp / 128 blocks of kpb = 128 bases (one launch of each pass per block, each streaming
    // X); k <= 128: nblk = 1, kpb = kp.  All per-block buffers are slices of the allocations below.
    int nblk = 1, kpb = 0;
    float* Wsplit = nullptr;   // nblk x (d x 2kpb)   [W_hi | W_lo] of each block of bases
    float* Gsplit = nullptr;   // nblk x (kp x 2kpb)  [G_hi | G_lo] column slice of each block, all kp rows
    CUtensorMap mapW_b[4], mapG_b[4], mapH_xb[2][4];   // per-block maps (k > 128)
    CUtensorMap mapX_h, mapX_x, mapW, mapG, mapH_h[2], mapH_x[2];
    CUtensorMap mapX_p, mapH_p[2];   // TS kernels: plain (unswizzled) 128-column x 32-row boxes
    CUtensorMap mapX_p64, mapH_p64[2], mapW64, mapG64;   // the same with 64-row boxes (k_h_update_tsr<KP, 64>)
    int ts_rs = 64;                  // rows per stage of the TS H-update kernel (PYMFB_TS_RS=32: the round-1 kernel)
    CUtensorMap mapH_a[2];           // H as the A operand of the H.H^T tasks (128-row boxes, rows >= kp zero-filled)
    int hh_tasks = 0, hh_cols_per_task = 0;
    bool use_ts = false;             // k <= 64: A operand from TMEM (k_*_ts), else both operands in smem
    bool use_ts2 = false;            // EXPERIMENT (PYMFB_TS2=1, kp = 64): CTA-pair H-update kernel (kernels_ts2.cuh)
    bool use_tc2 = false;            // EXPERIMENT (PYMFB_TC2=1, 128-wide blocks of bases): CTA-pair SS H-update kernel (kernels_tc2.cuh)
    int h_tiles = 0, x_rb = 0, x_cols_per_task = 0, x_tasks = 0;
    float* dbg = nullptr;      // optional raw-accumulator dump (tests/tc_probe.cu)
    const float* Dp = nullptr; // Semi-NMF: G+ H and G- H of the H buffer being updated (set by the scheduler), else null
    const float* Dn = nullptr;
    float* xpart = nullptr;    // deterministic combine of the X H^T / H H^T column splits: x_splits copies of A, then
    float* xpartB = nullptr;   //   hh_tasks copies of B (null: fp32 atomics)
    int x_splits = 0;
    bool center = false;       // TS kernels: contract against the centered W / G (see "centering" above)
    float* xsum = nullptr;     // n_loc column sums of X (center)
    bool xsum_valid = false;
    float* wmean = nullptr;    // kp column means of W, kp column means of G, CM_SPLITS x kp partials
    float* gmean = nullptr;
    float* cm_part = nullptr;
    int ss_pf = 0;             // SS kernels: L2 prefetch distance of X in stages (PYMFB_SS_PF)
    int xrev = 0;              // experiment (PYMFB_XREV=1): the X H^T pass walks the column ranges backwards, hoping to find the
                               // tail of the H-update pass in L2 - measured neutral on cfg2 / cfg3 / cfg4 k=64, so off
    int seg_c = 1;             // stages per segment of the W^T X contraction (= kp / 32: the G H chain length)
    int seg_x = 8;             // stages per segment of the X H^T / H H^T contractions (SS kernels: PYMFB_SEG_X; TS kernels: SEG_STAGES)
    float lam_h = 0.f;         // BNMF penalty weight of the next H-update launch (0 = plain NMF), set by the scheduler
    std::string err;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}
// 2-D fp32 row-major matrix (rows x cols, leading dimension ld), box = 32 columns x box_rows, 128B swizzle,
// out-of-bounds elements read as zero.
inline bool make_map(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                     bool mn_major, std::string* err) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { *err = "cuTensorMapEncodeTiled not available"; return false; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { *err = "cuTensorMapEncodeTiled failed with code " + std::to_string((int)r); return false; }
    return true;
}

// 3-D map of a matrix in the layout of common.cuh: dims (columns inside a panel, rows, panels).  swz: 0 = none (plain
// box), 1 = SWIZZLE_128B (K-major operand), 2 = SWIZZLE_128B_ATOM_32B (MN-major operand).  Row-major = one panel.
inline bool make_map3(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int64_t xps, int xsh,
                      int box_cols, int box_rows, int swz, std::string* err) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { *err = "cuTensorMapEncodeTiled not available"; return false; }
    const bool paneled = xps != 0;
    const int64_t pw = paneled ? ((int64_t)1 << xsh) : cols;
    const int64_t npan = paneled ? (cols + pw - 1) / pw : 1;
    cuuint64_t dims[3] = {(cuuint64_t)pw, (cuuint64_t)rows, (cuuint64_t)npan};
    cuuint64_t strides[2] = {(cuuint64_t)ld * sizeof(float), (cuuint64_t)(paneled ? xps : ld * rows) * sizeof(float)};
    cuuint32_t box[3] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1u};
    cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUtensorMapSwizzle sw = swz == 0 ? CU_TENSOR_MAP_SWIZZLE_NONE : swz == 1 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    // a row-major matrix is one panel: plain 2-D map (tma_load_x issues the 2-D instruction for it)
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, paneled ? 3 : 2, (void*)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { *err = "cuTensorMapEncodeTiled(3-D) failed with code " + std::to_string((int)r); return false; }
    return true;
}

// plain (unswizzled) map: box = box_cols x box_rows
inline bool make_map_plain(CUtensorMap* m, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                           int box_rows, std::string* err) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { *err = "cuTensorMapEncodeTiled not available"; return false; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
    cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { *err = "cuTensorMapEncodeTiled(plain) failed with code " + std::to_string((int)r); return false; }
    return true;
}

inline bool tc_supported(int64_t d, int64_t n_loc, int kp, int64_t ldx, const float* X, std::string* why) {
    if (kp % 32 != 0 || kp < 32 || (kp > 128 && (kp % 128 != 0 || kp > 512))) { *why = "k (padded) must be 32..128 in steps of 32, or 256 / 384 / 512"; return false; }
    if (ldx % 4 != 0 || ((uintptr_t)X & 15) != 0) { *why = "X must be 16-byte aligned with ld % 4 == 0"; return false; }
    if (d >= (1LL << 31) || n_loc >= (1LL << 31) - 256) { *why = "dimension too large"; return false; }
    if (d < 64 || n_loc < 128) { *why = "problem too small for the tensor-core tiles"; return false; }
    return true;
}

template <int KP>
inline int ts_set_attrs() {
    cudaError_t e = cudaFuncSetAttribute(tc::k_h_update_ts<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TsCfg<KP>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_xht_ts<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TsCfg<KP>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_h_update_tsr<KP, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TsrCfg<KP, 64>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_h_update_tsr<KP, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TsrCfg<KP, 32>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_h_update_ts2w<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::TsCfg<KP>::SMEM_BYTES);
    return e == cudaSuccess ? 0 : 1;
}

template <int KP>
inline int tc_set_attrs() {
    cudaError_t e = cudaFuncSetAttribute(tc::k_h_update_tc<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::HCfg<KP>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_h_update_tc<KP, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::HCfg<KP>::SMEM_BYTES);
    if (e != cudaSuccess) return 1;
    e = cudaFuncSetAttribute(tc::k_xht_tc<KP>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::XCfg<KP>::SMEM_BYTES);
    return e == cudaSuccess ? 0 : 1;
}

#if defined(PYMFB_TRACE)
inline void tc_trace_dump(TcPlan& p) {
    const char* path = getenv("PYMFB_TRACE_FILE");
    if (!p.dbg || !path) return;
    const size_t n = (size_t)tc::TRACE_STAGES * 16;
    std::vector<long long> h(n);
    cudaDeviceSynchronize();
    if (cudaMemcpy(h.data(), p.dbg + (1 << 18), n * sizeof(long long), cudaMemcpyDeviceToHost) != cudaSuccess) return;
    FILE* f = fopen(path, "wb");
    if (!f) return;
    fwrite(h.data(), sizeof(long long), n, f);
    fclose(f);
    // fused-kernel event log (kernels_fused.cuh FTRACE): [count][(code, value, clock) ...]
    std::vector<long long> ev((size_t)(2 << 20) / sizeof(long long));
    if (cudaMemcpy(ev.data(), reinterpret_cast<char*>(p.dbg) + (2 << 20), (size_t)2 << 20, cudaMemcpyDeviceToHost) != cudaSuccess) return;
    std::string p2 = std::string(path) + ".events";
    f = fopen(p2.c_str(), "wb");
    if (!f) return;
    fwrite(ev.data(), sizeof(long long), ev.size(), f);
    fclose(f);
}
#endif
inline void tc_release(TcPlan& p) {
#if defined(PYMFB_TRACE)
    tc_trace_dump(p);
    if (p.dbg) { cudaFree(p.dbg); p.dbg = nullptr; }
#endif
    if (p.Wsplit) cudaFree(p.Wsplit);
    if (p.Gsplit) cudaFree(p.Gsplit);
    if (p.xpart) cudaFree(p.xpart);
    p.xpart = p.xpartB = nullptr;
    if (p.xsum) cudaFree(p.xsum);
    if (p.wmean) cudaFree(p.wmean);
    p.xsum = p.wmean = p.gmean = p.cm_part = nullptr; p.xsum_valid = false; p.center = false;
    for (int i = 0; i < 2; ++i) { if (p.Hs[i]) cudaFree(p.Hs[i]); p.Hs[i] = nullptr; p.hs_valid[i] = false; }
    p.Wsplit = p.Gsplit = nullptr;
    p.ready = false;
}

// product = true: a plan for the plain products of NNDSVD (tc_qtx / tc_xzt): SS kernels at every width, SEG_STAGES-stage
// segments (no ratio whose two chains must match), and always the deterministic combine of the X H^T splits.
inline int tc_plan(TcPlan& p, int device, int sm_count, int64_t d, int64_t n_loc, int k, int kp, const float* X,
                   int64_t ldx, int64_t ldh, const float* H0, const float* H1, int64_t xps, int xsh64, bool product = false) {
    tc_release(p);
    p.device = device; p.sm_count = sm_count; p.d = d; p.n_loc = n_loc; p.k = k; p.kp = kp; p.X = X; p.ldx = ldx; p.ldh = ldh;
    p.xps = xps; p.xsh64 = xsh64; p.xsh = xps != 0 ? xsh64 : tc::kNoPanel;
    p.Hbuf[0] = H0; p.Hbuf[1] = H1;
    p.nblk = kp > 128 ? kp / 128 : 1;
    p.kpb = kp > 128 ? 128 : kp;
    if (cudaMalloc(&p.Wsplit, (size_t)d * 2 * kp * sizeof(float)) != cudaSuccess) { p.err = "cudaMalloc Wsplit failed"; return 1; }
    if (cudaMalloc(&p.Gsplit, (size_t)kp * 2 * kp * sizeof(float)) != cudaSuccess) { p.err = "cudaMalloc Gsplit failed"; return 1; }
    for (int i = 0; i < 2; ++i) {
        if (cudaMalloc(&p.Hs[i], (size_t)2 * kp * ldh * sizeof(float)) != cudaSuccess) { p.err = "cudaMalloc Hs failed"; return 1; }
        cudaMemset(p.Hs[i], 0, (size_t)2 * kp * ldh * sizeof(float));
        p.hs_valid[i] = false;
    }
    bool ok = true;
    ok = ok && make_map3(&p.mapX_h, X, d, n_loc, ldx, xps, xsh64, 32, tc::R1, 2, &p.err);
    ok = ok && make_map3(&p.mapX_x, X, d, n_loc, ldx, xps, xsh64, 32, 128, 1, &p.err);
    ok = ok && make_map(&p.mapW, p.Wsplit, d, 2 * p.kpb, 2 * p.kpb, tc::R1, true, &p.err);
    ok = ok && make_map(&p.mapG, p.Gsplit, kp, 2 * p.kpb, 2 * p.kpb, tc::R1, true, &p.err);
    for (int b = 0; b < p.nblk; ++b) {
        ok = ok && make_map(&p.mapW_b[b], p.Wsplit + (size_t)b * d * 2 * p.kpb, d, 2 * p.kpb, 2 * p.kpb, tc::R1, true, &p.err);
        ok = ok && make_map(&p.mapG_b[b], p.Gsplit + (size_t)b * kp * 2 * p.kpb, kp, 2 * p.kpb, 2 * p.kpb, tc::R1, true, &p.err);
        for (int i = 0; i < 2; ++i)
            ok = ok && make_map(&p.mapH_xb[i][b], p.Hs[i] + (size_t)b * 2 * p.kpb * ldh, (ldh / 32) * 2 * p.kpb, 32, 32, 2 * p.kpb, false, &p.err);
    }
    for (int i = 0; i < 2; ++i) {
        ok = ok && make_map3(&p.mapH_h[i], p.Hbuf[i], kp, n_loc, ldh, 0, kNoPanelShift, 32, tc::R1, 2, &p.err);
        ok = ok && make_map(&p.mapH_x[i], p.Hs[i], (ldh / 32) * 2 * p.kpb, 32, 32, 2 * p.kpb, false, &p.err);   // [H_hi ; H_lo] chunks as B (block 0)
        ok = ok && make_map3(&p.mapH_a[i], p.Hbuf[i], kp, n_loc, ldh, 0, kNoPanelShift, 32, 128, 1, &p.err);        // H as A
    }
    // (addressing the 128-column panels as one 2-D matrix of (panels * d) rows for this kernel, i.e. the 2-D TMA
    // instruction instead of the 3-D one, was measured: no difference)
    ok = ok && make_map3(&p.mapX_p, X, d, n_loc, ldx, xps, xsh64, tc::TILE_COLS, tc::R1, 0, &p.err);
    for (int i = 0; i < 2; ++i) ok = ok && make_map3(&p.mapH_p[i], p.Hbuf[i], kp, n_loc, ldh, 0, kNoPanelShift, tc::TILE_COLS, tc::R1, 0, &p.err);
    if (kp <= 64) {      // 64-row boxes of the TS H-update kernel (rows beyond the matrix - H and G have kp rows - read as zero)
        ok = ok && make_map3(&p.mapX_p64, X, d, n_loc, ldx, xps, xsh64, tc::TILE_COLS, 64, 0, &p.err);
        for (int i = 0; i < 2; ++i) ok = ok && make_map3(&p.mapH_p64[i], p.Hbuf[i], kp, n_loc, ldh, 0, kNoPanelShift, tc::TILE_COLS, 64, 0, &p.err);
        ok = ok && make_map(&p.mapW64, p.Wsplit, d, 2 * p.kpb, 2 * p.kpb, 64, true, &p.err);
        ok = ok && make_map(&p.mapG64, p.Gsplit, kp, 2 * p.kpb, 2 * p.kpb, 64, true, &p.err);
    }
    if (!ok) return 1;
    // TS H-update kernel: k <= 32 runs k_h_update_tsr with 64-row stages (cfg2 0.674 -> 0.664 ms, 8192 x 524288 k=32 2.97 -> 2.69 ms);
    // k = 64 keeps k_h_update_ts (32 rows, separate empty / aempty commits): there 64-row stages leave only two TMEM A slots
    // (4.07-4.28 vs 3.71 ms on cfg4 k=64) and the single-commit 32-row variant measured 3.86-3.94 vs 3.71 ms, same box.
    // PYMFB_TS_RS = 64 / 32 force k_h_update_tsr<KP, 64 / 32>, 1 forces k_h_update_ts.
    { const char* e = getenv("PYMFB_TS_RS"); p.ts_rs = e ? atoi(e) : (kp == 32 ? 64 : 1); }
    {
        const char* force_ss = getenv("PYMFB_TC_FORCE_SS");
        p.use_ts = !product && kp <= 64 && !(force_ss && force_ss[0] == '1');
        if (p.use_ts && (kp == 32 ? ts_set_attrs<32>() : ts_set_attrs<64>())) { p.err = "cudaFuncSetAttribute (TS kernels) failed"; return 1; }
    }
    int rc = p.kpb == 32 ? tc_set_attrs<32>() : p.kpb == 64 ? tc_set_attrs<64>() : p.kpb == 96 ? tc_set_attrs<96>() : tc_set_attrs<128>();
    if (rc) { p.err = "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed"; return 1; }
#if defined(PYMFB_TRACE)
    {
        const size_t bytes = (size_t)4 << 20;   // [0,1 MB) accumulator dumps | [1 MB, 1.5 MB) stage trace | [2 MB, 4 MB) fused-kernel event log
        if (cudaMalloc(&p.dbg, bytes) != cudaSuccess) { p.err = "cudaMalloc trace buffer failed"; return 1; }
        cudaMemset(p.dbg, 0, bytes);
    }
#endif
    p.h_tiles = (int)((n_loc + tc::TILE_COLS - 1) / tc::TILE_COLS);
    { const char* e = getenv("PYMFB_XREV"); p.xrev = (e && e[0] == '1') ? 1 : 0; }
    { const char* e = getenv("PYMFB_SS_PF"); p.ss_pf = e ? std::max(0, atoi(e)) : 0; }
    {   // Bias of the H-update ratio C / D (see "Segments"): the C chain is kept as short as the D chain (kp / 32
        // stages).  The TS kernels drain C at least every 2 stages (64 rows, the stage of k_h_update_tsr<KP, 64>, so
        // that every TS schedule drains at the same rows; k <= 32: 8 MMAs against 4).  The operands stay uncentered: centering
        // (PYMFB_CENTER=1, experiments only) turns the error of an entry of C into eps * w_mean * sum(x), which on
        // parts-based data is far larger than the entry itself (tests/test_elementwise.py).
        // PYMFB_SEG_C overrides the segment length for experiments.
        const char* e = getenv("PYMFB_SEG_C");
        const char* ce = getenv("PYMFB_CENTER");
        p.center = p.use_ts && ce && ce[0] == '1';
        p.seg_c = (e && atoi(e) > 0) ? atoi(e)
                : ((p.center || product) ? tc::SEG_STAGES : std::max(p.use_ts ? 2 : 1, kp / tc::R1));
        if (p.center) {
            if (cudaMalloc(&p.xsum, (size_t)n_loc * sizeof(float)) != cudaSuccess) { p.err = "cudaMalloc xsum failed"; return 1; }
            if (cudaMalloc(&p.wmean, (size_t)(2 + tc::CM_SPLITS) * kp * sizeof(float)) != cudaSuccess) { p.err = "cudaMalloc wmean failed"; return 1; }
            p.gmean = p.wmean + kp;
            p.cm_part = p.wmean + 2 * kp;
            p.xsum_valid = false;
        }
    }
    // X H^T tasks: (row block, column range); ~4 tasks per SM, each a multiple of 32 columns.  Column ranges are not
    // capped in length: the row-block CTAs of a range share its [H_hi ; H_lo] chunks through L2, where k_xht_tc keeps
    // them by loading X evict_first and H evict_last (k_xht_ts measured no gain from either).  Few splits keep the
    // partial copies within the budget of the ordered combine below (cfg3 on one GPU: 37 splits of 888 chunks, 310 MB).
    p.x_rb = (int)((d + 127) / 128);
    const int64_t chunks = (n_loc + 31) / 32;
    int64_t splits = std::max<int64_t>(1, (4LL * sm_count + p.x_rb - 1) / p.x_rb);
    {   // make #tasks a multiple of the CTA count: 608 tasks on 148 CTAs ran 5 rounds with the last 11 % full
        auto gcd = [](int64_t a, int64_t b) { while (b) { int64_t t = a % b; a = b; b = t; } return a; };
        const int64_t m = sm_count / gcd(p.x_rb, sm_count);
        splits = std::max<int64_t>(m, (splits + m / 2) / m * m);
    }
    splits = std::min(splits, chunks);
    // Column ranges are whole segments (SEG_STAGES stages) wherever n allows, for X H^T and H H^T alike: the W update
    // is the ratio A / (W B), so the accumulation chains of A and B must have the same length (see "Segments").
    { const char* e = getenv("PYMFB_SEG_X"); p.seg_x = (!p.use_ts && e && atoi(e) > 0) ? atoi(e) : (p.use_ts ? tc::SEG_STAGES : PYMFB_SS_SEG_X); }
    const int64_t segx = p.seg_x;
    auto seg_round = [&](int64_t per) { return (per >= segx) ? (per + segx - 1) / segx * segx : per; };
    const int64_t chunks_per = seg_round((chunks + splits - 1) / splits);
    p.x_cols_per_task = (int)(chunks_per * 32);
    splits = (chunks + chunks_per - 1) / chunks_per;
    p.x_tasks = (int)(splits * p.x_rb);
    {   // H H^T tasks (TS kernels): ~one short task per SM, never shorter than the X H^T chains
        int64_t hsplits = std::min<int64_t>(chunks, sm_count);
        int64_t hper = seg_round((chunks + hsplits - 1) / hsplits);
        if (hper < segx) hper = std::min<int64_t>(chunks_per, segx);
        p.hh_cols_per_task = (int)(hper * 32);
        p.hh_tasks = (int)((chunks + hper - 1) / hper);
    }
    {   // Deterministic combine (bit-reproducible W): partial copies instead of atomics while they stay below 1 GiB
        // (every bench workload fits; PYMFB_DETERMINISTIC=1 forces, =0 disables)
        p.x_splits = p.x_tasks / p.x_rb;
        const size_t bytes = ((size_t)p.x_splits * d * kp + (size_t)p.hh_tasks * kp * kp) * sizeof(float);
        const char* e = getenv("PYMFB_DETERMINISTIC");
        const bool want = product || (e ? e[0] == '1' : bytes <= ((size_t)1 << 30));
        if (want) {
            if (cudaMalloc(&p.xpart, bytes) != cudaSuccess) { p.err = "cudaMalloc X.H^T partial copies failed"; return 1; }
            p.xpartB = p.xpart + (size_t)p.x_splits * d * kp;
        }
    }
    p.ready = true;
    return 0;
}

// refresh [W_hi | W_lo] and [G_hi | G_lo] after W / G changed
inline int tc_after_gram(TcPlan& p, const DevState* st, const float* W, const float* G, cudaStream_t stream, int64_t* launches) {
    const int64_t nw = p.d * p.kpb, ng = (int64_t)p.kp * p.kpb;
    if (p.center) {        // nblk == 1, kpb == kp
        if (!p.xsum_valid) {
            tc::k_colsum_x<<<(unsigned)((p.n_loc + 255) / 256), 256, 0, stream>>>(p.X, p.ldx, p.d, p.n_loc, p.xsum, p.xps, p.xsh64);
            p.xsum_valid = true;
            *launches += 1;
        }
        const int wsplits = (int)std::min<int64_t>(tc::CM_SPLITS, std::max<int64_t>(1, p.d / 64));
        tc::k_colsum_partial<<<wsplits, 256, 0, stream>>>(st, W, p.d, p.kp, p.kp, p.cm_part);
        tc::k_split_hilo_centered<<<(unsigned)std::min<int64_t>((nw + 255) / 256, 4 * p.sm_count), 256, 0, stream>>>(
            st, W, p.d, p.kp, p.kp, p.cm_part, wsplits, p.d, p.k, p.Wsplit, p.wmean);
        // G: kp x kp, one block: the "partials" are the rows of G themselves (rows >= k are zero)
        tc::k_split_hilo_centered<<<1, 256, 0, stream>>>(st, G, p.kp, p.kp, p.kp, G, p.kp, p.k, p.k, p.Gsplit, p.gmean);
        *launches += 3;
        return cudaGetLastError() == cudaSuccess ? 0 : 1;
    }
    for (int b = 0; b < p.nblk; ++b) {
        tc::k_split_hilo<<<(unsigned)((nw + 255) / 256), 256, 0, stream>>>(st, W, p.d, p.kp, b * p.kpb, p.kpb, p.Wsplit + (size_t)b * p.d * 2 * p.kpb);
        tc::k_split_hilo<<<(unsigned)((ng + 255) / 256), 256, 0, stream>>>(st, G, p.kp, p.kp, b * p.kpb, p.kpb, p.Gsplit + (size_t)b * p.kp * 2 * p.kpb);
    }
    *launches += 2 * p.nblk;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

template <int KP>
inline void tc_launch_h(TcPlan& p, const DevState* st, int hsrc, float* Hn, cudaStream_t stream) {
    const int grid = std::min(p.h_tiles, p.sm_count);
    for (int b = 0; b < p.nblk; ++b) {        // one launch per block of <= 128 bases (k <= 128: one launch)
        const size_t hoff = (size_t)b * p.kpb * p.ldh;
        tc::k_h_update_tc<KP><<<grid, tc::HCfg<KP>::THREADS, tc::HCfg<KP>::SMEM_BYTES, stream>>>(
            p.mapX_h, p.mapW_b[b], p.mapH_h[hsrc], p.mapG_b[b], st, p.Hbuf[hsrc] + hoff, Hn + hoff, p.Hs[hsrc ^ 1] + 2 * hoff,
            p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, p.dbg, p.kp, p.seg_c, p.lam_h,
            p.Dp ? p.Dp + hoff : nullptr, p.Dn ? p.Dn + hoff : nullptr, p.xsh, p.ss_pf);
    }
}
// experiment knob: PYMFB_GRID caps the CTA count of the H-update kernels (per-SM pipeline capacity measurements)
inline int grid_cap(int grid) {
    static const int cap = [] { const char* e = getenv("PYMFB_GRID"); return e ? atoi(e) : 0; }();
    return cap > 0 ? std::min(grid, cap) : grid;
}
template <int KP>
inline void ts_launch_h(TcPlan& p, const DevState* st, int hsrc, float* Hn, cudaStream_t stream) {
    const int grid = grid_cap(std::min(p.h_tiles, p.sm_count));
    if (p.ts_rs == 64) {
        tc::k_h_update_tsr<KP, 64><<<grid, tc::TsrCfg<KP, 64>::THREADS, tc::TsrCfg<KP, 64>::SMEM_BYTES, stream>>>(
            p.mapX_p64, p.mapW64, p.mapH_p64[hsrc], p.mapG64, st, p.Hbuf[hsrc], Hn, p.Hs[hsrc ^ 1], p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, p.dbg,
            std::max(1, p.seg_c / 2), p.lam_h, p.Dp, p.Dn, p.center ? p.wmean : nullptr, p.gmean, p.xsum, p.xsh);
        return;
    }
    if (p.ts_rs == 2) {
        tc::k_h_update_ts2w<KP><<<grid, tc::TsCfg<KP>::THREADS, tc::TsCfg<KP>::SMEM_BYTES, stream>>>(
            p.mapX_p, p.mapW, p.mapH_p[hsrc], p.mapG, st, p.Hbuf[hsrc], Hn, p.Hs[hsrc ^ 1], p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, p.dbg, p.seg_c, p.lam_h, p.Dp, p.Dn,
            p.center ? p.wmean : nullptr, p.gmean, p.xsum, p.xsh);
        return;
    }
    if (p.ts_rs == 32) {
        tc::k_h_update_tsr<KP, 32><<<grid, tc::TsrCfg<KP, 32>::THREADS, tc::TsrCfg<KP, 32>::SMEM_BYTES, stream>>>(
            p.mapX_p, p.mapW, p.mapH_p[hsrc], p.mapG, st, p.Hbuf[hsrc], Hn, p.Hs[hsrc ^ 1], p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, p.dbg,
            p.seg_c, p.lam_h, p.Dp, p.Dn, p.center ? p.wmean : nullptr, p.gmean, p.xsum, p.xsh);
        return;
    }
    tc::k_h_update_ts<KP><<<grid, tc::TsCfg<KP>::THREADS, tc::TsCfg<KP>::SMEM_BYTES, stream>>>(
        p.mapX_p, p.mapW, p.mapH_p[hsrc], p.mapG, st, p.Hbuf[hsrc], Hn, p.Hs[hsrc ^ 1], p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, p.dbg, p.seg_c, p.lam_h, p.Dp, p.Dn,
        p.center ? p.wmean : nullptr, p.gmean, p.xsum, p.xsh);
}
template <int KP>
inline void ts_launch_x(TcPlan& p, const DevState* st, int hsrc, float* P, cudaStream_t stream) {
    const int ntasks = p.x_tasks + p.hh_tasks;
    const int grid = std::min(ntasks, p.sm_count);
    tc::k_xht_ts<KP><<<grid, tc::X_THREADS, tc::TsCfg<KP>::SMEM_BYTES, stream>>>(
        p.mapX_x, p.mapH_x[hsrc], p.mapH_a[hsrc], st, P, P + p.d * p.kp, (int)p.d, (int)p.n_loc, p.x_cols_per_task,
        p.x_rb, p.x_tasks, p.hh_cols_per_task, ntasks, p.dbg, p.xpart, p.xpartB, p.xsh, p.xrev);
}
inline int tc_h_update(TcPlan& p, const DevState* st, const float* Hc, float* Hn, cudaStream_t stream, int64_t* launches) {
    const int hsrc = (Hc == p.Hbuf[0]) ? 0 : 1;
    p.hs_valid[hsrc ^ 1] = true;    // the epilogue writes [H_hi ; H_lo] of the new H
    if (p.use_ts) {
        if (p.kp == 32) ts_launch_h<32>(p, st, hsrc, Hn, stream); else ts_launch_h<64>(p, st, hsrc, Hn, stream);
        *launches += 1;
        return cudaGetLastError() == cudaSuccess ? 0 : 1;
    }
    switch (p.kpb) {
        case 32: tc_launch_h<32>(p, st, hsrc, Hn, stream); break;
        case 64: tc_launch_h<64>(p, st, hsrc, Hn, stream); break;
        case 96: tc_launch_h<96>(p, st, hsrc, Hn, stream); break;
        default: tc_launch_h<128>(p, st, hsrc, Hn, stream); break;
    }
    *launches += p.nblk;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

template <int KP>
inline void tc_launch_x(TcPlan& p, const DevState* st, int hsrc, float* P, cudaStream_t stream) {
    const int grid = std::min(p.x_tasks, p.sm_count);
    for (int b = 0; b < p.nblk; ++b)
        tc::k_xht_tc<KP><<<grid, tc::XCfg<KP>::THREADS, tc::XCfg<KP>::SMEM_BYTES, stream>>>(
            p.mapX_x, p.mapH_xb[hsrc][b], st, P + b * p.kpb, (int)p.d, (int)p.n_loc, p.x_cols_per_task, p.x_rb, p.x_tasks,
            p.dbg, p.kp, p.xpart ? p.xpart + b * p.kpb : nullptr, (int64_t)p.d * p.kp, p.xsh, p.xrev, p.ss_pf, p.seg_x);
}
// true when the launch also produced H H^T (so the caller skips its own H H^T kernel): the TS kernels run it as
// extra tasks of the same launch, the SS kernels as a second launch with H itself as the streamed operand
inline bool tc_xht_includes_hht(const TcPlan& p) { return true; }
// H H^T on the SS kernels: the X.H^T kernel with X := H (kp rows, 128-row boxes zero-filled beyond kp)
template <int KP>
inline void tc_launch_hht(TcPlan& p, const DevState* st, int hsrc, float* PB, cudaStream_t stream) {
    const int hh_rb = (p.kp + 127) / 128;
    const int ntasks = p.hh_tasks * hh_rb;
    const int grid = std::min(ntasks, p.sm_count);
    for (int b = 0; b < p.nblk; ++b)
        tc::k_xht_tc<KP><<<grid, tc::XCfg<KP>::THREADS, tc::XCfg<KP>::SMEM_BYTES, stream>>>(
            p.mapH_a[hsrc], p.mapH_xb[hsrc][b], st, PB + b * p.kpb, p.kp, (int)p.n_loc, p.hh_cols_per_task, hh_rb, ntasks,
            nullptr, p.kp, p.xpartB ? p.xpartB + b * p.kpb : nullptr, (int64_t)p.kp * p.kp, tc::kNoPanel, 0, 0, p.seg_x);
}
inline int tc_xht(TcPlan& p, const DevState* st, const float* Hc, float* P, cudaStream_t stream, int64_t* launches) {
    const int hsrc = (Hc == p.Hbuf[0]) ? 0 : 1;
    if (!p.hs_valid[hsrc]) {
        for (int b = 0; b < p.nblk; ++b)
            tc::k_split_rows<<<4 * p.sm_count, 256, 0, stream>>>(st, Hc + (size_t)b * p.kpb * p.ldh, p.kpb, p.ldh,
                                                                p.Hs[hsrc] + (size_t)b * 2 * p.kpb * p.ldh);
        *launches += p.nblk;
        p.hs_valid[hsrc] = true;
    }
    auto sum_copies = [&]() {      // deterministic combine: P = sum of the splits' copies, in split order
        if (!p.xpart) return;
        const int64_t na = p.d * p.kp, nb = (int64_t)p.kp * p.kp;
        tc::k_sum_copies<<<(unsigned)std::min<int64_t>(((na + nb) / 4 + 255) / 256, 8 * p.sm_count), 256, 0, stream>>>(
            st, p.xpart, p.x_splits, na, P, p.xpartB, p.hh_tasks, nb, P + na);
        *launches += 1;
    };
    if (p.use_ts) {
        if (p.kp == 32) ts_launch_x<32>(p, st, hsrc, P, stream); else ts_launch_x<64>(p, st, hsrc, P, stream);
        *launches += 1;
        sum_copies();
        return cudaGetLastError() == cudaSuccess ? 0 : 1;
    }
    switch (p.kpb) {
        case 32: tc_launch_x<32>(p, st, hsrc, P, stream); break;
        case 64: tc_launch_x<64>(p, st, hsrc, P, stream); break;
        case 96: tc_launch_x<96>(p, st, hsrc, P, stream); break;
        default: tc_launch_x<128>(p, st, hsrc, P, stream); break;
    }
    float* PB = P + p.d * p.kp;
    switch (p.kpb) {
        case 32: tc_launch_hht<32>(p, st, hsrc, PB, stream); break;
        case 64: tc_launch_hht<64>(p, st, hsrc, PB, stream); break;
        case 96: tc_launch_hht<96>(p, st, hsrc, PB, stream); break;
        default: tc_launch_hht<128>(p, st, hsrc, PB, stream); break;
    }
    *launches += 2 * p.nblk;
    sum_copies();
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

// ---- the two products of an NNDSVD sweep on a product plan (tc_plan(..., product = true)): kp = b' bases, Hbuf = {Zt, Zt2}
template <int KP>
inline void tc_launch_qtx(TcPlan& p, const DevState* st, float* Zt, cudaStream_t stream) {
    const int grid = std::min(p.h_tiles, p.sm_count);
    for (int b = 0; b < p.nblk; ++b)      // mapH / mapG are never read in product mode: any valid map will do
        tc::k_h_update_tc<KP, true><<<grid, tc::HCfg<KP>::THREADS, tc::HCfg<KP>::SMEM_BYTES, stream>>>(
            p.mapX_h, p.mapW_b[b], p.mapX_h, p.mapW_b[b], st, nullptr, Zt + (size_t)b * p.kpb * p.ldh, nullptr,
            p.ldh, (int)p.d, (int)p.n_loc, p.h_tiles, nullptr, 0, p.seg_c, 0.f, nullptr, nullptr, p.xsh, p.ss_pf);
}
// Zt (kp x ldh) = Q^T X, Q: d x kp row-major
inline int tc_qtx(TcPlan& p, const DevState* st, const float* Q, float* Zt, cudaStream_t stream, int64_t* launches) {
    const int64_t nw = p.d * p.kpb;
    for (int b = 0; b < p.nblk; ++b)
        tc::k_split_hilo<<<(unsigned)((nw + 255) / 256), 256, 0, stream>>>(st, Q, p.d, p.kp, b * p.kpb, p.kpb, p.Wsplit + (size_t)b * p.d * 2 * p.kpb);
    switch (p.kpb) {
        case 32: tc_launch_qtx<32>(p, st, Zt, stream); break;
        case 64: tc_launch_qtx<64>(p, st, Zt, stream); break;
        case 96: tc_launch_qtx<96>(p, st, Zt, stream); break;
        default: tc_launch_qtx<128>(p, st, Zt, stream); break;
    }
    *launches += 2 * p.nblk;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
// Y (d x kp row-major) = X Zt2^T with Zt2 = Hbuf[1]: the X H^T pass, its column splits summed in split order
inline int tc_xzt(TcPlan& p, const DevState* st, float* Y, cudaStream_t stream, int64_t* launches) {
    for (int b = 0; b < p.nblk; ++b)
        tc::k_split_rows<<<4 * p.sm_count, 256, 0, stream>>>(st, p.Hbuf[1] + (size_t)b * p.kpb * p.ldh, p.kpb, p.ldh,
                                                            p.Hs[1] + (size_t)b * 2 * p.kpb * p.ldh);
    switch (p.kpb) {
        case 32: tc_launch_x<32>(p, st, 1, Y, stream); break;
        case 64: tc_launch_x<64>(p, st, 1, Y, stream); break;
        case 96: tc_launch_x<96>(p, st, 1, Y, stream); break;
        default: tc_launch_x<128>(p, st, 1, Y, stream); break;
    }
    const int64_t na = p.d * p.kp;
    tc::k_sum_copies<<<(unsigned)std::min<int64_t>((na / 4 + 255) / 256, 8 * p.sm_count), 256, 0, stream>>>(
        st, p.xpart, p.x_splits, na, Y, nullptr, 0, 0, nullptr);
    *launches += 2 * p.nblk + 1;
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace pymfb
