// kernels_simt.cuh - fp32 CUDA-core kernels of the NMF multiplicative-update path.
//
// These are (a) the small replicated steps that stay on CUDA cores in every configuration
// (W update, W^T W, the fp64 error combine, ||X||^2, casts, generators) and (b) the
// any-shape streaming kernels (H update pass, X H^T pass) used when the tcgen05 path does
// not apply (tiny / unaligned problems such as BASELINE cfg1, 1000x500 k=10).
//
// Reference arithmetic (pymf/nmf.py):
//   update_h  :122-126   H <- H * (W^T X) / ((W^T W) H + 1e-9)
//   update_w  :128-132   W <- W * (X H^T) / ((W H) H^T + 1e-9)   [= W (H H^T), re-associated]
//   frobenius :100-114   sqrt(sum((X - W H)^2)) = sqrt(||X||^2 - 2<W, X H^T> + <W^T W, H H^T>)
#pragma once
#include "common.cuh"

namespace pymfb {

constexpr int SIMT_THREADS = 256;
constexpr int TILE_N = 128;   // columns per CTA tile (4 per thread x 32 thread columns)
constexpr int TILE_DK = 16;   // contraction rows staged per step

// ---------------------------------------------------------------------------------------
// acc[i][j] += sum_r L[r][lcol0 + ty*TK + i] * R[r][rcol0 + tx*4 + j]   for r in [r_begin, r_end)
// L: rows x ldl (row-major), R: rows x ldr.  Columns of R >= r_ncols read as zero; rows are
// bounded by r_end.  Column kb of L must be < ldl (L is padded to a multiple of KB).
// 256 threads: tx = tid & 31 (4 R-columns each), ty = tid >> 5 (TK = KB/8 L-columns each).
// ---------------------------------------------------------------------------------------
template <int KB>
__device__ __forceinline__ void tile_mac(float (&acc)[KB / 8][4],
                                         const float* __restrict__ L, int64_t ldl, int lcol0,
                                         const float* __restrict__ R, int64_t ldr, int64_t rcol0,
                                         int64_t r_ncols, int64_t r_begin, int64_t r_end,
                                         float (*Rs)[TILE_DK][TILE_N], float (*Ls)[TILE_DK][KB]) {
    constexpr int TK = KB / 8;
    const int tid = threadIdx.x;
    const int tx = tid & 31, ty = tid >> 5;
    constexpr int R_F4 = TILE_DK * TILE_N / 4 / SIMT_THREADS;   // float4 per thread for R (2)
    constexpr int L_F4_TOTAL = TILE_DK * KB / 4;                // float4 in an L chunk
    float4 rreg[R_F4];
    float4 lreg;

    auto load_chunk = [&](int64_t r0) {
#pragma unroll
        for (int t = 0; t < R_F4; ++t) {
            int f = tid + t * SIMT_THREADS;
            int row = f / (TILE_N / 4), c4 = f % (TILE_N / 4);
            int64_t r = r0 + row, c = rcol0 + c4 * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < r_end && c < r_ncols) {
                v = *reinterpret_cast<const float4*>(R + r * ldr + c);
                if (c + 1 >= r_ncols) v.y = 0.f;
                if (c + 2 >= r_ncols) v.z = 0.f;
                if (c + 3 >= r_ncols) v.w = 0.f;
            }
            rreg[t] = v;
        }
        lreg = make_float4(0.f, 0.f, 0.f, 0.f);
        if (tid < L_F4_TOTAL) {
            int row = tid / (KB / 4), c4 = tid % (KB / 4);
            int64_t r = r0 + row;
            if (r < r_end) lreg = *reinterpret_cast<const float4*>(L + r * ldl + lcol0 + c4 * 4);
        }
    };
    auto store_chunk = [&](int buf) {
#pragma unroll
        for (int t = 0; t < R_F4; ++t) {
            int f = tid + t * SIMT_THREADS;
            int row = f / (TILE_N / 4), c4 = f % (TILE_N / 4);
            *reinterpret_cast<float4*>(&Rs[buf][row][c4 * 4]) = rreg[t];
        }
        if (tid < L_F4_TOTAL) {
            int row = tid / (KB / 4), c4 = tid % (KB / 4);
            *reinterpret_cast<float4*>(&Ls[buf][row][c4 * 4]) = lreg;
        }
    };

    if (r_begin >= r_end) return;
    load_chunk(r_begin);
    store_chunk(0);
    __syncthreads();
    int buf = 0;
    for (int64_t r0 = r_begin; r0 < r_end; r0 += TILE_DK) {
        const bool has_next = r0 + TILE_DK < r_end;
        if (has_next) load_chunk(r0 + TILE_DK);
        // each TILE_DK-row step is summed on its own and then added: an fp32 chain of n products carries up to n
        // roundings, and at k >= 512 (G H) that alone exceeded 1e-5 on small entries (tests/test_elementwise.py)
        float part[TK][4];
#pragma unroll
        for (int r = 0; r < TILE_DK; ++r) {
            float4 x = *reinterpret_cast<const float4*>(&Rs[buf][r][tx * 4]);
            float w[TK];
#pragma unroll
            for (int i = 0; i < TK; ++i) w[i] = Ls[buf][r][ty * TK + i];
#pragma unroll
            for (int i = 0; i < TK; ++i) {
                part[i][0] = r == 0 ? w[i] * x.x : fmaf(w[i], x.x, part[i][0]);
                part[i][1] = r == 0 ? w[i] * x.y : fmaf(w[i], x.y, part[i][1]);
                part[i][2] = r == 0 ? w[i] * x.z : fmaf(w[i], x.z, part[i][2]);
                part[i][3] = r == 0 ? w[i] * x.w : fmaf(w[i], x.w, part[i][3]);
            }
        }
#pragma unroll
        for (int i = 0; i < TK; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] += part[i][j];
        if (has_next) store_chunk(buf ^ 1);
        __syncthreads();
        buf ^= 1;
    }
}

// ---------------------------------------------------------------------------------------
// H update pass (pymf/nmf.py:122-126), any shape.
//   grid.x = column tiles of 128, grid.y = k blocks of KB rows, grid.z = splits of the contraction over d.
//   C = W^T X  (contract over d),  D = G H (contract over kp),  Hn = H * C / (D + 1e-9)
// Hc is read (all kp rows, for D), Hn is written (rows of this k block) -> ping-pong buffers.
// Few-column problems (cfg1: n = 500 -> 4 tiles) would run on 4 SMs: with gridDim.z > 1 every CTA contracts
// rows_per_split rows of X, parks its partial C in Cpart, and the CTA that arrives LAST on the tile's ticket sums
// the partials in split order (deterministic) and applies the update.  The ticket is reset for the next launch.
// ---------------------------------------------------------------------------------------
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_h_update_simt(const DevState* __restrict__ st, const float* __restrict__ X, int64_t ldx,
                const float* __restrict__ W, const float* __restrict__ G,
                const float* __restrict__ Hc, float* __restrict__ Hn, int64_t ldh,
                int64_t d, int64_t n_loc, int kp, float lam, const float* __restrict__ Gneg,
                int64_t rows_per_split, float* __restrict__ Cpart, unsigned* __restrict__ tickets,
                float* __restrict__ zero_buf, int64_t zero_count, int64_t xps, int xsh) {
    // Gneg != nullptr: Semi-NMF (pymf/snmf.py:72-90) - G is then G+ and Gneg is G-
    if (st->stop) return;
    if (zero_buf != nullptr) {   // clear the [X H^T | H H^T] partial buffer for the pass that follows (saves a k_zero launch)
        const int64_t nb = (int64_t)gridDim.x * gridDim.y * gridDim.z;
        const int64_t b = ((int64_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        for (int64_t i = b * blockDim.x + threadIdx.x; i < zero_count; i += nb * blockDim.x) zero_buf[i] = 0.f;
    }
    constexpr int TK = KB / 8;
    __shared__ __align__(16) float Rs[2][TILE_DK][TILE_N];
    __shared__ __align__(16) float Ls[2][TILE_DK][KB];
    __shared__ bool is_last;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t col0 = (int64_t)blockIdx.x * TILE_N;
    const int kb0 = blockIdx.y * KB;

    float c[TK][4], dd[TK][4];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { c[i][j] = 0.f; dd[i][j] = 0.f; }

    const int nsplit = (int)gridDim.z;
    const int64_t r_begin = (int64_t)blockIdx.z * rows_per_split;
    const int64_t r_end = nsplit > 1 ? min(d, r_begin + rows_per_split) : d;
    {   // the 128-column tile lies inside one panel of X (common.cuh): panel-adjusted base, bound at the panel's end
        const int64_t pend = ((col0 >> xsh) + 1) << xsh;
        tile_mac<KB>(c, W, kp, kb0, X + xpanel_off(col0, xps, xsh), ldx, col0, min(n_loc, pend), r_begin, r_end, Rs, Ls);   // W^T X (this CTA's rows)
    }
    if (nsplit > 1) {
        const int64_t tile_id = (int64_t)blockIdx.y * gridDim.x + blockIdx.x;
        float* part = Cpart + (tile_id * nsplit) * (KB * TILE_N);                  // [split][KB][TILE_N] of this tile
        float* mine = part + (int64_t)blockIdx.z * (KB * TILE_N);
#pragma unroll
        for (int i = 0; i < TK; ++i)
            *reinterpret_cast<float4*>(mine + (ty * TK + i) * TILE_N + tx * 4) = make_float4(c[i][0], c[i][1], c[i][2], c[i][3]);
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) is_last = (atomicAdd(&tickets[tile_id], 1u) == (unsigned)(nsplit - 1));
        __syncthreads();
        if (!is_last) return;                                                      // block-uniform
        __threadfence();
#pragma unroll
        for (int i = 0; i < TK; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) c[i][j] = 0.f;
        for (int sp = 0; sp < nsplit; ++sp) {
#pragma unroll
            for (int i = 0; i < TK; ++i) {
                const float4 v = __ldcg(reinterpret_cast<const float4*>(part + (int64_t)sp * (KB * TILE_N) + (ty * TK + i) * TILE_N + tx * 4));
                c[i][0] += v.x; c[i][1] += v.y; c[i][2] += v.z; c[i][3] += v.w;
            }
        }
        if (threadIdx.x == 0) tickets[tile_id] = 0u;
    }
    tile_mac<KB>(dd, G, kp, kb0, Hc, ldh, col0, n_loc, 0, kp, Rs, Ls);    // G H (G symmetric)

    const int64_t col = col0 + tx * 4;
    if (Gneg != nullptr) {                                                // uniform over the launch
        float dn[TK][4];
#pragma unroll
        for (int i = 0; i < TK; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) dn[i][j] = 0.f;
        tile_mac<KB>(dn, Gneg, kp, kb0, Hc, ldh, col0, n_loc, 0, kp, Rs, Ls);   // G- H
        if (col >= n_loc) return;
#pragma unroll
        for (int i = 0; i < TK; ++i) {
            const int krow = kb0 + ty * TK + i;
            const float4 h = *reinterpret_cast<const float4*>(Hc + (int64_t)krow * ldh + col);
            float4 o;
            o.x = snmf_ratio(h.x, c[i][0], dd[i][0], dn[i][0]);
            o.y = (col + 1 < n_loc) ? snmf_ratio(h.y, c[i][1], dd[i][1], dn[i][1]) : 0.f;
            o.z = (col + 2 < n_loc) ? snmf_ratio(h.z, c[i][2], dd[i][2], dn[i][2]) : 0.f;
            o.w = (col + 3 < n_loc) ? snmf_ratio(h.w, c[i][3], dd[i][3], dn[i][3]) : 0.f;
            *reinterpret_cast<float4*>(Hn + (int64_t)krow * ldh + col) = o;
        }
        return;
    }
    if (col >= n_loc) return;
#pragma unroll
    for (int i = 0; i < TK; ++i) {
        const int krow = kb0 + ty * TK + i;
        const float4 h = *reinterpret_cast<const float4*>(Hc + (int64_t)krow * ldh + col);
        float4 o;
        o.x = mu_ratio(h.x, c[i][0], dd[i][0], lam);
        o.y = (col + 1 < n_loc) ? mu_ratio(h.y, c[i][1], dd[i][1], lam) : 0.f;
        o.z = (col + 2 < n_loc) ? mu_ratio(h.z, c[i][2], dd[i][2], lam) : 0.f;
        o.w = (col + 3 < n_loc) ? mu_ratio(h.w, c[i][3], dd[i][3], lam) : 0.f;
        *reinterpret_cast<float4*>(Hn + (int64_t)krow * ldh + col) = o;
    }
}

// ---------------------------------------------------------------------------------------
// Out_partial[split][kb0 + ., col] = sum_{r in split} L[r][kb0 + .] * R[r][col]
// Used for G = W^T W (L = R = W).  Deterministic: partials are summed in fixed order by
// k_sum_partials, so every rank derives a bit-identical G from its bit-identical W.
//   grid.x = column tiles (of kp), grid.y = k blocks, grid.z = row splits.
// ---------------------------------------------------------------------------------------
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_ltr_partial_simt(const DevState* __restrict__ st, const float* __restrict__ L, int64_t ldl,
                   const float* __restrict__ R, int64_t ldr, int64_t r_ncols, int64_t rows,
                   int64_t rows_per_split, float* __restrict__ partial, int64_t out_ld,
                   int64_t out_rows, int64_t rps = 0, int rsh = kNoPanelShift) {
    // rps / rsh: panel layout of R when R is the data matrix X (common.cuh); row-major by default
    if (st->stop) return;
    constexpr int TK = KB / 8;
    __shared__ __align__(16) float Rs[2][TILE_DK][TILE_N];
    __shared__ __align__(16) float Ls[2][TILE_DK][KB];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t col0 = (int64_t)blockIdx.x * TILE_N;
    const int kb0 = blockIdx.y * KB;
    const int64_t r_begin = (int64_t)blockIdx.z * rows_per_split;
    const int64_t r_end = min(rows, r_begin + rows_per_split);
    float acc[TK][4];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    tile_mac<KB>(acc, L, ldl, kb0, R + xpanel_off(col0, rps, rsh), ldr, col0, min(r_ncols, ((col0 >> rsh) + 1) << rsh),
                 r_begin, r_end, Rs, Ls);
    float* out = partial + (int64_t)blockIdx.z * out_rows * out_ld;
    const int64_t col = col0 + tx * 4;
#pragma unroll
    for (int i = 0; i < TK; ++i) {
        const int krow = kb0 + ty * TK + i;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (col + j < r_ncols) out[(int64_t)krow * out_ld + col + j] = acc[i][j];
    }
}

__global__ void k_sum_partials(const DevState* __restrict__ st, const float* __restrict__ partial,
                               int nsplit, int64_t count, float* __restrict__ out) {
    if (st->stop) return;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    float s = 0.f;
    for (int p = 0; p < nsplit; ++p) s += partial[(int64_t)p * count + i];
    out[i] = s;
}

// ---------------------------------------------------------------------------------------
// P[row][kb0 + .] += sum_{c in column range} X[row][c] * H[kb0 + .][c]       (X H^T partials)
// Also used for H H^T (X := H, rows := kp).  Accumulated with fp32 atomics into the packed
// partial buffer that is all-reduced over ranks.
//   grid.x = row blocks of 128, grid.y = column splits, grid.z = k blocks.
// ---------------------------------------------------------------------------------------
constexpr int XHT_CK = 32;
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_xht_simt(const DevState* __restrict__ st, const float* __restrict__ X, int64_t ldx, int64_t rows,
           const float* __restrict__ H, int64_t ldh, int64_t n_loc, int64_t cols_per_split,
           float* __restrict__ P, int64_t ldp, int nrb_x, int64_t rows_h, float* __restrict__ PB,
           float* __restrict__ Ppart, int64_t part_stride,
           int64_t xps = 0, int xsh = kNoPanelShift) {
    // Row blocks [0, nrb_x) of the grid compute X H^T; when PB != nullptr the remaining row blocks compute H H^T in
    // the same launch (the streamed operand is then H itself, rows_h rows, output PB) - one launch instead of two.
    // Column splits (gridDim.y) are combined DETERMINISTICALLY when Ppart != nullptr: every split stores its block in
    // copy blockIdx.y of the [A | B] layout (part_stride floats apart) and k_sum_copies adds the copies in split
    // order into P afterwards (no clearing, no atomics: W is bit-reproducible from run to run; an in-kernel
    // "last arrival sums" variant cost cfg1 8.7 us per iteration in fences and ticket round trips).
    // Ppart == nullptr: fp32 atomics into a cleared P.
    if (st->stop) return;
    const int64_t out_off = ((int)blockIdx.x >= nrb_x) ? (PB - P) : 0;
    if ((int)blockIdx.x >= nrb_x) { X = H; ldx = ldh; rows = rows_h; P = PB; xps = 0; xsh = kNoPanelShift; }
    constexpr int TK = KB / 8;
    __shared__ float Xs[128][XHT_CK + 1];
    __shared__ __align__(16) float Hs[XHT_CK][KB];
    const int tid = threadIdx.x;
    const int tr = tid & 31, tk = tid >> 5;
    const int64_t row0 = (int64_t)((int)blockIdx.x >= nrb_x ? (int)blockIdx.x - nrb_x : (int)blockIdx.x) * 128;
    const int kb0 = blockIdx.z * KB;
    const int64_t c_begin = (int64_t)blockIdx.y * cols_per_split;
    const int64_t c_end = min(n_loc, c_begin + cols_per_split);

    float acc[4][TK];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < TK; ++j) acc[i][j] = 0.f;

    for (int64_t c0 = c_begin; c0 < c_end; c0 += XHT_CK) {
        // X chunk: 128 rows x 32 cols
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            int f = tid + t * SIMT_THREADS;
            int row = f >> 3, c4 = f & 7;
            int64_t r = row0 + row, c = c0 + c4 * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < rows && c < c_end) {
                v = *reinterpret_cast<const float4*>(X + xpanel_off(c0, xps, xsh) + r * ldx + c);   // 32-column chunk: one panel
                if (c + 1 >= c_end) v.y = 0.f;
                if (c + 2 >= c_end) v.z = 0.f;
                if (c + 3 >= c_end) v.w = 0.f;
            }
            Xs[row][c4 * 4 + 0] = v.x; Xs[row][c4 * 4 + 1] = v.y;
            Xs[row][c4 * 4 + 2] = v.z; Xs[row][c4 * 4 + 3] = v.w;
        }
        // H chunk: KB rows x 32 cols, stored transposed [col][k]
        for (int f = tid; f < KB * XHT_CK / 4; f += SIMT_THREADS) {
            int krow = f >> 3, c4 = f & 7;
            int64_t c = c0 + c4 * 4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c < c_end) {
                v = *reinterpret_cast<const float4*>(H + (int64_t)(kb0 + krow) * ldh + c);
                if (c + 1 >= c_end) v.y = 0.f;
                if (c + 2 >= c_end) v.z = 0.f;
                if (c + 3 >= c_end) v.w = 0.f;
            }
            Hs[c4 * 4 + 0][krow] = v.x; Hs[c4 * 4 + 1][krow] = v.y;
            Hs[c4 * 4 + 2][krow] = v.z; Hs[c4 * 4 + 3][krow] = v.w;
        }
        __syncthreads();
#pragma unroll 8
        for (int c = 0; c < XHT_CK; ++c) {
            float x[4], h[TK];
#pragma unroll
            for (int i = 0; i < 4; ++i) x[i] = Xs[tr + 32 * i][c];
#pragma unroll
            for (int j = 0; j < TK; ++j) h[j] = Hs[c][tk * TK + j];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < TK; ++j) acc[i][j] = fmaf(x[i], h[j], acc[i][j]);
        }
        __syncthreads();
    }
    if (Ppart == nullptr) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t r = row0 + tr + 32 * i;
            if (r < rows) {
#pragma unroll
                for (int j = 0; j < TK; ++j) atomicAdd(P + r * ldp + kb0 + tk * TK + j, acc[i][j]);
            }
        }
        return;
    }
    // deterministic mode: this split's block goes into its own copy of the [A | B] layout (or straight into P when
    // there is only one split); k_sum_copies then adds the copies in split order
    float* dst = ((int)gridDim.y > 1) ? Ppart + (int64_t)blockIdx.y * part_stride + out_off : P;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int64_t r = row0 + tr + 32 * i;
        if (r < rows) {
#pragma unroll
            for (int j = 0; j < TK; ++j) dst[r * ldp + kb0 + tk * TK + j] = acc[i][j];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Semi-NMF helpers (pymf/snmf.py:67-90).
// ---------------------------------------------------------------------------------------
// G+ = (|G| + G)/2, G- = (|G| - G)/2                                            (:73-77, applied to W^T W, :81-83)
__global__ void k_split_posneg(const DevState* __restrict__ st, const float* __restrict__ G, int64_t cnt,
                               float* __restrict__ Gpos, float* __restrict__ Gneg) {
    if (st->stop) return;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < cnt) { const float g = G[i]; Gpos[i] = fmaxf(g, 0.f); Gneg[i] = fmaxf(-g, 0.f); }
}

// Dp = G+ H, Dn = G- H (kp x n_loc each) for the tensor-core H-update kernels, whose epilogue reads them
// instead of their own G H accumulator in Semi-NMF mode.  Same tiling as k_h_update_simt.
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_gh_posneg_simt(const DevState* __restrict__ st, const float* __restrict__ Gpos, const float* __restrict__ Gneg,
                 const float* __restrict__ Hc, int64_t ldh, int64_t n_loc, int kp,
                 float* __restrict__ Dp, float* __restrict__ Dn) {
    if (st->stop) return;
    constexpr int TK = KB / 8;
    __shared__ __align__(16) float Rs[2][TILE_DK][TILE_N];
    __shared__ __align__(16) float Ls[2][TILE_DK][KB];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t col0 = (int64_t)blockIdx.x * TILE_N;
    const int kb0 = blockIdx.y * KB;
    float dp[TK][4], dn[TK][4];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { dp[i][j] = 0.f; dn[i][j] = 0.f; }
    tile_mac<KB>(dp, Gpos, kp, kb0, Hc, ldh, col0, n_loc, 0, kp, Rs, Ls);
    tile_mac<KB>(dn, Gneg, kp, kb0, Hc, ldh, col0, n_loc, 0, kp, Rs, Ls);
    const int64_t col = col0 + tx * 4;
    if (col >= n_loc) return;
#pragma unroll
    for (int i = 0; i < TK; ++i) {
        const int64_t o = (int64_t)(kb0 + ty * TK + i) * ldh + col;
        *reinterpret_cast<float4*>(Dp + o) = make_float4(dp[i][0], dp[i][1], dp[i][2], dp[i][3]);
        *reinterpret_cast<float4*>(Dn + o) = make_float4(dn[i][0], dn[i][1], dn[i][2], dn[i][3]);
    }
}

// Binv = inverse of the leading k x k block of B = H H^T (row-major, leading dimension kp), fp64 Gauss-Jordan
// with partial pivoting in ONE CTA (np.linalg.inv of pymf/snmf.py:70 is LU with partial pivoting; k <= 128 here).
// work: k x 2k doubles [B | I].  A singular B leaves inf / nan in Binv (the reference raises LinAlgError).
__global__ void __launch_bounds__(256)
k_inv_f64(const DevState* __restrict__ st, const float* __restrict__ B, int kp, int k,
          double* __restrict__ work, double* __restrict__ Binv) {
    if (st->stop) return;
    const int n2 = 2 * k;
    __shared__ int s_piv;
    __shared__ double s_red[256];
    __shared__ int s_idx[256];
    for (int f = threadIdx.x; f < k * n2; f += blockDim.x) {
        const int r = f / n2, c = f % n2;
        work[f] = c < k ? (double)B[(int64_t)r * kp + c] : (c - k == r ? 1.0 : 0.0);
    }
    __syncthreads();
    for (int p = 0; p < k; ++p) {
        // pivot search in column p, rows p..k-1
        double best = -1.0; int bi = p;
        for (int r = p + threadIdx.x; r < k; r += blockDim.x) {
            const double v = fabs(work[(int64_t)r * n2 + p]);
            if (v > best) { best = v; bi = r; }
        }
        s_red[threadIdx.x] = best; s_idx[threadIdx.x] = bi;
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
            if (threadIdx.x < s) {
                const double o = s_red[threadIdx.x + s];
                const int oi = s_idx[threadIdx.x + s];
                if (o > s_red[threadIdx.x] || (o == s_red[threadIdx.x] && oi < s_idx[threadIdx.x])) {
                    s_red[threadIdx.x] = o; s_idx[threadIdx.x] = oi;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) s_piv = s_idx[0];
        __syncthreads();
        const int q = s_piv;
        if (q != p)
            for (int c = threadIdx.x; c < n2; c += blockDim.x) {
                const double t = work[(int64_t)p * n2 + c];
                work[(int64_t)p * n2 + c] = work[(int64_t)q * n2 + c];
                work[(int64_t)q * n2 + c] = t;
            }
        __syncthreads();
        const double inv = 1.0 / work[(int64_t)p * n2 + p];
        __syncthreads();
        for (int c = threadIdx.x; c < n2; c += blockDim.x) work[(int64_t)p * n2 + c] *= inv;
        __syncthreads();
        // eliminate column p from every other row; the factors are read before any row is changed
        for (int f = threadIdx.x; f < k * n2; f += blockDim.x) {
            const int r = f / n2, c = f % n2;
            if (r == p || c == p) continue;
            work[f] -= work[(int64_t)r * n2 + p] * work[(int64_t)p * n2 + c];
        }
        __syncthreads();
        for (int r = threadIdx.x; r < k; r += blockDim.x)
            if (r != p) work[(int64_t)r * n2 + p] = 0.0;
        __syncthreads();
    }
    for (int f = threadIdx.x; f < k * k; f += blockDim.x) Binv[f] = work[(int64_t)(f / k) * n2 + k + f % k];
}

// Semi-NMF W update (pymf/snmf.py:67-70): W = (X H^T) (H H^T)^-1 = A Binv, fp64 accumulation; columns >= k stay 0.
__global__ void __launch_bounds__(SIMT_THREADS)
k_update_w_snmf(const DevState* __restrict__ st, const float* __restrict__ A, const double* __restrict__ Binv,
                float* __restrict__ Wn, int64_t d, int kp, int k) {
    if (st->stop) return;
    extern __shared__ float ws[];   // UW_ROWS_S x kp rows of A
    constexpr int ROWS = 8;
    const int64_t row0 = (int64_t)blockIdx.x * ROWS;
    const int nrows = (int)min((int64_t)ROWS, d - row0);
    for (int f = threadIdx.x; f < nrows * kp; f += blockDim.x) ws[f] = A[row0 * kp + f];
    __syncthreads();
    for (int f = threadIdx.x; f < nrows * kp; f += blockDim.x) {
        const int r = f / kp, j = f % kp;
        double s = 0.0;
        if (j < k)
            for (int l = 0; l < k; ++l) s = fma((double)ws[r * kp + l], Binv[(int64_t)l * k + j], s);
        Wn[(row0 + r) * kp + j] = (float)s;
    }
}

// ---------------------------------------------------------------------------------------
// W update (pymf/nmf.py:128-132), replicated on every rank, O(d k^2):
//   Wn[i][j] = W[i][j] * A[i][j] / (sum_l W[i][l] B[l][j] + 1e-9)
// UW_ROWS rows of W per CTA staged in shared memory.  A thread owns ONE column j for a group of UW_RT rows, so that an
// element B[l][j] (read through L1/L2, coalesced over j) is loaded once per UW_RT outputs and the W values are
// shared-memory broadcasts (ncu, cold: 80 -> 60 us at 16384 x 128; the W update is ~1 % of a cfg3 step on 8 GPUs).  Every output is
// summed in blocks of UW_SEG terms, the block sums added in order.
// ---------------------------------------------------------------------------------------
constexpr int UW_ROWS = 8;      // rows per CTA
constexpr int UW_RT = 4;        // rows per thread
constexpr int UW_SEG = 16;      // terms per partial sum of W B
__global__ void __launch_bounds__(SIMT_THREADS)
k_update_w(const DevState* __restrict__ st, const float* __restrict__ W, const float* __restrict__ A,
           const float* __restrict__ B, float* __restrict__ Wn, int64_t d, int kp, float lam) {
    if (st->stop) return;
    extern __shared__ float ws[];   // UW_ROWS x kp
    const int64_t row0 = (int64_t)blockIdx.x * UW_ROWS;
    const int nrows = (int)min((int64_t)UW_ROWS, d - row0);
    for (int f = threadIdx.x; f < UW_ROWS * kp; f += blockDim.x) ws[f] = f < nrows * kp ? W[row0 * kp + f] : 0.f;
    __syncthreads();
    // work item = (row group rg of UW_RT rows, column j)
    for (int f = threadIdx.x; f < (UW_ROWS / UW_RT) * kp; f += blockDim.x) {
        const int rg = f / kp, j = f % kp;
        const float* wr = ws + rg * UW_RT * kp;
        float s[UW_RT];
#pragma unroll
        for (int r = 0; r < UW_RT; ++r) s[r] = 0.f;
        for (int l0 = 0; l0 < kp; l0 += UW_SEG) {      // blocked sum: one fp32 chain over kp = 512 exceeded 1e-5
            float t[UW_RT];
#pragma unroll
            for (int r = 0; r < UW_RT; ++r) t[r] = 0.f;
#pragma unroll 4
            for (int l = l0; l < l0 + UW_SEG; ++l) {    // kp is a multiple of UW_SEG
                const float b = __ldg(B + (int64_t)l * kp + j);
#pragma unroll
                for (int r = 0; r < UW_RT; ++r) t[r] = fmaf(wr[r * kp + l], b, t[r]);
            }
#pragma unroll
            for (int r = 0; r < UW_RT; ++r) s[r] += t[r];
        }
#pragma unroll
        for (int r = 0; r < UW_RT; ++r) {
            if (rg * UW_RT + r < nrows) {
                const int64_t o = (row0 + rg * UW_RT + r) * kp + j;
                Wn[o] = mu_ratio(wr[r * kp + j], A[o], s[r], lam);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// Error (pymf/nmf.py:100-114 by the trace identity) + converged() (:134-139), fp64 combine.
//   ferr = sqrt(max(0, ||X||^2 - 2 <W, A> + <G, B>)),  A = X H^T, B = H H^T, G = W^T W.
// Block partial sums are combined in fixed order by the last block (deterministic, so all
// ranks take the same stop decision).
// ---------------------------------------------------------------------------------------
constexpr int ERR_BLOCKS = 128;
__global__ void __launch_bounds__(256)
k_err(DevState* __restrict__ st, const float* __restrict__ W, const float* __restrict__ A,
      int64_t n_wa, const float* __restrict__ G, const float* __restrict__ B, int64_t n_gb,
      double* __restrict__ scratch /* 2*ERR_BLOCKS */, double* __restrict__ ferr,
      double n_samples, int early_stop, int direct) {
    if (st->stop) return;
    __shared__ double s_wa[256], s_gb[256];
    __shared__ bool is_last;
    double wa = 0.0, gb = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_wa;
         i += (int64_t)gridDim.x * blockDim.x)
        wa += (double)W[i] * (double)A[i];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_gb;
         i += (int64_t)gridDim.x * blockDim.x)
        gb += (double)G[i] * (double)B[i];
    s_wa[threadIdx.x] = wa; s_gb[threadIdx.x] = gb;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) { s_wa[threadIdx.x] += s_wa[threadIdx.x + s]; s_gb[threadIdx.x] += s_gb[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        scratch[blockIdx.x] = s_wa[0];
        scratch[ERR_BLOCKS + blockIdx.x] = s_gb[0];
        __threadfence();
        unsigned t = atomicAdd(&st->ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last && threadIdx.x == 0) {
        __threadfence();
        double twa = 0.0, tgb = 0.0;
        for (int b = 0; b < (int)gridDim.x; ++b) {
            twa += ((volatile double*)scratch)[b];
            tgb += ((volatile double*)scratch)[ERR_BLOCKS + b];
        }
        double e2 = direct ? st->resid : st->xx - 2.0 * twa + tgb;
        // near-exact fit: the identity cancels (see kTraceCancel).  Flag it for the host and take no convergence
        // decision from a value that is mostly rounding noise.
        const bool cancelled = !direct && e2 < kTraceCancel * st->xx;
        if (cancelled) st->cancel = 1;
        double e = sqrt(e2 > 0.0 ? e2 : 0.0);
        st->last_ferr = e;
        st->ticket = 0;
        if (ferr) {
            const int iter = st->it;       // device-side iteration counter (reset by the host at the start of a run)
            st->it = iter + 1;
            ferr[iter] = e;
            if (early_stop && iter > 1 && !cancelled) {
                double derr = fabs(e - ferr[iter - 1]) / n_samples;
                if (derr < kEpsConv) { st->stop = 1; st->n_exec = iter + 1; }
            }
        }
    }
}

// ||X||_F^2 in fp64 (once per data set).
constexpr int XX_BLOCKS = 1184;   // 8 x 148
__global__ void __launch_bounds__(256)
k_xx(DevState* __restrict__ st, const float* __restrict__ X, int64_t ldx, int64_t d, int64_t n_loc,
     double* __restrict__ scratch /* XX_BLOCKS */, int64_t xps, int xsh) {
    __shared__ double s[256];
    __shared__ bool is_last;
    double acc = 0.0;
    const int64_t n4 = (n_loc + 3) / 4;
    const int64_t total = d * n4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / n4, c = (i % n4) * 4;
        const float4 v = *reinterpret_cast<const float4*>(X + xpanel_off(c, xps, xsh) + r * ldx + c);
        float p = v.x * v.x;
        if (c + 1 < n_loc) p = fmaf(v.y, v.y, p);
        if (c + 2 < n_loc) p = fmaf(v.z, v.z, p);
        if (c + 3 < n_loc) p = fmaf(v.w, v.w, p);
        acc += (double)p;
    }
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int k = 128; k > 0; k >>= 1) {
        if (threadIdx.x < k) s[threadIdx.x] += s[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        scratch[blockIdx.x] = s[0];
        __threadfence();
        is_last = (atomicAdd(&st->ticket2, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last && threadIdx.x == 0) {
        __threadfence();
        double t = 0.0;
        for (int b = 0; b < (int)gridDim.x; ++b) t += ((volatile double*)scratch)[b];
        st->xx_local = t;
        st->xx = t;          // overwritten by the all-reduce when there are several ranks
        st->ticket2 = 0;
    }
}


// ---------------------------------------------------------------------------------------
// Direct residual  sum_{r,c} (X[r][c] - (W H)[r][c])^2  (pymf/nmf.py:110 as written), used for
// small problems where one more pass is cheap: the trace identity cancels catastrophically
// when ||X - WH||^2 << ||X||^2 (e.g. the reference's own 3x50 test matrix, which k=4 fits
// exactly).  Wt = W^T (kp x ldwt, zero padded).  grid.x = column tiles, grid.y = row blocks of KB.
// fp32 products, fp64 accumulation of squares, deterministic final sum.
// ---------------------------------------------------------------------------------------
__global__ void k_transpose_w(const DevState* __restrict__ st, const float* __restrict__ W, int64_t d, int kp,
                              float* __restrict__ Wt, int64_t ldwt) {
    if (st->stop) return;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= d * kp) return;
    const int64_t r = i / kp;
    const int l = (int)(i % kp);
    Wt[(int64_t)l * ldwt + r] = W[i];
}

template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_resid_simt(DevState* __restrict__ st, const float* __restrict__ X, int64_t ldx,
             const float* __restrict__ Wt, int64_t ldwt, const float* __restrict__ H, int64_t ldh,
             int64_t d, int64_t n_loc, int kp, double* __restrict__ partial, int64_t xps, int xsh) {
    if (st->stop) return;
    constexpr int TK = KB / 8;
    __shared__ __align__(16) float Rs[2][TILE_DK][TILE_N];
    __shared__ __align__(16) float Ls[2][TILE_DK][KB];
    __shared__ double red[SIMT_THREADS];
    __shared__ bool is_last;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t col0 = (int64_t)blockIdx.x * TILE_N;
    const int r0 = blockIdx.y * KB;
    float acc[TK][4];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    tile_mac<KB>(acc, Wt, ldwt, r0, H, ldh, col0, n_loc, 0, kp, Rs, Ls);   // (W H) tile
    double s = 0.0;
    const int64_t col = col0 + tx * 4;
#pragma unroll
    for (int i = 0; i < TK; ++i) {
        const int64_t r = r0 + ty * TK + i;
        if (r < d && col < n_loc) {
            const float4 x = *reinterpret_cast<const float4*>(X + xpanel_off(col0, xps, xsh) + r * ldx + col);
            float e = x.x - acc[i][0];
            s += (double)e * (double)e;
            if (col + 1 < n_loc) { e = x.y - acc[i][1]; s += (double)e * (double)e; }
            if (col + 2 < n_loc) { e = x.z - acc[i][2]; s += (double)e * (double)e; }
            if (col + 3 < n_loc) { e = x.w - acc[i][3]; s += (double)e * (double)e; }
        }
    }
    red[threadIdx.x] = s;
    __syncthreads();
    for (int k = SIMT_THREADS / 2; k > 0; k >>= 1) {
        if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
        __syncthreads();
    }
    const unsigned nblocks = gridDim.x * gridDim.y;
    if (threadIdx.x == 0) {
        partial[blockIdx.y * gridDim.x + blockIdx.x] = red[0];
        __threadfence();
        is_last = (atomicAdd(&st->ticket3, 1u) == nblocks - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double t = 0.0;
        for (unsigned b = threadIdx.x; b < nblocks; b += SIMT_THREADS) t += ((volatile double*)partial)[b];
        red[threadIdx.x] = t;     // fixed assignment of partials to threads -> deterministic
        __syncthreads();
        for (int k = SIMT_THREADS / 2; k > 0; k >>= 1) {
            if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
            __syncthreads();
        }
        if (threadIdx.x == 0) { st->resid_local = red[0]; st->resid = red[0]; st->ticket3 = 0; }
    }
}

// --- small utilities ---------------------------------------------------------------------
__global__ void k_zero(const DevState* __restrict__ st, float* __restrict__ p, int64_t count) {
    if (st->stop) return;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < count; i += stride) p[i] = 0.f;
}

// dst (rows x ldd, fp32) <- src (rows x cols, T contiguous with leading dimension lds)
template <typename T>
__global__ void k_cast_in(const T* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd,
                          int64_t rows, int64_t cols, int64_t dcol0 = 0, int64_t xps = 0, int xsh = kNoPanelShift) {
    // dst element (r, dcol0 + c) of a matrix in the layout of common.cuh (row-major by default; dst = its base)
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < rows * cols; i += stride) {
        const int64_t r = i / cols, c = dcol0 + i % cols;
        dst[xpanel_off(c, xps, xsh) + r * ldd + c] = (float)src[r * lds + (c - dcol0)];
    }
}
// Ingest: rows x cols block of a host-layout staging buffer (element type T, leading dimension lds) -> X in the
// layout of common.cuh at (row, dcol0 + col); dst is X's base advanced by (first row) * ldd.  One thread moves four
// consecutive columns (cols and dcol0 are multiples of 4 except for the ragged tail), blockIdx.y strides the rows:
// no integer division per element (k_cast_in's i / cols made the scatter of a 64 MiB chunk cost as much as its DMA).
template <typename T>
__global__ void __launch_bounds__(256)
k_place_x(const T* __restrict__ src, int64_t lds, float* __restrict__ dst, int64_t ldd, int64_t rows, int64_t cols,
          int64_t dcol0, int64_t xps, int xsh) {
    const int64_t c4 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (c4 >= cols) return;
    const int64_t c = dcol0 + c4;
    float* out = dst + xpanel_off(c, xps, xsh) + c;
    const bool vec = c4 + 3 < cols && ((c & 3) == 0) && ((ldd & 3) == 0) && ((xps & 3) == 0);
    for (int64_t r = blockIdx.y; r < rows; r += gridDim.y) {
        const T* in = src + r * lds + c4;
        if (vec) {
            *reinterpret_cast<float4*>(out + r * ldd) = make_float4((float)in[0], (float)in[1], (float)in[2], (float)in[3]);
        } else {
            for (int j = 0; j < 4 && c4 + j < cols; ++j) {
                const int64_t cj = c + j;
                dst[xpanel_off(cj, xps, xsh) + r * ldd + cj] = (float)in[j];
            }
        }
    }
}
template <typename T>
__global__ void k_cast_out(const float* __restrict__ src, int64_t lds, T* __restrict__ dst, int64_t ldd,
                           int64_t rows, int64_t cols) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < rows * cols; i += stride) {
        const int64_t r = i / cols, c = i % cols;
        dst[r * ldd + c] = (T)src[r * lds + c];
    }
}

// dst[r][c] = U[0,1) hash(seed, r * gen_ld + gen_col0 + c)  for r < rows, c < cols (pad stays 0)
__global__ void k_gen_uniform(float* __restrict__ dst, int64_t ldd, int64_t rows, int64_t cols,
                              uint64_t seed, int64_t gen_ld, int64_t gen_col0, int64_t xps = 0, int xsh = kNoPanelShift) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < rows * cols; i += stride) {
        const int64_t r = i / cols, c = i % cols;
        dst[xpanel_off(c, xps, xsh) + r * ldd + c] = hash_uniform(seed, (uint64_t)(r * gen_ld + gen_col0 + c));
    }
}

__global__ void k_fill(float* __restrict__ p, int64_t count, float v) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < count; i += stride) p[i] = v;
}

}  // namespace pymfb
