// kernels_sparse.cuh - the passes over a sparse X (pymfb_upload_x_csc): CUDA-core fp32 FMA, fp32 accumulation in a
// fixed order, so every result is deterministic without atomics.
//
// X is held twice on the device:
//   CSC               colptr (int64, n_local + 1), rowidx (int32, rows strictly increasing within a column), vals (fp32,
//                     zero-padded to a multiple of 4 so that k_xx reads it as a 1 x nnz row)    -> H update, residual
//   column-panel CSR  for each panel of pw consecutive columns the panel's entries by row: rowptr[p * d + r] .. rowptr[p * d
//                     + r + 1] are row r's entries in panel p, column order kept (stable sort)   -> X H^T
// The panel split keeps the rows of H^T one X H^T launch gathers (pw x kp fp32) inside about half of the L2.
//
// Per iteration (the dense k x k x n products stay on the CUDA cores, kernels_simt.cuh):
//   D  <- G H  (or G+ H, G- H for Semi-NMF)         k_gh_simt / k_gh_posneg_simt
//   H' <- ratio(H, W^T X, D), H'^T                  k_h_update_csc        (CSC, gathers rows of W)
//   A  <- X H'^T                                    k_xht_csr, one launch per panel (CSR, gathers rows of H'^T)
//   B  <- H' H'^T = (H'^T)^T H'^T                   k_ltr_partial_simt + k_sum_partials on H'^T
#pragma once
#include "common.cuh"
#include "kernels_simt.cuh"

namespace pymfb {
namespace sp {

constexpr int SP_THREADS = 256;
constexpr int SP_COLS_PER_GROUP = 8;     // columns one lane group contracts in a k_h_update_csc tile
constexpr int SP_HEAVY = 512;            // a column with more non-zeros is contracted by all groups of the CTA

// pymfb_upload_x_csc / pymfb_upload_x_sparse_device validation: bits of the flag
enum { BAD_START = 1, BAD_PTR_ORDER = 2, BAD_END = 4, BAD_ROW = 8, BAD_ROW_ORDER = 16, BAD_COL = 32 };

// One warp per column.  Entries are only read inside [0, nnz) and only for columns whose pointers are ordered.
__global__ void k_csc_validate(const int64_t* __restrict__ colptr, const int32_t* __restrict__ rowidx, int64_t n,
                               int64_t nnz, int64_t d, int* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    int bad = 0;
    if (warp == 0 && lane == 0) {
        if (colptr[0] != 0) bad |= BAD_START;
        if (colptr[n] != nnz) bad |= BAD_END;
    }
    for (int64_t c = warp; c < n; c += nwarps) {
        const int64_t a = colptr[c], b = colptr[c + 1];
        if (b < a) { bad |= BAD_PTR_ORDER; continue; }
        if (a < 0 || b > nnz) continue;      // then colptr[0] != 0, colptr[n] != nnz or a later decrease is flagged
        for (int64_t e = a + lane; e < b; e += 32) {
            const int32_t r = rowidx[e];
            if (r < 0 || (int64_t)r >= d) bad |= BAD_ROW;
            if (e > a && rowidx[e - 1] >= r) bad |= BAD_ROW_ORDER;
        }
    }
    if (bad) atomicOr(flag, bad);
}

// colof[e] = column of CSC entry e (one warp per column)
__global__ void k_csc_cols(const int64_t* __restrict__ colptr, int64_t n, int32_t* __restrict__ colof) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t c = warp; c < n; c += nwarps)
        for (int64_t e = colptr[c] + lane; e < colptr[c + 1]; e += 32) colof[e] = (int32_t)c;
}

// sort key (panel, row) and payload (entry index) of every CSC entry
__global__ void k_csr_keys(const int32_t* __restrict__ rowidx, const int32_t* __restrict__ colof, int64_t nnz, int64_t d,
                           int64_t pw, uint64_t* __restrict__ keys, uint32_t* __restrict__ perm) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        keys[e] = (uint64_t)(colof[e] / pw) * (uint64_t)d + (uint64_t)rowidx[e];
        perm[e] = (uint32_t)e;
    }
}

__global__ void k_csr_gather(const uint32_t* __restrict__ perm, const int32_t* __restrict__ colof,
                             const float* __restrict__ vals, int64_t nnz, int32_t* __restrict__ ccol,
                             float* __restrict__ cval) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride) {
        const uint32_t e = perm[i];
        ccol[i] = colof[e];
        cval[i] = vals[e];
    }
}

// rowptr[key] = first position of a sorted key >= key, key in [0, nkeys]
__global__ void k_csr_rowptr(const uint64_t* __restrict__ skeys, int64_t nnz, int64_t nkeys, int64_t* __restrict__ rowptr) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k <= nkeys; k += stride) {
        int64_t lo = 0, hi = nnz;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (skeys[mid] < (uint64_t)k) lo = mid + 1; else hi = mid;
        }
        rowptr[k] = lo;
    }
}

// ---------------------------------------------------------------------------------------
// Device canonicalisation (pymfb_upload_x_sparse_device): a COO, CSR or CSC input with index type T (int32 / int64),
// in any order and with duplicates, becomes the canonical CSC of pymfb_upload_x_csc.
//   check    k_sp_check_ptr (CSR / CSC pointers), k_sp_check_idx (every index in range); nothing below runs unless
//            both passed
//   keys     key = col * d + row, payload = input position (k_sp_keys_coo, or k_sp_keys_ptr for CSR / CSC)
//   sort     stable radix sort (sort_pairs in pymfb.cu): duplicates end up adjacent, in input order
//   runs     k_sp_heads + an in-place inclusive scan give each run of equal keys its output slot; k_sp_sum_runs adds
//            the run in fp64 in input order and rounds once to fp32 (explicit zeros are kept, as scipy's
//            sum_duplicates keeps them)
//   colptr   k_sp_colptr: binary search of c * d in the unique keys
// ---------------------------------------------------------------------------------------
// ptr (m + 1 entries): ptr[0] == 0, ptr[m] == nnz, non-decreasing
template <typename T>
__global__ void k_sp_check_ptr(const T* __restrict__ ptr, int64_t m, int64_t nnz, int* __restrict__ flag) {
    const int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    int bad = 0;
    if (i0 == 0) {
        if (ptr[0] != 0) bad |= BAD_START;
        if ((int64_t)ptr[m] != nnz) bad |= BAD_END;
    }
    for (int64_t i = i0; i < m; i += stride)
        if (ptr[i + 1] < ptr[i]) bad |= BAD_PTR_ORDER;
    if (bad) atomicOr(flag, bad);
}

// every idx[e] in [0, bound), else `bit`
template <typename T>
__global__ void k_sp_check_idx(const T* __restrict__ idx, int64_t nnz, int64_t bound, int bit, int* __restrict__ flag) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    int bad = 0;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        const int64_t v = (int64_t)idx[e];
        if (v < 0 || v >= bound) bad = bit;
    }
    if (bad) atomicOr(flag, bad);
}

template <typename T>
__global__ void k_sp_keys_coo(const T* __restrict__ rows, const T* __restrict__ cols, int64_t nnz, int64_t d,
                              uint64_t* __restrict__ keys, uint32_t* __restrict__ perm) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += stride) {
        keys[e] = (uint64_t)cols[e] * (uint64_t)d + (uint64_t)rows[e];
        perm[e] = (uint32_t)e;
    }
}

// CSR (ptr = d + 1 row pointers, idx = columns) or CSC (ptr = n + 1 column pointers, idx = rows): one warp per row /
// column.  Only after k_sp_check_ptr has passed: a bad pointer array would write outside keys / perm.
template <typename T>
__global__ void k_sp_keys_ptr(const T* __restrict__ ptr, const T* __restrict__ idx, int64_t m, int64_t d, int csc,
                              uint64_t* __restrict__ keys, uint32_t* __restrict__ perm) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t o = warp; o < m; o += nwarps)
        for (int64_t e = (int64_t)ptr[o] + lane; e < (int64_t)ptr[o + 1]; e += 32) {
            const uint64_t i = (uint64_t)idx[e];
            keys[e] = csc ? (uint64_t)o * (uint64_t)d + i : i * (uint64_t)d + (uint64_t)o;
            perm[e] = (uint32_t)e;
        }
}

// head[i] = 1 where a run of equal sorted keys starts
__global__ void k_sp_heads(const uint64_t* __restrict__ skeys, int64_t nnz, uint32_t* __restrict__ head) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride)
        head[i] = (i == 0 || skeys[i] != skeys[i - 1]) ? 1u : 0u;
}

// One thread per run: the run's values summed in fp64 in input order (the stable sort kept it), rounded once to fp32,
// stored at slot[i] - 1 (slot = inclusive scan of the heads) with its row and its key.  A run of many duplicates is
// added by one thread, serially: fine for the few duplicates real data has, slow for a pathological input.
template <typename V>
__global__ void k_sp_sum_runs(const uint64_t* __restrict__ skeys, const uint32_t* __restrict__ sperm,
                              const uint32_t* __restrict__ slot, const V* __restrict__ vals, int64_t nnz, int64_t d,
                              int32_t* __restrict__ rowidx, float* __restrict__ vout, uint64_t* __restrict__ ukeys) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride) {
        const uint64_t key = skeys[i];
        if (i > 0 && skeys[i - 1] == key) continue;
        double s = 0.0;
        int64_t j = i;
        do { s += (double)vals[sperm[j]]; ++j; } while (j < nnz && skeys[j] == key);
        const int64_t o = (int64_t)slot[i] - 1;
        rowidx[o] = (int32_t)(key % (uint64_t)d);
        vout[o] = (float)s;
        ukeys[o] = key;
    }
}

// colptr[c] = first unique key >= c * d, c in [0, n]
__global__ void k_sp_colptr(const uint64_t* __restrict__ ukeys, int64_t nu, int64_t n, int64_t d, int64_t* __restrict__ colptr) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c <= n; c += stride) {
        const uint64_t k = (uint64_t)c * (uint64_t)d;
        int64_t lo = 0, hi = nu;
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (ukeys[mid] < k) lo = mid + 1; else hi = mid;
        }
        colptr[c] = lo;
    }
}

// Ht (n_loc x kp) = H^T, H kp x ldh.  Rebuilds H^T after the host or a generator set H.
__global__ void k_h_transpose(const DevState* __restrict__ st, const float* __restrict__ H, int64_t ldh, int64_t n_loc,
                              int kp, float* __restrict__ Ht) {
    if (st->stop) return;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_loc * kp; i += stride) {
        const int64_t c = i / kp;
        const int j = (int)(i % kp);
        Ht[i] = H[(int64_t)j * ldh + c];
    }
}

// D = G H (kp x n_loc): the single-output form of k_gh_posneg_simt, same tiling and the same tile_mac order as the
// G H of k_h_update_simt.
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_gh_simt(const DevState* __restrict__ st, const float* __restrict__ G, const float* __restrict__ Hc, int64_t ldh,
          int64_t n_loc, int kp, float* __restrict__ D) {
    if (st->stop) return;
    constexpr int TK = KB / 8;
    __shared__ __align__(16) float Rs[2][TILE_DK][TILE_N];
    __shared__ __align__(16) float Ls[2][TILE_DK][KB];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t col0 = (int64_t)blockIdx.x * TILE_N;
    const int kb0 = blockIdx.y * KB;
    float acc[TK][4];
#pragma unroll
    for (int i = 0; i < TK; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    tile_mac<KB>(acc, G, kp, kb0, Hc, ldh, col0, n_loc, 0, kp, Rs, Ls);
    const int64_t col = col0 + tx * 4;
    if (col >= n_loc) return;
#pragma unroll
    for (int i = 0; i < TK; ++i)
        *reinterpret_cast<float4*>(D + (int64_t)(kb0 + ty * TK + i) * ldh + col) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
}

// acc += x * row[4 l .. 4 l + 3] over entries [e0, e1) in order; rows of Src (ld floats) picked by idx.  The entries
// are summed in blocks of SP_SEG, the block sums added to acc in order (a single fp32 chain over hundreds of entries
// carries as many roundings).
constexpr int SP_SEG = 32;
__device__ __forceinline__ void gather_mac_seq(float4& acc, const int32_t* __restrict__ idx, const float* __restrict__ val,
                                               int64_t e0, int64_t e1, const float* __restrict__ Src, int64_t ld, int off) {
    int64_t e = e0;
    for (; e + 4 <= e1; e += 4) {            // four gathers in flight, accumulated in entry order
        float x[4];
        float4 w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { x[u] = val[e + u]; w[u] = *reinterpret_cast<const float4*>(Src + (int64_t)idx[e + u] * ld + off); }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            acc.x = fmaf(x[u], w[u].x, acc.x); acc.y = fmaf(x[u], w[u].y, acc.y);
            acc.z = fmaf(x[u], w[u].z, acc.z); acc.w = fmaf(x[u], w[u].w, acc.w);
        }
    }
    for (; e < e1; ++e) {
        const float x = val[e];
        const float4 w = *reinterpret_cast<const float4*>(Src + (int64_t)idx[e] * ld + off);
        acc.x = fmaf(x, w.x, acc.x); acc.y = fmaf(x, w.y, acc.y);
        acc.z = fmaf(x, w.z, acc.z); acc.w = fmaf(x, w.w, acc.w);
    }
}

__device__ __forceinline__ void gather_mac(float4& acc, const int32_t* __restrict__ idx, const float* __restrict__ val,
                                           int64_t e0, int64_t e1, const float* __restrict__ Src, int64_t ld, int off) {
    for (int64_t b = e0; b < e1; b += SP_SEG) {
        float4 part = make_float4(0.f, 0.f, 0.f, 0.f);
        gather_mac_seq(part, idx, val, b, min(e1, b + SP_SEG), Src, ld, off);
        acc.x += part.x; acc.y += part.y; acc.z += part.z; acc.w += part.w;
    }
}

// ---------------------------------------------------------------------------------------
// Sparse H update (pymf/nmf.py:122-126, pymf/bnmf.py:78-85, pymf/snmf.py:72-90):
//   Hn = ratio(Hc, W^T X, D) and Ht = Hn^T, for k rows [kb0, kb0 + KBLK) and a tile of TCOL columns.
// A group of KBLK / 4 lanes contracts one column over its non-zeros in row order (lane l owns k rows 4 l .. 4 l + 3 and
// gathers them from W with one float4 load).  A column with more than SP_HEAVY non-zeros is split into one contiguous
// chunk per group instead, and the chunks are added in group order through shared memory (a power-law column does not
// hold up its tile).  W^T X is staged in shared memory, so the epilogue reads H and D and writes Hn row by row
// (coalesced), and writes Ht column by column (coalesced).  Dn != nullptr: Semi-NMF, D = G+ H and Dn = G- H.
//   grid.x = column tiles, grid.y = k blocks of KBLK.
// ---------------------------------------------------------------------------------------
template <int KBLK>
__global__ void __launch_bounds__(SP_THREADS)
k_h_update_csc(const DevState* __restrict__ st, const int64_t* __restrict__ colptr, const int32_t* __restrict__ rowidx,
               const float* __restrict__ vals, const float* __restrict__ W, int kp,
               const float* __restrict__ Hc, float* __restrict__ Hn, int64_t ldh, float* __restrict__ Ht,
               const float* __restrict__ D, const float* __restrict__ Dn, float lam, int64_t n_loc) {
    if (st->stop) return;
    constexpr int L = KBLK / 4;                      // lanes per column
    constexpr int NG = SP_THREADS / L;               // column groups per CTA
    constexpr int TCOL = NG * SP_COLS_PER_GROUP;     // columns per CTA tile
    __shared__ float Cs[KBLK][TCOL + 1];
    __shared__ __align__(16) float red[NG][KBLK];
    __shared__ int heavy[TCOL];
    __shared__ int nheavy;
    const int g = threadIdx.x / L, l = threadIdx.x % L;
    const int64_t col0 = (int64_t)blockIdx.x * TCOL;
    const int kb0 = blockIdx.y * KBLK;
    const int off = kb0 + 4 * l;
    if (threadIdx.x == 0) nheavy = 0;
    __syncthreads();
    for (int q = g; q < TCOL; q += NG) {
        const int64_t c = col0 + q;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < n_loc) {
            const int64_t a = colptr[c], b = colptr[c + 1];
            if (b - a > SP_HEAVY) {                  // group-uniform
                if (l == 0) heavy[atomicAdd(&nheavy, 1)] = q;
                continue;
            }
            gather_mac(acc, rowidx, vals, a, b, W, kp, off);
        }
        Cs[4 * l + 0][q] = acc.x; Cs[4 * l + 1][q] = acc.y; Cs[4 * l + 2][q] = acc.z; Cs[4 * l + 3][q] = acc.w;
    }
    __syncthreads();
    const int nh = nheavy;
    for (int h = 0; h < nh; ++h) {                   // the order of the list does not change any column's sum
        const int q = heavy[h];
        const int64_t a = colptr[col0 + q], b = colptr[col0 + q + 1];
        const int64_t per = (b - a + NG - 1) / NG;
        const int64_t e0 = min(b, a + g * per), e1 = min(b, e0 + per);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        gather_mac(acc, rowidx, vals, e0, e1, W, kp, off);
        *reinterpret_cast<float4*>(&red[g][4 * l]) = acc;
        __syncthreads();
        if (threadIdx.x < KBLK) {
            float s = 0.f;
            for (int gg = 0; gg < NG; ++gg) s += red[gg][threadIdx.x];
            Cs[threadIdx.x][q] = s;
        }
        __syncthreads();
    }
    for (int f = threadIdx.x; f < KBLK * TCOL; f += SP_THREADS) {
        const int j = f / TCOL, q = f % TCOL;
        const int64_t c = col0 + q;
        if (c >= n_loc) continue;
        const int64_t o = (int64_t)(kb0 + j) * ldh + c;
        const float h = Hc[o];
        const float v = Dn != nullptr ? snmf_ratio(h, Cs[j][q], D[o], Dn[o]) : mu_ratio(h, Cs[j][q], D[o], lam);
        Hn[o] = v;
        Cs[j][q] = v;
    }
    __syncthreads();
    for (int f = threadIdx.x; f < KBLK * TCOL; f += SP_THREADS) {
        const int q = f / KBLK, j = f % KBLK;
        const int64_t c = col0 + q;
        if (c < n_loc) Ht[c * kp + kb0 + j] = Cs[j][q];
    }
}

// ---------------------------------------------------------------------------------------
// Sparse X H^T, one column panel: A[r, kb0 + 4 l ..] (+)= sum over row r's entries of the panel, in column order, of
// x_rc Ht[c, kb0 + 4 l ..].  The first panel stores, the later ones add what the same thread stored, so A is
// deterministic.  rowptr: this panel's d + 1 offsets.  grid.x = row blocks of SP_THREADS / (KBLK / 4) rows, grid.y = k
// blocks of KBLK.
// ---------------------------------------------------------------------------------------
template <int KBLK>
__global__ void __launch_bounds__(SP_THREADS, 4)
k_xht_csr(const DevState* __restrict__ st, const int64_t* __restrict__ rowptr, const int32_t* __restrict__ ccol,
          const float* __restrict__ cval, const float* __restrict__ Ht, int kp, float* __restrict__ A, int64_t d, int first) {
    if (st->stop) return;
    constexpr int L = KBLK / 4, NG = SP_THREADS / L;
    const int g = threadIdx.x / L, l = threadIdx.x % L;
    const int64_t r = (int64_t)blockIdx.x * NG + g;
    if (r >= d) return;
    const int off = blockIdx.y * KBLK + 4 * l;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    gather_mac(acc, ccol, cval, rowptr[r], rowptr[r + 1], Ht, kp, off);
    float4* out = reinterpret_cast<float4*>(A + r * kp + off);
    if (!first) {
        const float4 o = *out;
        acc.x = o.x + acc.x; acc.y = o.y + acc.y; acc.z = o.z + acc.z; acc.w = o.w + acc.w;
    }
    *out = acc;
}

// x_rc of CSC column c (0 when absent): binary search in the column's sorted rows
__device__ __forceinline__ float csc_at(const int64_t* __restrict__ colptr, const int32_t* __restrict__ rowidx,
                                        const float* __restrict__ vals, int64_t r, int64_t c) {
    int64_t lo = colptr[c], hi = colptr[c + 1];
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int32_t v = rowidx[mid];
        if (v == r) return vals[mid];
        if (v < r) lo = mid + 1; else hi = mid;
    }
    return 0.f;
}

// ---------------------------------------------------------------------------------------
// Direct residual sum (X - W H)^2 as written (pymf/nmf.py:110) for a sparse X: k_resid_simt with x_rc looked up in
// the CSC.  fp32 W H tile, fp64 accumulation of squares, deterministic final sum (partials + ticket).
// ---------------------------------------------------------------------------------------
template <int KB>
__global__ void __launch_bounds__(SIMT_THREADS)
k_resid_csc(DevState* __restrict__ st, const int64_t* __restrict__ colptr, const int32_t* __restrict__ rowidx,
            const float* __restrict__ vals, const float* __restrict__ Wt, int64_t ldwt, const float* __restrict__ H,
            int64_t ldh, int64_t d, int64_t n_loc, int kp, double* __restrict__ partial) {
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
        if (r < d) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (col + j < n_loc) {
                    const float e = csc_at(colptr, rowidx, vals, r, col + j) - acc[i][j];
                    s += (double)e * (double)e;
                }
            }
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
        red[threadIdx.x] = t;
        __syncthreads();
        for (int k = SIMT_THREADS / 2; k > 0; k >>= 1) {
            if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k];
            __syncthreads();
        }
        if (threadIdx.x == 0) { st->resid_local = red[0]; st->resid = red[0]; st->ticket3 = 0; }
    }
}

}  // namespace sp
}  // namespace pymfb
