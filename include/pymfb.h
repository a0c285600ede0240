/*
 * pymfb.h - C ABI of libpymfb.so: the B200-native NMF multiplicative-update engine.
 *
 * The reference (nils-werner/pymf) has no FFI / plugin registry: its boundary for this
 * path is the Python class pymf.NMF (pymf/nmf.py:23-202).  This header is the thin
 * C layer a binding for that class sits on; `pymf_b200/nmf.py` is that binding
 * (ctypes).  Each entry point names the reference code it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no exceptions cross the ABI.
 *   - every function returns 0 on success, non-zero on failure;
 *     pymfb_last_error() returns a thread-local message for the last failure.
 *   - one context per GPU, one CUDA stream per context, a context is not re-entrant.
 *   - matrices are row-major.  X is d x n_local (features x samples, pymf/nmf.py:34),
 *     W is d x k (:42), H is k x n_local (:43).  With more than one rank, X and H are
 *     block-sharded by COLUMNS; W is replicated.
 *   - dtype codes: PYMFB_F32 = 0, PYMFB_F64 = 1.  The device computes in fp32 storage
 *     (3xTF32 tensor-core products with fp32 accumulation, fp64 scalar combines).
 */
#ifndef PYMFB_H
#define PYMFB_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pymfb_ctx pymfb_ctx;

#define PYMFB_F32 0
#define PYMFB_F64 1

/* pymfb_run flags == keyword arguments of NMF.factorize (pymf/nmf.py:141-142) */
#define PYMFB_COMPUTE_W   1u   /* compute_w   (:183-184) */
#define PYMFB_COMPUTE_H   2u   /* compute_h   (:186-187) */
#define PYMFB_COMPUTE_ERR 4u   /* compute_err (:189-190) */
#define PYMFB_EARLY_STOP  8u   /* the `i > 1 and converged(i)` break (:198-202) */

/* kernel-path selection (pymfb_set_option PYMFB_OPT_PATH) */
#define PYMFB_PATH_AUTO 0      /* tcgen05 kernels when the shape allows, else SIMT */
#define PYMFB_PATH_SIMT 1      /* fp32 CUDA-core kernels (exact fp32 FMA) */
#define PYMFB_PATH_TC   2      /* tcgen05 3xTF32 kernels; error if the shape is unsupported */
#define PYMFB_PATH_SPARSE 3    /* reported only: the sparse passes of a context holding a CSC X (pymfb_upload_x_csc);
                                  setting PYMFB_PATH_SIMT / _TC on such a context is an error */

#define PYMFB_OPT_PATH 1

/* how frobenius_norm is evaluated (pymfb_set_option PYMFB_OPT_ERR_MODE) */
#define PYMFB_ERR_AUTO   0     /* direct for small problems (d*n*k <= 2^28), trace identity otherwise */
#define PYMFB_ERR_TRACE  1     /* sqrt(||X||^2 - 2<W, X H^T> + <W^T W, H H^T>): no extra pass over X */
#define PYMFB_ERR_DIRECT 2     /* sqrt(sum((X - W H)^2)) as written in pymf/nmf.py:110: one more pass */
#define PYMFB_OPT_ERR_MODE 2

/* CUDA-graph replay of the iteration body (pymfb_set_option PYMFB_OPT_GRAPH).  Launch-bound
 * problems (X up to 16 Mi elements, single rank, plain NMF) replay two iterations - one ping-pong
 * period of the W / H buffers - as one cudaGraphLaunch; results are those of the plain launches. */
#define PYMFB_GRAPH_AUTO 0     /* small problems only */
#define PYMFB_GRAPH_OFF  1
#define PYMFB_GRAPH_ON   2     /* whenever the loop is replayable (any size) */
#define PYMFB_OPT_GRAPH 3

/* pass family of pymfb_nndsvd (pymfb_set_option PYMFB_OPT_NNDSVD_PATH, value PYMFB_PATH_*): it has its own, since its
 * block width (not k) decides what the tensor-core kernels take */
#define PYMFB_OPT_NNDSVD_PATH 4

/* Library / ABI version (major*1000 + minor). */
int pymfb_version(void);

/* Message of the last failing call on this thread ("" if none). */
const char* pymfb_last_error(void);

/* Number of visible CUDA devices (0 when there is no driver / GPU); never fails. */
int pymfb_device_count(void);

/*
 * Create an engine for a d x n_local shard of a d x n_global problem with k bases.
 * Replaces NMF.__init__ (pymf/nmf.py:71-97).  col0 = global index of the shard's first
 * column (only used by the synthetic generator).  Allocates W, H, the packed
 * [X H^T | H H^T] reduction buffers and scratch on `device`.
 */
int pymfb_create(pymfb_ctx** out, int device, int64_t d, int64_t n_local, int64_t n_global,
                 int64_t col0, int k);
int pymfb_destroy(pymfb_ctx* ctx);

int pymfb_set_option(pymfb_ctx* ctx, int option, int64_t value);

/*
 * BNMF penalty - the binary-factor variant of the same loop (pymf/bnmf.py:22-123, a subclass
 * that overrides update_w / update_h only).  With lamb > 0 the update kernels' ratio epilogue
 * becomes   H <- H * (W^T X + 3 lamb_h H^2) / (G H + 2 lamb_h H^3 + lamb_h H + 1e-9)   (:79-82)
 *           W <- W * (X H^T + 3 lamb_w W^2) / (W B + 2 lamb_w W^3 + lamb_w W + 1e-9)   (:87-90)
 * and after every H update lamb_w *= increase_w, lamb_h *= increase_h (:84-85; BNMF.factorize
 * starts both at 1/niter, :117-118, with _LAMB_INCREASE_W/H = 1.1, :75-76).  lamb = 0 (the
 * default) is plain NMF (the same arithmetic as not calling this).  get_penalty returns the current
 * weights (the reference's _lamb_W / _lamb_H after factorize).
 */
int pymfb_set_penalty(pymfb_ctx* ctx, double lamb_w, double lamb_h, double increase_w, double increase_h);
int pymfb_get_penalty(pymfb_ctx* ctx, double* lamb_w, double* lamb_h);

/*
 * Semi-NMF - another override of the same two hooks (pymf/snmf.py:22-90): X and W may be signed,
 * H stays non-negative.  With PYMFB_VARIANT_SNMF the loop's steps become
 *   W <- (X H^T) (H H^T)^-1                                                         (:67-70)
 *   H <- H * sqrt(((W^T X)+ + G- H) / ((W^T X)- + G+ H + 1e-9)),  G = W^T W,
 *        m+ = (|m| + m)/2, m- = (|m| - m)/2                                         (:72-90)
 * on the same passes: the X H^T / H H^T reductions feed a fp64 k x k inverse (k <= 512, one CTA), the
 * H-update pass keeps its W^T X contraction and switches its epilogue.  Error, early stop, flags
 * and sharding are those of NMF.
 */
#define PYMFB_VARIANT_NMF  0
#define PYMFB_VARIANT_SNMF 1
int pymfb_set_variant(pymfb_ctx* ctx, int variant);

/*
 * Multi-GPU (one process per GPU).  Rank 0 calls pymfb_comm_unique_id (128 bytes, an
 * ncclUniqueId), the host layer broadcasts it, every rank calls pymfb_comm_init.
 * After that pymfb_prepare / pymfb_run sum the packed [X H^T | H H^T] partials (and
 * ||X||^2) over ranks with one NCCL all-reduce per iteration on the context's stream.
 * No counterpart in the reference (it is single-process).
 */
int pymfb_comm_unique_id(void* out128);
int pymfb_comm_init(pymfb_ctx* ctx, const void* uid128, int world, int rank);

/*
 * Shared communicator: creating an NCCL communicator and running its first collective costs
 * 1-2 s (measured: a fresh NMF object per call paid 1.4 s + 0.7 s at 2 GPUs).  A host layer that
 * builds several contexts over the same ranks creates the communicator ONCE (comm_create, same
 * uid hand-shake as comm_init), attaches it to every context (comm_attach: the context borrows
 * it; contexts sharing one communicator must not run concurrently) and destroys it at exit.
 */
int pymfb_comm_create(void** comm_out, int device, const void* uid128, int world, int rank);
int pymfb_comm_attach(pymfb_ctx* ctx, void* comm, int world, int rank);
int pymfb_comm_destroy(void* comm);

/*
 * Data residency - replaces `self.data = data` (pymf/nmf.py:93) and the `data[:,:]`
 * full reads (:110,125,131).
 *   bind_x    borrow a device pointer (fp32, row-major, leading dimension ld elements,
 *             ld % 4 == 0, 16-byte aligned); the caller keeps it alive.
 *   upload_x  copy a host matrix (fp32 or fp64, leading dimension ld elements) into a
 *             context-owned fp32 device copy through a pinned, double-buffered staging ring.
 *   gen_x     fill the context-owned X with the synthetic U[0,1) generator
 *             (element (r, c) = hash(seed, r*n_global + col0 + c), see oracle/nmf_oracle.py).
 */
int pymfb_bind_x(pymfb_ctx* ctx, const float* x_dev, int64_t ld);
int pymfb_upload_x(pymfb_ctx* ctx, const void* x_host, int dtype, int64_t ld);
int pymfb_gen_x(pymfb_ctx* ctx, uint64_t seed);

/*
 * Sparse X in compressed sparse column form: colptr (n_local + 1 entries), rowidx and values (nnz entries each, values
 * fp32 or fp64 by dtype, cast to fp32 on the device).  The arrays are validated on the device before any kernel indexes
 * with them - colptr[0] == 0, colptr non-decreasing, colptr[n_local] == nnz, 0 <= row < d, rows strictly increasing
 * within a column - and a malformed matrix returns non-zero with the broken rules in pymfb_last_error().
 * On success the sparse X becomes current: the dense X and the tensor-core plan are freed, pymfb_active_path reports
 * PYMFB_PATH_SPARSE, and the loop (pymfb_run, pymfb_frobenius, pymfb_enqueue) runs the sparse passes: the H update over
 * the CSC, X H^T over a column-panel CSR built on the device.  A later pymfb_upload_x / pymfb_bind_x / pymfb_gen_x
 * switches back to dense data.  pymfb_nndsvd on a sparse context is an error.  nnz < 2^31.
 * PYMFB_SPARSE_PANEL=<columns> (environment, read at each upload) forces the CSR panel width.
 */
int pymfb_upload_x_csc(pymfb_ctx* ctx, const int64_t* colptr /* n_local+1 */, const int32_t* rowidx,
                       const void* values, int dtype, int64_t nnz);

/*
 * Sparse X already on the device, in any order and with duplicates; the library makes the CSC of pymfb_upload_x_csc
 * from it on the device.
 *   layout  PYMFB_LAYOUT_COO: a = row ids, b = column ids (nnz each)
 *           PYMFB_LAYOUT_CSR: a = d + 1 row pointers, b = column ids (nnz)
 *           PYMFB_LAYOUT_CSC: a = n_local + 1 column pointers, b = row ids (nnz)
 *   index_dtype PYMFB_I32 / PYMFB_I64 (a and b alike), values nnz entries of dtype PYMFB_F32 / PYMFB_F64.
 * Every array must be device memory of the context's device (checked with cudaPointerGetAttributes).  The arrays are
 * checked on the device before any kernel indexes with them - pointers[0] == 0, pointers non-decreasing,
 * pointers[last] == nnz, 0 <= row < d, 0 <= column < n_local - and a malformed input returns non-zero with the broken
 * rules in pymfb_last_error(); the context then keeps its previous X.  The canonical form:
 *   entries sorted by (column, row) with a stable radix sort; the entries of one (row, column) summed in fp64 in
 *   input order and rounded once to fp32 (explicit zeros are kept, as scipy's sum_duplicates keeps them); int32
 *   rows strictly increasing within a column, int64 column pointers, fp32 values zero-padded to a multiple of 4.
 * The same input gives the same arrays on every call.  From there on the call is pymfb_upload_x_csc's (validation,
 * CSR build, the sparse X becomes current).  It returns after the arrays have been read: the caller may free them
 * afterwards.  Temporaries: about 24 bytes per input entry plus the CUB sort scratch, freed before returning.
 * nnz < 2^31.
 */
#define PYMFB_LAYOUT_COO 0
#define PYMFB_LAYOUT_CSR 1
#define PYMFB_LAYOUT_CSC 2
#define PYMFB_I32 2
#define PYMFB_I64 3
int pymfb_upload_x_sparse_device(pymfb_ctx* ctx, int layout, const void* a, const void* b, int index_dtype,
                                 const void* values, int dtype, int64_t nnz);

/*
 * Ingest fast path (SURVEY 8f rank 2, the step before the hot path).  pymfb_upload_x looks at
 * its source pointer: PAGE-LOCKED host memory (pymfb_host_alloc, cudaHostAlloc/Register, torch
 * pin_memory) is read by the copy engines directly - fp32 in one strided DMA into X, fp64 in
 * row chunks through a device staging pair with the fp64->fp32 cast overlapped - with no
 * host-side copy; pageable memory goes through the pinned staging ring filled by host threads.
 * pymfb_last_upload_pinned tells which one the last upload took (1 = direct DMA).
 * pymfb_host_alloc / pymfb_host_free hand out page-locked buffers for callers that build X in
 * place (numpy arrays are wrapped around them by pymf_b200.pinned_empty).
 */
int pymfb_host_alloc(void** out, size_t bytes);
/*
 * Panel-streamed ingest - replaces the `data[:,:]` convention of pymf/nmf.py:110,125,131 (which exists so that
 * `data` may be an h5py dataset, pymf/kmeans.py:71) for sources that are NOT host arrays: the host layer reads
 * column panels data[:, c0:c1] into two page-locked panel buffers and hands each to upload_x_panel, so the host
 * never holds more than two panels of X while the device copy is assembled.
 *   upload_x_begin   make the context-owned X current (padding zeroed)
 *   upload_x_panel   columns [col0, col0 + ncols) <- host panel (d x ncols, fp32 / fp64, leading dimension ld);
 *                    asynchronous for page-locked panels: `slot` (0 / 1) names the panel buffer, and
 *   upload_x_wait    blocks until the DMA that last read `slot` has finished (call before refilling the buffer)
 *   upload_x_end     waits for everything and re-plans the kernels for the new data
 */
int pymfb_upload_x_begin(pymfb_ctx* ctx);
int pymfb_upload_x_panel(pymfb_ctx* ctx, const void* panel_host, int dtype, int64_t ld, int64_t col0, int64_t ncols, int slot);
int pymfb_upload_x_wait(pymfb_ctx* ctx, int slot);
int pymfb_upload_x_end(pymfb_ctx* ctx);
int pymfb_host_free(void* ptr);
int pymfb_last_upload_pinned(pymfb_ctx* ctx);
/* pymfb_host_alloc places the buffer on the NUMA node of the CURRENT device when the OS exposes one (mmap +
 * mbind + cudaHostRegister; plain cudaHostAlloc otherwise, or with PYMFB_NO_NUMA set).
 * device_numa_node: node of a device (-1 unknown); host_node_of: node that holds an address. */
int pymfb_device_numa_node(int device);
int pymfb_host_node_of(const void* ptr);

/*
 * Factor access - the .W / .H attributes (pymf/nmf.py:42-43,116-120,173-177).
 * Host pointers are dense row-major d x k / k x n_local of the given dtype.
 * gen_w / gen_h fill from the synthetic generator (W: element (r,c)=hash(seed, r*k+c);
 * H: hash(seed, r*n_global + col0 + c)).
 */
int pymfb_set_w(pymfb_ctx* ctx, const void* w_host, int dtype);
int pymfb_set_h(pymfb_ctx* ctx, const void* h_host, int dtype);
int pymfb_get_w(pymfb_ctx* ctx, void* w_host, int dtype);
int pymfb_get_h(pymfb_ctx* ctx, void* h_host, int dtype);
int pymfb_gen_w(pymfb_ctx* ctx, uint64_t seed);
int pymfb_gen_h(pymfb_ctx* ctx, uint64_t seed);

/*
 * NNDSVD initialisation - replaces NNDSVD.update_w (pymf/nndsvd.py:79-108): W and H of the context are set to the
 * non-negative double SVD start of Boutsidis & Gallopoulos, ready for pymfb_run (warm start) or pymfb_get_w/h.
 * The leading k singular triplets of X come from subspace iteration (its two products per sweep are the
 * contractions of the H-update and X H^T passes); the reference's second SVD of max(0, s_i u_i v_i^T) is taken
 * in closed form.  max_iter <= 0 / tol <= 0 / extra_iter < 0 select the defaults (100 sweeps at most, Ritz values
 * settled to 3e-7 relative, then 6 more sweeps).  sigma_out (k doubles, may be null) receives the singular
 * values.  k <= 200.
 * Column-sharded contexts (world > 1, collective: every rank calls it): X and H are this rank's columns, everything of
 * length d is replicated.  The fp64 Gram matrix of Q^T X, X Z^T and the column norms of the second SVD are summed over
 * the ranks on the context's stream; W, sigma_out and iters_done come out bit-identical on every rank, H holds the
 * rank's columns of the unsharded result.
 * Pass family: the tensor-core passes (3xTF32) when the shard allows them and d * n_local > 2^24 (>= 2^32 on one GPU
 * when k > 102, where their block is wider), else the fp32 CUDA-core passes; PYMFB_OPT_NNDSVD_PATH forces either (PYMFB_PATH_TC fails on an unsupported shape).
 */
int pymfb_nndsvd(pymfb_ctx* ctx, int max_iter, double tol, int extra_iter, int* iters_done, double* sigma_out);
/* The last pymfb_nndsvd of this context: its pass family (PYMFB_PATH_SIMT / PYMFB_PATH_TC, 0 before the first call)
 * and the relative change of the leading k Ritz values in its last sweep. */
int pymfb_nndsvd_info(pymfb_ctx* ctx, int* path, double* change);

/*
 * Run `niter` iterations of the factorize() loop (pymf/nmf.py:182-202): per iteration
 * update_w (:128-132), then update_h (:122-126), then frobenius_norm (:100-114) and
 * converged (:134-139), selected by `flags`.  ferr_host (niter doubles, may be NULL
 * unless PYMFB_COMPUTE_ERR) receives the per-iteration errors; *n_iter_done the
 * number of iterations executed and *n_ferr the number of valid ferr entries
 * (n_iter_done - 1 after an early stop, because the reference drops entry i, :201).
 * One host synchronisation at the end; the stop decision is taken on the device.
 */
int pymfb_run(pymfb_ctx* ctx, int niter, unsigned flags, double* ferr_host,
              int* n_iter_done, int* n_ferr);

/* ||X - W H||_F for the current factors (pymf/nmf.py:100-114), trace identity, fp64 combine. */
int pymfb_frobenius(pymfb_ctx* ctx, double* out);

/* Enqueue-only variant for benchmarking: enqueue niter iterations on the context's
 * stream without synchronising (no early stop read-back).  pymfb_sync waits. */
int pymfb_enqueue(pymfb_ctx* ctx, int niter, unsigned flags);
int pymfb_sync(pymfb_ctx* ctx);

/* The context's CUDA stream (cudaStream_t) so callers can record events on it. */
void* pymfb_stream(pymfb_ctx* ctx);

/* Timing helpers on the context's stream (CUDA events): returns elapsed ms. */
int pymfb_event_create(void** ev);
int pymfb_event_record(pymfb_ctx* ctx, void* ev);
int pymfb_event_elapsed_ms(void* ev_start, void* ev_stop, float* ms);
int pymfb_event_destroy(void* ev);

/* Average device time (ms) of the dominant streaming kernel(s) over the launches since
 * the last pymfb_kernel_timing_reset, measured with CUDA events on the launch stream
 * when timing is enabled (enable = 1).  which: 0 = H-update pass, 1 = X H^T pass. */
int pymfb_kernel_timing(pymfb_ctx* ctx, int enable);
int pymfb_kernel_timing_read(pymfb_ctx* ctx, int which, double* avg_ms, int64_t* launches);

/* Kernel launches issued by this context so far (all kernels of this library). */
int64_t pymfb_launch_count(pymfb_ctx* ctx);

/* Graph launches issued so far (each replays two iterations; their kernels are included in
 * pymfb_launch_count). */
int64_t pymfb_graph_replays(pymfb_ctx* ctx);

/* Which path the context resolved to for its data: PYMFB_PATH_SIMT, PYMFB_PATH_TC or PYMFB_PATH_SPARSE. */
int pymfb_active_path(pymfb_ctx* ctx);

/* Write a buffer larger than L2 (flush between timed iterations of small problems). */
int pymfb_flush_l2(pymfb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* PYMFB_H */
