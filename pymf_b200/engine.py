"""Engine: one libpymfb context (= one GPU, one column shard of X and H).

Thin object wrapper over the C ABI; all arithmetic happens in the CUDA library.  The
reference has no counterpart below the NMF class - this is the layer pymf.NMF's hooks
(update_w / update_h / frobenius_norm, pymf/nmf.py:100-132) are rebuilt on.
"""
import ctypes as C

import numpy as np

from . import _lib


def _dtype_code(a):
    if a.dtype == np.float32:
        return _lib.F32
    if a.dtype == np.float64:
        return _lib.F64
    raise TypeError("expected float32/float64, got %s" % a.dtype)


class _PinnedBlock(object):
    """Owner of one pymfb_host_alloc buffer; numpy arrays made by pinned_empty keep it alive."""

    def __init__(self, nbytes):
        self._lib = _lib.load()
        self.ptr = C.c_void_p()
        _lib.check(self._lib.pymfb_host_alloc(C.byref(self.ptr), int(nbytes)))
        self.nbytes = int(nbytes)

    def __del__(self):
        try:
            if self.ptr is not None and self.ptr.value:
                self._lib.pymfb_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(shape, dtype=np.float32):
    """Uninitialised numpy array in PAGE-LOCKED host memory (pymfb_host_alloc).

    Build ``data`` in such an array (or in ``torch.empty(..., pin_memory=True).numpy()``) and
    ``NMF(data, ...)`` uploads it with direct DMA - no host-side staging copy - instead of the
    pageable path (the ``data[:,:]`` read of pymf/nmf.py:110,125,131 done once, at PCIe speed).
    """
    dtype = np.dtype(dtype)
    shape = (int(shape),) if np.isscalar(shape) else tuple(int(s) for s in shape)
    count = int(np.prod(shape)) if len(shape) else 1
    block = _PinnedBlock(max(1, count * dtype.itemsize))
    buf = (C.c_char * block.nbytes).from_address(block.ptr.value)
    buf._pymfb_block = block                      # the ctypes buffer (numpy's .base) owns the allocation
    return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)


def panel_ranges(d, n, itemsize, panel_bytes=64 << 20):
    """Column panels (first column, width) of a d x n source for the panel-streamed ingest: about panel_bytes each,
    widths a multiple of 128 columns (except the last), at least 128."""
    pw = int(panel_bytes) // (int(d) * int(itemsize))
    pw = n if pw >= n else max(128, pw // 128 * 128)
    pw = max(1, min(pw, n))
    return pw, [(c0, min(pw, n - c0)) for c0 in range(0, n, pw)]


def numa_info(array=None, device=0):
    """(NUMA node of the GPU, NUMA node holding the first page of `array`), -1 where unknown."""
    lib = _lib.load()
    gpu = int(lib.pymfb_device_numa_node(int(device)))
    host = int(lib.pymfb_host_node_of(C.c_void_p(array.ctypes.data))) if array is not None else -1
    return gpu, host


class Engine(object):
    def __init__(self, d, n_local, k, device=0, n_global=None, col0=0, path=None):
        self._lib = _lib.load()
        self.d, self.n_local, self.k = int(d), int(n_local), int(k)
        self.n_global = int(n_local if n_global is None else n_global)
        self.col0 = int(col0)
        self.device = int(device)
        self._ctx = C.c_void_p()
        self._keepalive = None
        _lib.check(self._lib.pymfb_create(C.byref(self._ctx), self.device, self.d, self.n_local,
                                          self.n_global, self.col0, self.k))
        if path is not None:
            self.set_path(path)

    # -- lifetime ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self._lib.pymfb_destroy(self._ctx)
            self._ctx = C.c_void_p()
            self._keepalive = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- options / comm -----------------------------------------------------------------
    def set_path(self, path):
        code = {"auto": _lib.PATH_AUTO, "simt": _lib.PATH_SIMT, "tc": _lib.PATH_TC}.get(path, path)
        _lib.check(self._lib.pymfb_set_option(self._ctx, _lib.OPT_PATH, int(code)))

    def set_nndsvd_path(self, path):
        """'auto' | 'simt' | 'tc': pass family of nndsvd()."""
        code = {"auto": _lib.PATH_AUTO, "simt": _lib.PATH_SIMT, "tc": _lib.PATH_TC}.get(path, path)
        _lib.check(self._lib.pymfb_set_option(self._ctx, _lib.OPT_NNDSVD_PATH, int(code)))

    def set_err_mode(self, mode):
        """'auto' | 'trace' (trace identity, no extra pass) | 'direct' (||X - WH|| as written)."""
        code = {"auto": _lib.ERR_AUTO, "trace": _lib.ERR_TRACE, "direct": _lib.ERR_DIRECT}.get(mode, mode)
        _lib.check(self._lib.pymfb_set_option(self._ctx, _lib.OPT_ERR_MODE, int(code)))

    def set_graph_mode(self, mode):
        """'auto' (small problems) | 'off' | 'on': CUDA-graph replay of the iteration body."""
        code = {"auto": _lib.GRAPH_AUTO, "off": _lib.GRAPH_OFF, "on": _lib.GRAPH_ON}.get(mode, mode)
        _lib.check(self._lib.pymfb_set_option(self._ctx, _lib.OPT_GRAPH, int(code)))

    @property
    def graph_replays(self):
        return int(self._lib.pymfb_graph_replays(self._ctx))

    def set_variant(self, variant):
        """'nmf' | 'snmf': which update rules the loop applies (pymf/nmf.py:122-132 / pymf/snmf.py:67-90)."""
        code = {"nmf": _lib.VARIANT_NMF, "snmf": _lib.VARIANT_SNMF}.get(variant, variant)
        _lib.check(self._lib.pymfb_set_variant(self._ctx, int(code)))

    def set_penalty(self, lamb_w, lamb_h, increase_w=1.0, increase_h=1.0):
        """BNMF penalty weights of the next iteration and their growth per H update (pymf/bnmf.py:70-90)."""
        _lib.check(self._lib.pymfb_set_penalty(self._ctx, float(lamb_w), float(lamb_h),
                                               float(increase_w), float(increase_h)))

    def get_penalty(self):
        lw, lh = C.c_double(0.0), C.c_double(0.0)
        _lib.check(self._lib.pymfb_get_penalty(self._ctx, C.byref(lw), C.byref(lh)))
        return lw.value, lh.value

    @property
    def active_path(self):
        return {_lib.PATH_SIMT: "simt", _lib.PATH_TC: "tc",
                _lib.PATH_SPARSE: "sparse"}.get(self._lib.pymfb_active_path(self._ctx), "?")

    @staticmethod
    def comm_unique_id():
        buf = C.create_string_buffer(128)
        _lib.check(_lib.load().pymfb_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, uid, world, rank):
        buf = C.create_string_buffer(bytes(uid), 128)
        _lib.check(self._lib.pymfb_comm_init(self._ctx, buf, int(world), int(rank)))

    @staticmethod
    def comm_create(uid, world, rank, device):
        """A communicator that outlives engines (pymfb_comm_create); attach it with comm_attach."""
        buf = C.create_string_buffer(bytes(uid), 128)
        comm = C.c_void_p()
        _lib.check(_lib.load().pymfb_comm_create(C.byref(comm), int(device), buf, int(world), int(rank)))
        return comm

    def comm_attach(self, comm, world, rank):
        self._comm_keepalive = comm
        _lib.check(self._lib.pymfb_comm_attach(self._ctx, comm, int(world), int(rank)))

    # -- data -----------------------------------------------------------------------------
    def upload_x(self, x):
        """x: host array (d x n_local), float32 or float64, last axis contiguous."""
        x = np.asarray(x)
        if x.shape != (self.d, self.n_local):
            raise ValueError("data shape %r != (%d, %d)" % (x.shape, self.d, self.n_local))
        if x.dtype not in (np.float32, np.float64):
            x = x.astype(np.float64)
        if x.strides[1] != x.itemsize or x.strides[0] % x.itemsize or x.strides[0] < x.shape[1] * x.itemsize:
            x = np.ascontiguousarray(x)
        ld = x.strides[0] // x.itemsize
        _lib.check(self._lib.pymfb_upload_x(self._ctx, x.ctypes.data_as(C.c_void_p), _dtype_code(x), ld))

    def upload_x_panels(self, source, panel_bytes=64 << 20):
        """Assemble the device copy of X from column panels ``source[:, c0:c1]`` of an h5py-like object (anything
        with ``.shape`` and 2-D slicing that is not a host array).  Two page-locked panel buffers alternate: one is
        being filled from the source while the copy engine reads the other, so the host never holds more than two
        panels (plus whatever temporary the source's own ``__getitem__`` returns).  Returns the panel width."""
        d, n = self.d, self.n_local
        if tuple(source.shape) != (d, n):
            raise ValueError("data shape %r != (%d, %d)" % (tuple(source.shape), d, n))
        dt = np.dtype(getattr(source, "dtype", np.float64))
        dt = np.dtype(np.float32) if dt == np.float32 else np.dtype(np.float64)
        pw, ranges = panel_ranges(d, n, dt.itemsize, panel_bytes)
        bufs = [pinned_empty((d, pw), dt), pinned_empty((d, pw), dt)]
        _lib.check(self._lib.pymfb_upload_x_begin(self._ctx))
        for i, (c0, w) in enumerate(ranges):
            slot = i & 1
            _lib.check(self._lib.pymfb_upload_x_wait(self._ctx, slot))          # the DMA that last read this buffer
            view = bufs[slot][:, :w]
            if w == pw and hasattr(source, "read_direct"):                      # h5py: straight into the pinned buffer
                source.read_direct(bufs[slot], np.s_[:, c0:c0 + w])
            else:
                view[...] = source[:, c0:c0 + w]
            _lib.check(self._lib.pymfb_upload_x_panel(self._ctx, view.ctypes.data_as(C.c_void_p), _dtype_code(view), pw, c0, w, slot))
        _lib.check(self._lib.pymfb_upload_x_end(self._ctx))
        return pw

    def upload_x_csc(self, indptr, indices, values):
        """Sparse X (d x n_local) in compressed sparse column form: indptr (n_local + 1, int64), indices (row of each
        non-zero, int32, strictly increasing within a column), values (float32 / float64).  The library checks the
        arrays before it uses them and raises PymfbError on a malformed matrix.  The context then runs the sparse
        passes (active_path "sparse") until a dense X is uploaded."""
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        indices = np.ascontiguousarray(indices, dtype=np.int32)
        values = np.ascontiguousarray(values)
        if values.dtype not in (np.float32, np.float64):
            values = values.astype(np.float64)
        if indptr.shape != (self.n_local + 1,):
            raise ValueError("indptr shape %r != (%d,)" % (indptr.shape, self.n_local + 1))
        if indices.ndim != 1 or values.shape != indices.shape:
            raise ValueError("indices %r and values %r must be 1-D of the same length" % (indices.shape, values.shape))
        _lib.check(self._lib.pymfb_upload_x_csc(self._ctx, indptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                                indices.ctypes.data_as(C.POINTER(C.c_int32)),
                                                values.ctypes.data_as(C.c_void_p), _dtype_code(values), int(indices.size)))

    def upload_x_sparse_device(self, layout, a, b, values):
        """Sparse X (d x n_local) from 1-D torch tensors, canonicalised by the library on the device (entries sorted,
        duplicates summed; the form is documented at pymfb_upload_x_sparse_device): layout "coo" (a = row ids,
        b = column ids), "csr" (a = d + 1 row pointers, b = column ids) or "csc" (a = n_local + 1 column pointers,
        b = row ids).  a and b int32 or int64 alike, values float32 / float64.  CPU tensors are copied to this
        engine's device (the library refuses memory of another device); torch's current stream there is
        synchronised before the library reads the arrays, and they are only read during the call."""
        import torch                                         # already imported: the arguments are torch tensors
        code = {"coo": _lib.LAYOUT_COO, "csr": _lib.LAYOUT_CSR, "csc": _lib.LAYOUT_CSC}[layout]
        dev = torch.device("cuda", self.device)
        a, b, values = ((t.to(dev) if not t.is_cuda else t).contiguous() for t in (a, b, values))
        torch.cuda.current_stream(dev).synchronize()
        nnz = int(b.numel())
        na = {"coo": nnz, "csr": self.d + 1, "csc": self.n_local + 1}[layout]
        for t, want, what in ((a, na, "a"), (b, nnz, "b"), (values, nnz, "values")):
            if t.dim() != 1 or t.numel() != want or (want > 1 and t.stride(0) != 1):
                raise ValueError("%s: expected a contiguous 1-D tensor of %d entries, got shape %r"
                                 % (what, want, tuple(t.shape)))
        index = {"torch.int32": _lib.I32, "torch.int64": _lib.I64}
        if str(a.dtype) not in index or b.dtype != a.dtype:
            raise TypeError("index tensors must both be int32 or both int64, got %s / %s" % (a.dtype, b.dtype))
        vcode = {"torch.float32": _lib.F32, "torch.float64": _lib.F64}.get(str(values.dtype))
        if vcode is None:
            raise TypeError("values must be float32 or float64, got %s" % values.dtype)
        _lib.check(self._lib.pymfb_upload_x_sparse_device(self._ctx, code, C.c_void_p(a.data_ptr()),
                                                          C.c_void_p(b.data_ptr()), index[str(a.dtype)],
                                                          C.c_void_p(values.data_ptr()), vcode, nnz))

    @property
    def last_upload_pinned(self):
        """True if the last upload_x read page-locked memory by direct DMA."""
        return bool(self._lib.pymfb_last_upload_pinned(self._ctx))

    def bind_x_device(self, ptr, ld, keepalive=None):
        """Borrow a device pointer (fp32 row-major d x n_local, leading dimension ld)."""
        self._keepalive = keepalive
        _lib.check(self._lib.pymfb_bind_x(self._ctx, C.c_void_p(int(ptr)), int(ld)))

    def gen_x(self, seed):
        _lib.check(self._lib.pymfb_gen_x(self._ctx, int(seed)))

    def gen_w(self, seed):
        _lib.check(self._lib.pymfb_gen_w(self._ctx, int(seed)))

    def gen_h(self, seed):
        _lib.check(self._lib.pymfb_gen_h(self._ctx, int(seed)))

    def _host_in(self, a, shape, what):
        a = np.ascontiguousarray(a)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if a.shape != shape:
            raise ValueError("%s shape %r != %r" % (what, a.shape, shape))
        return a

    def set_w(self, w):
        w = self._host_in(w, (self.d, self.k), "W")
        _lib.check(self._lib.pymfb_set_w(self._ctx, w.ctypes.data_as(C.c_void_p), _dtype_code(w)))

    def set_h(self, h):
        h = self._host_in(h, (self.k, self.n_local), "H")
        _lib.check(self._lib.pymfb_set_h(self._ctx, h.ctypes.data_as(C.c_void_p), _dtype_code(h)))

    @staticmethod
    def _host_out(out, shape, dtype):
        """Use `out` as the download target when it is a dense float32/float64 array of the right shape."""
        if (isinstance(out, np.ndarray) and out.shape == shape and out.dtype in (np.float32, np.float64)
                and out.flags.c_contiguous and out.flags.writeable):
            return out
        return np.empty(shape, dtype=dtype)

    def get_w(self, dtype=np.float64, out=None):
        """Current W as a host array; written straight into `out` when it is dense f32/f64 (no extra copy)."""
        out = self._host_out(out, (self.d, self.k), dtype)
        _lib.check(self._lib.pymfb_get_w(self._ctx, out.ctypes.data_as(C.c_void_p), _dtype_code(out)))
        return out

    def get_h(self, dtype=np.float64, out=None):
        out = self._host_out(out, (self.k, self.n_local), dtype)
        _lib.check(self._lib.pymfb_get_h(self._ctx, out.ctypes.data_as(C.c_void_p), _dtype_code(out)))
        return out

    # -- the loop ---------------------------------------------------------------------------
    def run(self, niter, compute_w=True, compute_h=True, compute_err=True, early_stop=True):
        """niter iterations of W-update, H-update, error.  Returns (ferr array, iterations done)."""
        flags = ((_lib.COMPUTE_W if compute_w else 0) | (_lib.COMPUTE_H if compute_h else 0) |
                 (_lib.COMPUTE_ERR if compute_err else 0) | (_lib.EARLY_STOP if early_stop else 0))
        ferr = np.zeros(max(int(niter), 1), dtype=np.float64)
        done, nf = C.c_int(0), C.c_int(0)
        _lib.check(self._lib.pymfb_run(self._ctx, int(niter), flags,
                                       ferr.ctypes.data_as(C.POINTER(C.c_double)),
                                       C.byref(done), C.byref(nf)))
        return ferr[:nf.value].copy(), done.value

    def nndsvd(self, max_iter=0, tol=0.0, extra_iter=-1):
        """Set the device W / H to the NNDSVD start (pymf/nndsvd.py:79-108).  Returns (singular values, sweeps)."""
        sig = np.zeros(self.k, dtype=np.float64)
        it = C.c_int(0)
        _lib.check(self._lib.pymfb_nndsvd(self._ctx, int(max_iter), float(tol), int(extra_iter), C.byref(it),
                                          sig.ctypes.data_as(C.POINTER(C.c_double))))
        path, change = C.c_int(0), C.c_double(0.0)
        _lib.check(self._lib.pymfb_nndsvd_info(self._ctx, C.byref(path), C.byref(change)))
        self.nndsvd_path = {_lib.PATH_SIMT: "simt", _lib.PATH_TC: "tc"}.get(path.value, "?")   # pass family it ran
        self.nndsvd_change = change.value         # relative change of the Ritz values in its last sweep
        return sig, it.value

    def frobenius(self):
        out = C.c_double(0.0)
        _lib.check(self._lib.pymfb_frobenius(self._ctx, C.byref(out)))
        return out.value

    # -- benchmarking helpers -----------------------------------------------------------------
    def enqueue(self, niter, compute_w=True, compute_h=True, compute_err=True):
        flags = ((_lib.COMPUTE_W if compute_w else 0) | (_lib.COMPUTE_H if compute_h else 0) |
                 (_lib.COMPUTE_ERR if compute_err else 0))
        _lib.check(self._lib.pymfb_enqueue(self._ctx, int(niter), flags))

    def sync(self):
        _lib.check(self._lib.pymfb_sync(self._ctx))

    def flush_l2(self):
        _lib.check(self._lib.pymfb_flush_l2(self._ctx))

    def event(self):
        ev = C.c_void_p()
        _lib.check(self._lib.pymfb_event_create(C.byref(ev)))
        return ev

    def record(self, ev):
        _lib.check(self._lib.pymfb_event_record(self._ctx, ev))

    def elapsed_ms(self, ev0, ev1):
        ms = C.c_float(0.0)
        _lib.check(self._lib.pymfb_event_elapsed_ms(ev0, ev1, C.byref(ms)))
        return ms.value

    def kernel_timing(self, enable):
        _lib.check(self._lib.pymfb_kernel_timing(self._ctx, 1 if enable else 0))

    def kernel_timing_read(self, which):
        avg, cnt = C.c_double(0.0), C.c_int64(0)
        _lib.check(self._lib.pymfb_kernel_timing_read(self._ctx, int(which), C.byref(avg), C.byref(cnt)))
        return avg.value, cnt.value

    @property
    def launch_count(self):
        return int(self._lib.pymfb_launch_count(self._ctx))
