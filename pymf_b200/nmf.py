"""pymf.NMF on B200: host-side mirror of the reference class (pymf/nmf.py:23-202).

Same constructor, ``factorize`` signature, hooks and attributes as the reference, so code
written against ``pymf.NMF`` runs unchanged; the arithmetic of ``update_w`` (:128-132),
``update_h`` (:122-126), ``frobenius_norm`` (:100-114) and the ``converged`` early stop
(:134-139,198-202) runs in libpymfb's sm_100a kernels (see ``engine.py`` / ``include/pymfb.h``).
There is no CPU path: without the built library or without a B200 every compute call raises.

Differences that are deliberate and documented in DESIGN.md:
  * device arithmetic is fp32 storage / 3xTF32 or fp32 FMA products / fp64 scalar combines;
    ``.W`` / ``.H`` come back in the dtype of the host arrays (float64 by default);
  * X is copied to the GPU on first use and cached (the reference re-reads ``data[:,:]`` on
    every call); assign ``mdl.data = ...`` to replace it;
  * sparse ``data`` is rejected by ``factorize`` (the reference only ever returned the
    ``-123456`` sentinel for it, :109-112) unless the object is built with ``sparse=True``: then
    ``data`` is a scipy.sparse matrix or a torch sparse tensor and every call runs the sparse passes of the library.
"""
import logging
import sys
import time

import numpy as np

from .engine import Engine

__all__ = ["NMF"]

_SENTINEL = -123456      # pymf/nmf.py:112


def _is_sparse(a):
    # A scipy sparse matrix can only exist if scipy.sparse is already imported; never import it here
    # (the first import costs ~0.15 s, which used to land inside the first factorize()).
    sp = sys.modules.get("scipy.sparse")
    try:
        return sp is not None and bool(sp.issparse(a))
    except Exception:
        return False


_TORCH_VALUES = ("float16", "bfloat16", "float32", "float64")


def _torch_sparse(a):
    """The torch module if `a` is a torch tensor of a sparse layout, else None (torch is never imported here)."""
    torch = sys.modules.get("torch")
    if torch is not None and isinstance(a, torch.Tensor) and a.layout != torch.strided:
        return torch
    return None


def _check_torch_sparse(t, torch, device):
    """Raise if the torch sparse tensor `t` cannot be factorized with sparse=True on CUDA device `device` (None: any)."""
    if t.layout not in (torch.sparse_coo, torch.sparse_csr, torch.sparse_csc):
        raise TypeError("sparse=True takes torch tensors of layout sparse_coo, sparse_csr or sparse_csc, got %s" % t.layout)
    if t.dim() != 2 or t.dense_dim() != 0:
        raise TypeError("sparse=True needs a 2-D torch sparse tensor without batch or dense (hybrid) dimensions, "
                        "got shape %r with %d dense dimensions" % (tuple(t.shape), t.dense_dim()))
    if str(t.dtype).replace("torch.", "") not in _TORCH_VALUES:
        raise TypeError("sparse=True needs float16, bfloat16, float32 or float64 values, got %s" % t.dtype)
    if device is not None and t.is_cuda and t.device.index != device:
        raise ValueError("the tensor is on %s but the object computes on cuda:%d; move it there first" % (t.device, device))


class _Factor(object):
    """Host array + bookkeeping for one of W / H.

    ``host``       the numpy array the user sees (identity preserved across updates, like the
                   reference's in-place ``*=`` / ``/=``, SURVEY 3.4)
    ``dev_newer``  the device copy holds newer values than ``host``
    ``host_dirty`` ``host`` may hold values the device has not seen (assigned, or handed out)
    """
    __slots__ = ("host", "dev_newer", "host_dirty", "user_owned")

    def __init__(self, host, user_owned=False):
        self.host = host
        self.dev_newer = False
        self.host_dirty = True
        self.user_owned = user_owned      # the caller holds a reference to `host`: keep it current (in-place contract)


class NMF(object):
    """
    NMF(data, num_bases=4)

    Non-negative Matrix Factorization with Lee-Seung multiplicative updates,
    ``|data - W*H|`` minimised over non-negative ``W`` (data_dimension x num_bases) and
    ``H`` (num_bases x num_samples).  Drop-in for ``pymf.NMF`` (pymf/nmf.py:23).

    Extra keyword-only arguments (no reference counterpart):
      device         CUDA device index (default: LOCAL_RANK or 0)
      process_group  ``True`` or a ``torch.distributed`` group: ``data`` is this rank's block
                     of COLUMNS, W is replicated, ``.H`` is the local block, ``.ferr`` is global
      path           "auto" | "simt" | "tc"  kernel family (default auto)
      sparse         ``True``: ``data`` is a 2-D scipy.sparse matrix or array (any format), or a 2-D torch sparse
                     tensor (``sparse_coo``, coalesced or not, ``sparse_csr`` or ``sparse_csc``; int32 / int64
                     indices; float16 / bfloat16 / float32 / float64 values; on the CPU or on ``device``),
                     factorized without densifying it; ``ferr`` / ``frobenius_norm()`` are the real ||data - W H||.
                     A torch tensor is put into canonical form on the GPU (entries sorted, duplicates summed in
                     float64 and rounded once to float32); the tensor itself is left as it is
    """

    _EPS = 10 ** -8                      # pymf/nmf.py:69
    _engine_factory = Engine             # tests substitute a checker-backed double here
    _variant = "nmf"                     # update rules the engine applies (subclasses: "snmf")

    def __init__(self, data, num_bases=4, **kw):
        device = kw.pop("device", None)
        self._pg = kw.pop("process_group", None)
        self._path = kw.pop("path", None)
        self._sparse = bool(kw.pop("sparse", False))
        if kw:
            raise TypeError("unexpected keyword arguments: %s" % ", ".join(sorted(kw)))
        if self._sparse:
            torch = _torch_sparse(data)
            if torch is not None:
                _check_torch_sparse(data, torch, None)                # the device is checked below, once it is known
            elif not _is_sparse(data):
                raise TypeError("sparse=True needs a scipy.sparse matrix or array or a torch sparse tensor as data, "
                                "got %s" % type(data).__name__)
            if self._path in ("simt", "tc"):
                raise ValueError("path=%r names a dense kernel family; sparse data runs on its own passes" % self._path)

        def setup_logging():                                   # pymf/nmf.py:73-90
            self._logger = logging.getLogger("pymf")
            if len(self._logger.handlers) < 1:
                ch = logging.StreamHandler()
                ch.setLevel(logging.DEBUG)
                ch.setFormatter(logging.Formatter("%(asctime)s [%(levelname)s] %(message)s"))
                self._logger.addHandler(ch)

        setup_logging()
        self._engine = None
        self._x_uploaded = False
        self._factors = {}
        self.timings = {}                                      # seconds of the last factorize(): upload_s, iterate_s, download_s
        self._data = data                                      # by reference, :93
        self._num_bases = num_bases                            # :94
        (self._data_dimension, n_local) = self._data.shape     # :97
        self._n_local = int(n_local)
        self._col0 = 0
        self._world, self._rank = 1, 0
        if self._pg is not None:
            self._init_distributed()
        self._num_samples = self._n_global if self._pg is not None else self._n_local
        if device is None:
            import os
            device = int(os.environ.get("LOCAL_RANK", "0")) if self._pg is not None else 0
        self._device = int(device)
        if self._sparse and _torch_sparse(data) is not None:
            _check_torch_sparse(data, _torch_sparse(data), self._device)

    # ------------------------------------------------------------------ distributed plumbing
    def _dist(self):
        import torch.distributed as dist
        return dist

    def _group(self):
        return None if self._pg is True else self._pg

    def _init_distributed(self):
        dist = self._dist()
        import torch
        g = self._group()
        self._world, self._rank = dist.get_world_size(g), dist.get_rank(g)
        sizes = [None] * self._world
        dist.all_gather_object(sizes, int(self._n_local), group=g)
        self._n_global = int(sum(sizes))
        self._col0 = int(sum(sizes[:self._rank]))

    # NCCL communicators are created once per (process group, device) and shared by every NMF object of this
    # process (creating one and warming it up costs 1-2 s; all ranks construct their objects in the same order,
    # so the cache stays in step across ranks).
    _comm_cache = {}

    def _attach_comm(self):
        eng = self._engine
        if not hasattr(eng, "comm_attach"):                    # engine doubles of the CPU tests
            box = [eng.comm_unique_id() if self._rank == 0 else None]
            self._broadcast(box)
            eng.comm_init(box[0], self._world, self._rank)
            return
        key = ("WORLD" if self._group() is None else id(self._group()), self._device, self._world, self._rank)
        comm = NMF._comm_cache.get(key)
        if comm is None:
            box = [eng.comm_unique_id() if self._rank == 0 else None]
            self._broadcast(box)
            comm = type(eng).comm_create(box[0], self._world, self._rank, self._device)
            NMF._comm_cache[key] = comm
        eng.comm_attach(comm, self._world, self._rank)

    def _broadcast(self, box):
        dist = self._dist()
        dist.broadcast_object_list(box, src=dist.get_global_rank(self._group(), 0)
                                   if self._group() is not None else 0, group=self._group())

    # ------------------------------------------------------------------ attributes
    @property
    def data(self):
        return self._data

    @data.setter
    def data(self, value):
        self._data = value
        self._x_uploaded = False

    def _get_factor(self, name):
        f = self._factors.get(name)
        if f is None:
            raise AttributeError("'NMF' object has no attribute '%s'" % name)
        if f.dev_newer:
            self._download(name, f)
        # Handed out: the caller may mutate it in place (mdl.W[...] = ...), which cannot be observed, so the
        # next device call re-uploads this factor.  An exact change check (keep a copy + compare) costs as
        # much host bandwidth as the upload it would save.
        f.host_dirty = True
        return f.host

    def _download(self, name, f):
        eng = self._engine
        fresh = (eng.get_w(np.float64, out=f.host) if name == "W"
                 else eng.get_h(np.float64, out=f.host))
        if fresh is not f.host:
            f.host[...] = fresh                       # in place: `mdl.W is W` stays true
        f.dev_newer = False

    def _set_factor(self, name, value):
        user_owned = isinstance(value, np.ndarray) and value.dtype.kind == "f" and value.flags.writeable
        if not user_owned:
            value = np.array(value, dtype=np.float64)
        self._factors[name] = _Factor(value, user_owned)

    W = property(lambda self: self._get_factor("W"), lambda self, v: self._set_factor("W", v),
                 lambda self: self._factors.pop("W", None))
    H = property(lambda self: self._get_factor("H"), lambda self, v: self._set_factor("H", v),
                 lambda self: self._factors.pop("H", None))

    # ------------------------------------------------------------------ engine
    def _ensure_engine(self):
        if self._sparse:
            if not (_is_sparse(self._data) or _torch_sparse(self._data) is not None):
                raise TypeError("sparse=True needs a scipy.sparse matrix or array or a torch sparse tensor as data")
        elif _is_sparse(self._data):
            raise TypeError("sparse data is not supported by the NMF multiplicative-update path")
        if self._engine is None:
            self._engine = self._engine_factory(self._data_dimension, self._n_local, self._num_bases,
                                                device=self._device, n_global=self._num_samples,
                                                col0=self._col0, path=self._path)
            if self._world > 1:
                self._attach_comm()
            if self._variant != "nmf":
                self._engine.set_variant(self._variant)
        if not self._x_uploaded:
            self._upload_data()
            self._x_uploaded = True
        return self._engine

    def _upload_data(self):
        x = self._data
        if self._sparse and _torch_sparse(x) is not None:
            self._upload_torch_sparse(x, _torch_sparse(x))
            return
        if self._sparse:
            # canonical CSC of a copy (the caller's matrix is left as it is): duplicates summed, rows sorted
            m = x.tocsc(copy=True)
            m.sum_duplicates()
            if m.shape != (self._data_dimension, self._n_local):
                raise ValueError("data shape %r != (%d, %d)" % (m.shape, self._data_dimension, self._n_local))
            vals = m.data if m.data.dtype in (np.float32, np.float64) else m.data.astype(np.float64)
            self._engine.upload_x_csc(np.ascontiguousarray(m.indptr, dtype=np.int64),
                                      np.ascontiguousarray(m.indices, dtype=np.int32), np.ascontiguousarray(vals))
            return
        torch = sys.modules.get("torch")             # a torch.Tensor implies torch is imported; never import it here
        if torch is not None:
            if isinstance(x, torch.Tensor):
                if x.is_cuda:
                    if x.dtype != torch.float32 or x.stride(1) != 1 or x.stride(0) % 4 or x.data_ptr() % 16:
                        x = x.to(torch.float32).contiguous()
                        if x.stride(0) % 4:
                            pad = (-x.shape[1]) % 4
                            x = torch.nn.functional.pad(x, (0, pad))[:, :self._n_local]
                    self._engine.bind_x_device(x.data_ptr(), x.stride(0), keepalive=x)
                    return
                x = x.numpy()
        if not isinstance(x, np.ndarray):
            if hasattr(x, "shape") and hasattr(x, "__getitem__") and len(getattr(x, "shape", ())) == 2:
                # h5py-style sources (the reason for the reference's `data[:,:]`, pymf/nmf.py:110,125,131): read
                # column panels data[:, c0:c1], never the whole matrix, straight into the device copy
                self._engine.upload_x_panels(x)
                return
            x = np.asarray(x)                        # lists / array-likes
        self._engine.upload_x(x)

    def _upload_torch_sparse(self, t, torch):
        """Hand the index and value arrays of a torch sparse tensor to the library as they are (no coalesce, no
        layout conversion): it validates them and builds the canonical CSC on the device."""
        _check_torch_sparse(t, torch, self._device)
        if tuple(t.shape) != (self._data_dimension, self._n_local):
            raise ValueError("data shape %r != (%d, %d)" % (tuple(t.shape), self._data_dimension, self._n_local))
        if t.layout == torch.sparse_coo:
            layout, a, b, vals = "coo", t._indices()[0], t._indices()[1], t._values()
        elif t.layout == torch.sparse_csr:
            layout, a, b, vals = "csr", t.crow_indices(), t.col_indices(), t.values()
        else:
            layout, a, b, vals = "csc", t.ccol_indices(), t.row_indices(), t.values()
        if vals.dtype in (torch.float16, torch.bfloat16):
            vals = vals.to(torch.float32)                    # exact
        self._engine.upload_x_sparse_device(layout, a, b, vals)

    def _sync_to_device(self):
        eng = self._ensure_engine()
        if self._world > 1:
            self._replicate_w()
        for name, setter in (("W", eng.set_w), ("H", eng.set_h)):
            f = self._factors.get(name)
            if f is not None and f.host_dirty:
                setter(f.host)
                f.host_dirty = False
                f.dev_newer = False
        return eng

    def _replicate_w(self):
        """W is REPLICATED across the ranks of the process group, but every rank draws (init_w) or is handed
        its own host copy.  Before any rank uploads a host-side W, rank 0's values are broadcast into every
        rank's array (in place), so the replicas start bit-identical whether or not the caller seeded numpy
        identically.  Collective: all ranks decide together (one small all-reduce of the dirty flags)."""
        import torch
        dist = self._dist()
        g = self._group()
        f = self._factors.get("W")
        backend = str(dist.get_backend(g))
        dev = torch.device("cuda", self._device) if "nccl" in backend else torch.device("cpu")
        flag = torch.tensor([1 if (f is not None and f.host_dirty) else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=g)
        if int(flag.item()) == 0:
            return
        if f is None:
            raise RuntimeError("W is set on some ranks of the process group but not on this one")
        if f.dev_newer:                                          # this rank's current values live on the device
            self._get_factor("W")
        src = dist.get_global_rank(g, 0) if g is not None else 0
        t = torch.from_numpy(np.ascontiguousarray(f.host, dtype=np.float64)).to(dev)
        dist.broadcast(t, src=src, group=g)
        f.host[...] = t.cpu().numpy()
        f.host_dirty = True

    def _mark_device_newer(self, name):
        f = self._factors[name]
        f.dev_newer = True

    # ------------------------------------------------------------------ reference hooks
    def frobenius_norm(self):
        """||data - W H||_F (pymf/nmf.py:100-114); -123456 if W/H are missing, or if data is sparse and the object
        was not built with sparse=True."""
        if "H" in self._factors and "W" in self._factors and (self._sparse or not _is_sparse(self._data)):
            return self._sync_to_device().frobenius()
        return _SENTINEL

    def init_w(self):                                                    # pymf/nmf.py:116-117
        self.W = np.random.random((self._data_dimension, self._num_bases))

    def init_h(self):                                                    # pymf/nmf.py:119-120
        if self._world > 1:
            # Same stream as a single-process run with the same seed (element (j, c) is draw j * n + c of numpy's
            # global generator, which cannot skip ahead): one ROW of the global H at a time, keeping our columns,
            # so a rank never holds more than its own k x n_local block plus one row.
            H = np.empty((self._num_bases, self._n_local))
            for j in range(self._num_bases):
                H[j] = np.random.random(self._num_samples)[self._col0:self._col0 + self._n_local]
            self.H = H
        else:
            self.H = np.random.random((self._num_bases, self._num_samples))

    def update_h(self):                                                  # pymf/nmf.py:122-126
        self._sync_to_device().run(1, compute_w=False, compute_h=True, compute_err=False, early_stop=False)
        self._mark_device_newer("H")

    def update_w(self):                                                  # pymf/nmf.py:128-132
        self._sync_to_device().run(1, compute_w=True, compute_h=False, compute_err=False, early_stop=False)
        self._mark_device_newer("W")

    def converged(self, i):                                              # pymf/nmf.py:134-139
        derr = np.abs(self.ferr[i] - self.ferr[i - 1]) / self._num_samples
        return bool(derr < self._EPS)

    def _hooks_overridden(self):
        """True when a subclass replaced a hook with Python code of its own.  ``_native_hooks`` names the
        class whose update_w / update_h run natively (NMF, or BNMF / SNMF for their own overrides)."""
        cls = type(self)
        native = self._native_hooks()
        return any(getattr(cls, h) is not getattr(base, h)
                   for h, base in (("update_w", native), ("update_h", native),
                                   ("frobenius_norm", NMF), ("converged", NMF)))

    @staticmethod
    def _native_hooks():
        return NMF

    # ------------------------------------------------------------------ the driver
    def factorize(self, niter=1, show_progress=False,
                  compute_w=True, compute_h=True, compute_err=True):
        """Factorize s.t. WH = data (pymf/nmf.py:141-202).

        niter, show_progress, compute_w, compute_h, compute_err as in the reference.
        Updates .W, .H and (if compute_err) .ferr.
        """
        self._logger.setLevel(logging.INFO if show_progress else logging.ERROR)   # :166-169

        if "W" not in self._factors:                                              # :173-174
            self.init_w()
        if "H" not in self._factors:                                              # :176-177
            self.init_h()

        if self._hooks_overridden():
            return self._factorize_template(niter, compute_w, compute_h, compute_err)

        t0 = time.perf_counter()
        eng = self._sync_to_device()
        t1 = time.perf_counter()
        ferr, done = eng.run(niter, compute_w=compute_w, compute_h=compute_h,
                             compute_err=compute_err, early_stop=True)
        t2 = time.perf_counter()
        if compute_w and done > 0:
            self._mark_device_newer("W")
        if compute_h and done > 0:
            self._mark_device_newer("H")
        # The reference updates W / H in place (pymf/nmf.py:125-126,131-132): an array the caller assigned and
        # still holds must show the new values after factorize() returns, not only after `.W` is read again.
        # Arrays this object created itself are brought back lazily, on first read.
        for name in ("W", "H"):
            f = self._factors[name]
            if f.user_owned and f.dev_newer:
                self._download(name, f)
        self.timings = {"upload_s": t1 - t0, "iterate_s": t2 - t1, "download_s": time.perf_counter() - t2}
        if compute_err:
            full = np.zeros(niter)                                                # :179-180
            full[:len(ferr)] = ferr
            self.ferr = full[:len(ferr)] if done < niter or len(ferr) < niter else full
        if show_progress:
            for i in range(done):                                                 # :191-194
                if compute_err and i < len(ferr):
                    self._logger.info('Iteration ' + str(i + 1) + '/' + str(niter) + ' FN:' + str(ferr[i]))
                else:
                    self._logger.info('Iteration ' + str(i + 1) + '/' + str(niter))

    def _factorize_template(self, niter, compute_w, compute_h, compute_err):
        """The reference's template-method loop, used when a subclass overrides a hook."""
        if compute_err:
            self.ferr = np.zeros(niter)
        for i in range(niter):
            if compute_w:
                self.update_w()
            if compute_h:
                self.update_h()
            if compute_err:
                self.ferr[i] = self.frobenius_norm()
                self._logger.info('Iteration ' + str(i + 1) + '/' + str(niter) + ' FN:' + str(self.ferr[i]))
            else:
                self._logger.info('Iteration ' + str(i + 1) + '/' + str(niter))
            if i > 1 and compute_err:
                if self.converged(i):
                    self.ferr = self.ferr[:i]
                    break
