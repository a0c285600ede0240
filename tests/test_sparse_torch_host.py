"""Host logic of NMF(torch_sparse_tensor, sparse=True) on CPU: which arrays reach the engine for every layout, index and
value dtype, the constructor errors, column sharding over gloo, and the import rule.  The engine double canonicalises
with the numpy reference below, which is also what the GPU tests (tests/test_sparse_torch.py) hold the library to."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sps
import torch
import torch.multiprocessing as mp

import pymf_b200
from oracle import nmf_oracle as O
from tests.test_sparse_host import SparseFakeEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- reference canonicalisation --------------------------------------------------------------------------------------
def reference_csc(rows, cols, vals, shape):
    """The canonical CSC of (rows, cols, vals) in their input order: (1) stable lexsort by (column, row), (2) the
    duplicates of each (row, column) summed in float64 in input order, (3) cast to float32, (4) a scipy CSC with
    int32 rows and int64 column pointers.  Explicit zeros stay."""
    d, n = shape
    rows, cols = np.asarray(rows, dtype=np.int64), np.asarray(cols, dtype=np.int64)
    order = np.lexsort((rows, cols))                        # stable: equal keys keep their input order
    key = cols[order] * d + rows[order]
    ukey, inv = np.unique(key, return_inverse=True)
    sums = np.bincount(inv.ravel(), weights=np.asarray(vals, dtype=np.float64)[order], minlength=ukey.size)
    indptr = np.searchsorted(ukey, np.arange(n + 1, dtype=np.int64) * d).astype(np.int64)
    return sps.csc_matrix((sums.astype(np.float32), (ukey % d).astype(np.int32), indptr), shape=shape)


def triplets(layout, a, b, vals, shape):
    """(rows, cols, float64 values) of the arrays handed to upload_x_sparse_device, in their storage order."""
    a, b = a.cpu().numpy().astype(np.int64), b.cpu().numpy().astype(np.int64)
    v = vals.cpu().to(torch.float64).numpy()
    if layout == "coo":
        return a, b, v
    outer = np.repeat(np.arange(a.size - 1, dtype=np.int64), np.diff(a))
    return (outer, b, v) if layout == "csr" else (b, outer, v)


def tensor_triplets(t):
    """triplets() of a torch sparse tensor, read from its storage without coalescing."""
    if t.layout == torch.sparse_coo:
        return triplets("coo", t._indices()[0], t._indices()[1], t._values(), t.shape)
    if t.layout == torch.sparse_csr:
        return triplets("csr", t.crow_indices(), t.col_indices(), t.values(), t.shape)
    return triplets("csc", t.ccol_indices(), t.row_indices(), t.values(), t.shape)


def reference_of(t):
    return reference_csc(*tensor_triplets(t), shape=tuple(t.shape))


def messy_coo(d, n, density, seed, dup=0.01, zeros=0, dtype=torch.float32):
    """Uncoalesced COO tensor: entries in random order, about `dup` of them repeated (with other values), `zeros`
    explicit zeros."""
    rng = np.random.RandomState(seed)
    nnz = max(1, int(d * n * density))
    key = np.unique(rng.randint(0, d * n, size=nnz).astype(np.int64))
    extra = key[rng.randint(0, key.size, size=int(np.ceil(dup * key.size)))]
    key = np.concatenate([key, extra])[rng.permutation(key.size + extra.size)]
    vals = 1.0 - rng.random_sample(key.size)
    if zeros:
        vals[rng.choice(key.size, size=min(zeros, key.size), replace=False)] = 0.0
    idx = torch.from_numpy(np.stack([key % d, key // d]))
    t = torch.sparse_coo_tensor(idx, torch.from_numpy(vals).to(dtype), (d, n), check_invariants=False)
    assert not t.is_coalesced()
    return t


def as_layout(coo, layout, index_dtype=torch.int64, shuffle_rows=False, seed=0):
    """coo (uncoalesced) as a CSR or CSC tensor holding the same entries, duplicates included, built from raw arrays.
    shuffle_rows: the entries of each CSC column in random order."""
    d, n = coo.shape
    rows, cols = coo._indices()[0].numpy(), coo._indices()[1].numpy()
    vals = coo._values()
    outer, inner = (rows, cols) if layout == "csr" else (cols, rows)
    m = d if layout == "csr" else n
    order = np.argsort(outer, kind="stable")
    if shuffle_rows:
        rng = np.random.RandomState(seed)
        order = np.lexsort((rng.random_sample(outer.size), outer))
    ptr = np.searchsorted(outer[order], np.arange(m + 1))
    p = torch.from_numpy(ptr).to(index_dtype)
    i = torch.from_numpy(inner[order].copy()).to(index_dtype)
    v = vals[torch.from_numpy(order)]
    if layout == "csr":
        return torch.sparse_csr_tensor(p, i, v, (d, n), check_invariants=False)
    return torch.sparse_csc_tensor(p, i, v, (d, n), check_invariants=False)


def test_reference_matches_scipy_sum_duplicates():
    t = messy_coo(30, 40, 0.2, 1, dup=0.3, zeros=5, dtype=torch.float64)
    rows, cols, vals = tensor_triplets(t)
    ref = reference_csc(rows, cols, vals, (30, 40))
    m = sps.coo_matrix((vals, (rows, cols)), shape=(30, 40)).tocsc()
    m.sum_duplicates()
    np.testing.assert_array_equal(ref.indptr, m.indptr)
    np.testing.assert_array_equal(ref.indices, m.indices)
    np.testing.assert_allclose(ref.data, m.data.astype(np.float32), rtol=1e-7)
    assert ref.nnz == m.nnz and np.sum(ref.data == 0) == np.sum(m.data == 0) > 0     # explicit zeros kept


# ---- engine double -----------------------------------------------------------------------------------------------------
class TorchSparseFakeEngine(SparseFakeEngine):
    """Takes upload_x_sparse_device with CPU tensors: records what it was handed and canonicalises with the reference."""

    def upload_x_sparse_device(self, layout, a, b, values):
        self.handed = (layout, a, b, values)
        rows, cols, vals = triplets(layout, a, b, values, (self.d, self.n_local))
        ref = reference_csc(rows, cols, vals, (self.d, self.n_local))
        self.X = ref.astype(np.float64).toarray()
        self.uploads["x"] += 1


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(pymf_b200.NMF, "_engine_factory", TorchSparseFakeEngine)
    return TorchSparseFakeEngine


LAYOUTS = ["coo", "csr", "csc"]
VALUE_DTYPES = [torch.float16, torch.bfloat16, torch.float32, torch.float64]


def _input(layout, index_dtype, value_dtype, seed=3):
    coo = messy_coo(23, 41, 0.2, seed, dup=0.1, zeros=2, dtype=value_dtype)
    return coo if layout == "coo" else as_layout(coo, layout, index_dtype, shuffle_rows=(layout == "csc"), seed=seed)


def _combos():
    out = []
    for layout in LAYOUTS:
        for idt in ([torch.int64] if layout == "coo" else [torch.int32, torch.int64]):
            for vdt in VALUE_DTYPES:
                out.append((layout, idt, vdt))
    return out


@pytest.mark.parametrize("layout,index_dtype,value_dtype", _combos(), ids=lambda v: str(v).replace("torch.", ""))
def test_arrays_reach_the_engine_and_the_input_is_untouched(fake, layout, index_dtype, value_dtype):
    t = _input(layout, index_dtype, value_dtype)
    before = [x.clone() for x in _parts(t)]
    m = pymf_b200.NMF(t, num_bases=2, sparse=True)
    m.factorize(niter=1)
    got, a, b, vals = m._engine.handed
    assert got == layout
    assert a.dtype == b.dtype == index_dtype
    assert vals.dtype == (torch.float64 if value_dtype == torch.float64 else torch.float32)
    parts = _parts(t)
    torch.testing.assert_close(a, parts[0], rtol=0, atol=0)
    torch.testing.assert_close(b, parts[1], rtol=0, atol=0)
    torch.testing.assert_close(vals, parts[2].to(vals.dtype), rtol=0, atol=0)      # widening is exact
    np.testing.assert_array_equal(m._engine.X, reference_of(t).astype(np.float64).toarray())
    for x, y in zip(before, _parts(t)):
        assert x.dtype == y.dtype and torch.equal(x, y)


def _parts(t):
    if t.layout == torch.sparse_coo:
        return t._indices()[0], t._indices()[1], t._values()
    if t.layout == torch.sparse_csr:
        return t.crow_indices(), t.col_indices(), t.values()
    return t.ccol_indices(), t.row_indices(), t.values()


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("cls", ["NMF", "BNMF", "SNMF"])
def test_trajectories_match_the_oracle_on_the_dense_matrix(fake, layout, cls):
    t = _input(layout, torch.int64, torch.float64, seed=5)
    Xd = reference_of(t).astype(np.float64).toarray()
    d, n, k = 23, 41, 4
    np.random.seed(7)
    W0, H0 = np.random.random((d, k)), np.random.random((k, n))
    m = getattr(pymf_b200, cls)(t, num_bases=k, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=6)
    W, H = W0.copy(), H0.copy()
    if cls == "NMF":
        ferr = O.factorize(Xd, W, H, niter=6)
    elif cls == "BNMF":
        ferr = O.bnmf_factorize(Xd, W, H, niter=6)
    else:
        W, ferr = O.snmf_factorize(Xd, W, H, niter=6)
    np.testing.assert_allclose(m.W, W, rtol=1e-12)
    np.testing.assert_allclose(m.H, H, rtol=1e-12)
    np.testing.assert_allclose(m.ferr, ferr, rtol=1e-12)
    assert m.frobenius_norm() == pytest.approx(np.linalg.norm(Xd - m.W.dot(m.H)), rel=1e-12)


def test_switching_between_scipy_torch_and_dense_data(fake, monkeypatch):
    t = _input("coo", torch.int64, torch.float32)
    ref = reference_of(t)
    m = pymf_b200.NMF(ref, num_bases=2, sparse=True)
    m.factorize(niter=1)
    m.data = t
    m.factorize(niter=1)
    assert m._engine.handed[0] == "coo" and m._engine.uploads["x"] == 2
    m.data = ref
    m.factorize(niter=1)
    assert m._engine.uploads["x"] == 3
    dense = pymf_b200.NMF(ref.toarray(), num_bases=2)
    dense.factorize(niter=1)
    with pytest.raises(TypeError):                              # a dense tensor on a sparse=True object
        m.data = torch.from_numpy(ref.toarray())
        m.factorize(niter=1)


def test_constructor_errors():
    t = _input("coo", torch.int64, torch.float32)
    dense = t.to_dense()
    with pytest.raises(TypeError):
        pymf_b200.NMF(dense, num_bases=2, sparse=True)
    with pytest.raises(TypeError):                              # 3-D
        pymf_b200.NMF(torch.sparse_coo_tensor(torch.zeros(3, 1, dtype=torch.int64), torch.ones(1), (2, 2, 2)),
                      num_bases=2, sparse=True)
    with pytest.raises(TypeError):                              # hybrid: a dense dimension
        pymf_b200.NMF(torch.sparse_coo_tensor(torch.zeros(2, 1, dtype=torch.int64), torch.ones(1, 3), (2, 2, 3)),
                      num_bases=2, sparse=True)
    with pytest.raises(TypeError):                              # batched CSR
        pymf_b200.NMF(torch.zeros(2, 3, 4).to_sparse_csr(), num_bases=2, sparse=True)
    for layout in ("to_sparse_bsr", "to_sparse_bsc"):
        with pytest.raises(TypeError):
            pymf_b200.NMF(getattr(torch.ones(4, 4), layout)((2, 2)), num_bases=2, sparse=True)
    for bad in (torch.int32, torch.int64, torch.bool, torch.complex64):
        with pytest.raises(TypeError):
            pymf_b200.NMF(torch.sparse_coo_tensor(t._indices(), torch.ones(t._nnz(), dtype=bad), t.shape),
                          num_bases=2, sparse=True)
    for path in ("simt", "tc"):
        with pytest.raises(ValueError):
            pymf_b200.NMF(t, num_bases=2, sparse=True, path=path)
    with pytest.raises(TypeError):
        pymf_b200.NNDSVD(t, num_bases=2, sparse=True)
    for cls in (pymf_b200.NMF, pymf_b200.BNMF, pymf_b200.SNMF):
        for x in (t, as_layout(t, "csr"), as_layout(t, "csc", torch.int32)):
            cls(x, num_bases=2, sparse=True)


def test_product_imports_neither_torch_nor_scipy():
    code = ("import sys\nimport pymf_b200\n"
            "bad = [m for m in ('torch', 'scipy', 'scipy.sparse') if m in sys.modules]\n"
            "assert not bad, bad\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]


# ---- two ranks over gloo, torch sparse column blocks ---------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _block(t, lo, hi):
    idx, vals = t._indices(), t._values()
    keep = (idx[1] >= lo) & (idx[1] < hi)
    return torch.sparse_coo_tensor(torch.stack([idx[0][keep], idx[1][keep] - lo]), vals[keep], (t.shape[0], hi - lo),
                                   check_invariants=False)


def _worker(rank, world, port, d, n, k, niter, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pymf_b200.NMF._engine_factory = TorchSparseFakeEngine
        t = messy_coo(d, n, 0.25, 42, dup=0.05, dtype=torch.float64)
        bounds = [int(round(n * r / float(world))) for r in range(world + 1)]
        lo, hi = bounds[rank], bounds[rank + 1]
        np.random.seed(9)
        m = pymf_b200.NMF(_block(t, lo, hi), num_bases=k, process_group=True, sparse=True)
        assert m._num_samples == n and m._col0 == lo
        m.factorize(niter=niter)
        np.savez(os.path.join(out, "r%d.npz" % rank), W=m.W, H=m.H, ferr=m.ferr, lo=lo, hi=hi)
    finally:
        dist.destroy_process_group()


def test_two_rank_torch_column_blocks_match_single_process(tmp_path):
    d, n, k, niter, world = 17, 101, 4, 10, 2
    mp.spawn(_worker, args=(world, _free_port(), d, n, k, niter, str(tmp_path)), nprocs=world, join=True)
    X = reference_of(messy_coo(d, n, 0.25, 42, dup=0.05, dtype=torch.float64)).astype(np.float64).toarray()
    np.random.seed(9)
    W, H = O.init_wh(d, n, k)
    ferr = O.factorize(X, W, H, niter=niter)
    parts = [np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world)]
    for p in parts:
        np.testing.assert_allclose(p["W"], W, rtol=1e-9)
        np.testing.assert_allclose(p["H"], H[:, int(p["lo"]):int(p["hi"])], rtol=1e-9)
        np.testing.assert_allclose(p["ferr"], ferr, rtol=1e-9)
    np.testing.assert_array_equal(parts[0]["W"], parts[1]["W"])
