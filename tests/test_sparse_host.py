"""Host logic of NMF(..., sparse=True) on CPU: scipy.sparse normalisation, the arrays handed to the engine, the
constructor errors and column sharding over gloo, with an oracle-backed engine double that densifies the CSC arrays."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sps
import torch.multiprocessing as mp

import pymf_b200
from oracle import nmf_oracle as O
from tests._fake_engine import FakeEngine


class SparseFakeEngine(FakeEngine):
    """FakeEngine plus upload_x_csc: records the arrays it was handed and densifies them."""

    def upload_x_csc(self, indptr, indices, values):
        self.csc = (indptr, indices, values)
        self.X = sps.csc_matrix((np.asarray(values, dtype=np.float64), indices, indptr),
                                shape=(self.d, self.n_local)).toarray()
        self.uploads["x"] += 1


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(pymf_b200.NMF, "_engine_factory", SparseFakeEngine)
    return SparseFakeEngine


def _matrix(d=23, n=41, density=0.2, seed=3):
    return sps.random(d, n, density=density, format="csc", random_state=np.random.RandomState(seed), dtype=np.float64)


@pytest.mark.parametrize("flags", [(True, True, True), (True, False, True), (False, True, True), (True, True, False)])
def test_trajectory_matches_oracle_on_the_dense_matrix(fake, flags):
    cw, ch, ce = flags
    X = _matrix()
    Xd = X.toarray()
    d, n, k = Xd.shape[0], Xd.shape[1], 4
    np.random.seed(7)
    W0, H0 = np.random.random((d, k)), np.random.random((k, n))
    m = pymf_b200.NMF(X, num_bases=k, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=6, compute_w=cw, compute_h=ch, compute_err=ce)
    W, H = W0.copy(), H0.copy()
    ferr = O.factorize(Xd, W, H, niter=6, compute_w=cw, compute_h=ch, compute_err=ce)
    np.testing.assert_allclose(m.W, W, rtol=1e-12)
    np.testing.assert_allclose(m.H, H, rtol=1e-12)
    if ce:
        np.testing.assert_allclose(m.ferr, ferr, rtol=1e-12)
    # warm start: a second factorize continues from the factors of the first
    m.factorize(niter=3, compute_w=cw, compute_h=ch, compute_err=ce)
    ferr2 = O.factorize(Xd, W, H, niter=3, compute_w=cw, compute_h=ch, compute_err=ce)
    np.testing.assert_allclose(m.W, W, rtol=1e-12)
    np.testing.assert_allclose(m.H, H, rtol=1e-12)
    if ce:
        np.testing.assert_allclose(m.ferr, ferr2, rtol=1e-12)
    assert m._engine.uploads["x"] == 1


def test_frobenius_norm_is_the_real_error(fake):
    X = _matrix()
    m = pymf_b200.NMF(X, num_bases=3, sparse=True)
    np.random.seed(1)
    m.W, m.H = np.random.random((23, 3)), np.random.random((3, 41))
    assert m.frobenius_norm() == pytest.approx(np.linalg.norm(X.toarray() - m.W.dot(m.H)), rel=1e-12)
    # without the keyword the reference's sentinel stays
    m2 = pymf_b200.NMF(X, num_bases=3)
    m2.W, m2.H = m.W, m.H
    assert m2.frobenius_norm() == -123456


def _inputs():
    base = _matrix(density=0.3, seed=5)
    coo = base.tocoo()
    # duplicates: split every value into two halves stored as separate entries, in shuffled order
    rng = np.random.RandomState(2)
    order = rng.permutation(2 * coo.nnz)
    rows = np.concatenate([coo.row, coo.row])[order]
    cols = np.concatenate([coo.col, coo.col])[order]
    vals = np.concatenate([coo.data * 0.25, coo.data * 0.75])[order]
    dup = sps.coo_matrix((vals, (rows, cols)), shape=base.shape)
    unsorted = base.copy()
    for c in range(unsorted.shape[1]):                      # reverse the rows within every column
        a, b = unsorted.indptr[c], unsorted.indptr[c + 1]
        unsorted.indices[a:b] = unsorted.indices[a:b][::-1].copy()
        unsorted.data[a:b] = unsorted.data[a:b][::-1].copy()
    unsorted.has_sorted_indices = False
    i64 = base.copy()
    i64.indices = i64.indices.astype(np.int64)
    i64.indptr = i64.indptr.astype(np.int64)
    return base, {
        "csc": base.copy(), "csr": base.tocsr(), "coo": base.tocoo(), "csc_array": sps.csc_array(base),
        "unsorted": unsorted, "duplicates": dup, "float32": base.astype(np.float32), "int64_indices": i64,
    }


def _snapshot(x):
    if x.format == "coo":
        return [np.array(a, copy=True) for a in (x.row, x.col, x.data)]
    return [np.array(a, copy=True) for a in (x.indptr, x.indices, x.data)]


@pytest.mark.parametrize("kind", ["csc", "csr", "coo", "csc_array", "unsorted", "duplicates", "float32", "int64_indices"])
def test_canonical_csc_reaches_the_engine_and_the_input_is_untouched(fake, kind):
    base, inputs = _inputs()
    x = inputs[kind]
    before = _snapshot(x)
    m = pymf_b200.NMF(x, num_bases=2, sparse=True)
    m.factorize(niter=1)
    indptr, indices, values = m._engine.csc
    assert indptr.dtype == np.int64 and indices.dtype == np.int32
    assert values.dtype == (np.float32 if kind == "float32" else np.float64)
    ref = base.astype(values.dtype)
    np.testing.assert_array_equal(indptr, ref.indptr)
    np.testing.assert_array_equal(indices, ref.indices)
    np.testing.assert_allclose(values, ref.data, rtol=1e-15 if kind != "float32" else 1e-7)
    for c in range(base.shape[1]):
        assert np.all(np.diff(indices[indptr[c]:indptr[c + 1]]) > 0)
    for a, b in zip(before, _snapshot(x)):
        np.testing.assert_array_equal(a, b)
        assert a.dtype == b.dtype


def test_assigning_data_uploads_again(fake):
    m = pymf_b200.NMF(_matrix(), num_bases=2, sparse=True)
    m.factorize(niter=1)
    other = _matrix(seed=9)
    m.data = other
    m.factorize(niter=1)
    assert m._engine.uploads["x"] == 2
    np.testing.assert_array_equal(m._engine.X, other.toarray())


def test_constructor_errors():
    X = _matrix()
    with pytest.raises(TypeError):
        pymf_b200.NMF(X.toarray(), num_bases=2, sparse=True)
    for path in ("simt", "tc"):
        with pytest.raises(ValueError):
            pymf_b200.NMF(X, num_bases=2, sparse=True, path=path)
    with pytest.raises(TypeError):
        pymf_b200.NNDSVD(X, num_bases=2, sparse=True)
    for cls in (pymf_b200.BNMF, pymf_b200.SNMF):
        with pytest.raises(TypeError):
            cls(X.toarray(), num_bases=2, sparse=True)
        cls(X, num_bases=2, sparse=True)


# ---- two ranks over gloo, sparse column blocks (as tests/test_dist_gloo.py does for dense blocks) ----
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, d, n, k, niter, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pymf_b200.NMF._engine_factory = SparseFakeEngine
        X = _matrix(d, n, 0.25, 42)
        bounds = [int(round(n * r / float(world))) for r in range(world + 1)]
        lo, hi = bounds[rank], bounds[rank + 1]
        np.random.seed(9)
        m = pymf_b200.NMF(X[:, lo:hi], num_bases=k, process_group=True, sparse=True)
        assert m._num_samples == n and m._col0 == lo
        m.factorize(niter=niter)
        np.savez(os.path.join(out, "r%d.npz" % rank), W=m.W, H=m.H, ferr=m.ferr, lo=lo, hi=hi)
    finally:
        dist.destroy_process_group()


def test_two_rank_sparse_column_blocks_match_single_process(tmp_path):
    d, n, k, niter, world = 17, 101, 4, 10, 2
    mp.spawn(_worker, args=(world, _free_port(), d, n, k, niter, str(tmp_path)), nprocs=world, join=True)
    X = _matrix(d, n, 0.25, 42).toarray()
    np.random.seed(9)
    W, H = O.init_wh(d, n, k)
    ferr = O.factorize(X, W, H, niter=niter)
    parts = [np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world)]
    for p in parts:
        np.testing.assert_allclose(p["W"], W, rtol=1e-9)
        np.testing.assert_allclose(p["H"], H[:, int(p["lo"]):int(p["hi"])], rtol=1e-9)
        np.testing.assert_allclose(p["ferr"], ferr, rtol=1e-9)
    np.testing.assert_array_equal(parts[0]["W"], parts[1]["W"])
