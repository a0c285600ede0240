"""The sparse passes (NMF / BNMF / SNMF on scipy.sparse data, pymfb_upload_x_csc) against the float64 oracle on the
densified matrix and against a float64 scipy.sparse restatement of the updates.  Needs a B200: run with `-m gpu`."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sps

import pymf_b200
from oracle import nmf_oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_WH = 1e-4
TOL_FERR = 1e-3


def rel(a, b):
    b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


def make_sparse(d, n, density, seed, power_law=False, empty=False, signed=False):
    """Seeded d x n CSC matrix, values U(0, 1] (U(-1, 1) if signed).  Column c draws counts[c] rows with replacement
    (duplicates dropped).  power_law: counts ~ (rank)^-0.9 scaled to the density (a few long columns, most short).
    empty: every 7th row and every 5th column has no entry."""
    rng = np.random.RandomState(seed)
    if power_law:
        w = 1.0 / np.arange(1, n + 1) ** 0.9
        counts = np.minimum(d, np.maximum(0, np.round(w / w.sum() * density * d * n))).astype(np.int64)
        counts = counts[rng.permutation(n)]
    else:
        counts = rng.binomial(d, density, size=n)
    cols = np.repeat(np.arange(n, dtype=np.int64), counts)
    key = np.unique(cols * d + rng.randint(0, d, size=cols.size))     # column-major, rows sorted, no duplicates
    indices = (key % d).astype(np.int32)
    indptr = np.searchsorted(key // d, np.arange(n + 1)).astype(np.int64)
    vals = rng.uniform(-1.0, 1.0, key.size) if signed else 1.0 - rng.random_sample(key.size)
    X = sps.csc_matrix((vals, indices, indptr), shape=(d, n))
    if empty:
        keep_r = np.ones(d)
        keep_r[::7] = 0
        keep_c = np.ones(n)
        keep_c[::5] = 0
        X = sps.csc_matrix(sps.diags(keep_r).dot(X).dot(sps.diags(keep_c)))
        X.eliminate_zeros()
    X.sort_indices()
    return X


def engine_for(X, k, err_mode="auto"):
    e = pymf_b200.Engine(X.shape[0], X.shape[1], k)
    e.set_err_mode(err_mode)
    e.upload_x_csc(X.indptr, X.indices, X.data)
    assert e.active_path == "sparse"
    return e


def init(d, n, k, seed):
    rng = np.random.RandomState(seed)
    return rng.random_sample((d, k)), rng.random_sample((k, n))


SHAPES = [
    ("37x53", dict(d=37, n=53, density=0.2), 5),
    ("300x777_empty", dict(d=300, n=777, density=0.05, empty=True), 10),
    ("1000x4096", dict(d=1000, n=4096, density=0.01), 32),
    ("2048x8192_powerlaw", dict(d=2048, n=8192, density=0.02, power_law=True), 64),
    ("512x2000_k1", dict(d=512, n=2000, density=0.05), 1),
    ("512x2000_k128", dict(d=512, n=2000, density=0.05), 128),
    ("512x2000_k600", dict(d=512, n=2000, density=0.05), 600),
]


@pytest.mark.parametrize("panel", [None, 256])
@pytest.mark.parametrize("err_mode", ["trace", "direct"])
@pytest.mark.parametrize("name,shape,k", SHAPES, ids=[s[0] for s in SHAPES])
def test_per_iteration_parity_with_oracle(monkeypatch, name, shape, k, err_mode, panel):
    if panel is not None:
        monkeypatch.setenv("PYMFB_SPARSE_PANEL", str(panel))
    X = make_sparse(seed=len(name), **shape)
    Xd = X.toarray()
    W, H = init(X.shape[0], X.shape[1], k, 3)
    e = engine_for(X, k, err_mode)
    try:
        e.set_w(W); e.set_h(H)
        for i in range(10):
            f, _ = e.run(1, early_stop=False)
            O.update_w(Xd, W, H)
            O.update_h(Xd, W, H)
            fr = O.frobenius_norm(Xd, W, H)
            assert rel(e.get_w(), W) < TOL_WH, (name, i)
            assert rel(e.get_h(), H) < TOL_WH, (name, i)
            assert abs(f[0] - fr) < TOL_FERR * fr, (name, i, f[0], fr)
    finally:
        e.close()


@pytest.mark.parametrize("name,shape,k", [SHAPES[1], SHAPES[3]], ids=[SHAPES[1][0], SHAPES[3][0]])
def test_bnmf_and_snmf(name, shape, k):
    X = make_sparse(seed=len(name), **shape)
    W0, H0 = init(X.shape[0], X.shape[1], k, 4)
    m = pymf_b200.BNMF(X, num_bases=k, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=8)
    W, H = W0.copy(), H0.copy()
    fr = O.bnmf_factorize(X.toarray(), W, H, niter=8)
    assert rel(m.W, W) < TOL_WH and rel(m.H, H) < TOL_WH
    assert np.max(np.abs(m.ferr - fr) / fr) < TOL_FERR
    Xs = make_sparse(seed=len(name), signed=True, **shape)
    m = pymf_b200.SNMF(Xs, num_bases=k, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=8)
    H = H0.copy()
    W, fr = O.snmf_factorize(Xs.toarray(), W0.copy(), H, niter=8)
    assert rel(m.W, W) < TOL_WH and rel(m.H, H) < TOL_WH
    assert np.max(np.abs(m.ferr - fr) / fr) < TOL_FERR


# ---- float64 scipy.sparse restatement of pymf/nmf.py:122-132 (the oracle's update_h / update_w without densifying) ----
def sp_update_h(X, W, H):
    H2 = np.dot(np.dot(W.T, W), H) + O.EPS_DENOM
    H *= np.asarray(X.T.dot(W)).T
    H /= H2


def sp_update_w(X, W, H):
    W2 = np.dot(np.dot(W, H), H.T) + O.EPS_DENOM
    W *= np.asarray(X.dot(H.T))
    W /= W2


def test_scipy_restatement_matches_oracle():
    X = make_sparse(300, 500, 0.03, 1)
    W, H = init(300, 500, 6, 2)
    Wo, Ho = W.copy(), H.copy()
    for _ in range(5):
        sp_update_w(X, W, H); sp_update_h(X, W, H)
        O.update_w(X.toarray(), Wo, Ho); O.update_h(X.toarray(), Wo, Ho)
    assert rel(W, Wo) < 1e-12 and rel(H, Ho) < 1e-12


def test_200_iteration_trajectory():
    X = make_sparse(4096, 16384, 0.01, 11)
    W, H = init(4096, 16384, 32, 12)
    e = engine_for(X, 32)
    try:
        e.set_w(W); e.set_h(H)
        at = 0
        for stop in (1, 50, 100, 200):
            e.run(stop - at, early_stop=False)
            for _ in range(stop - at):
                sp_update_w(X, W, H); sp_update_h(X, W, H)
            at = stop
            assert rel(e.get_w(), W) < TOL_WH, stop
            assert rel(e.get_h(), H) < TOL_WH, stop
    finally:
        e.close()


def test_sparse_path_matches_dense_path():
    X = make_sparse(1000, 4096, 0.02, 21)
    W, H = init(1000, 4096, 32, 22)
    out = []
    for sparse in (True, False):
        e = pymf_b200.Engine(1000, 4096, 32)
        try:
            if sparse:
                e.upload_x_csc(X.indptr, X.indices, X.data)
            else:
                e.upload_x(X.toarray().astype(np.float32))
            e.set_w(W); e.set_h(H)
            f, _ = e.run(20, early_stop=False)
            out.append((e.get_w(), e.get_h(), f))
        finally:
            e.close()
    assert rel(out[0][0], out[1][0]) < TOL_WH and rel(out[0][1], out[1][1]) < TOL_WH
    assert np.max(np.abs(out[0][2] - out[1][2]) / out[1][2]) < TOL_FERR


def test_runs_are_bit_identical():
    X = make_sparse(2048, 8192, 0.02, 31, power_law=True)
    W, H = init(2048, 8192, 64, 32)
    out = []
    for _ in range(2):
        e = engine_for(X, 64)
        try:
            e.set_w(W); e.set_h(H)
            f, _ = e.run(6, early_stop=False)
            out.append((e.get_w(np.float32), e.get_h(np.float32), f))
        finally:
            e.close()
    for a, b in zip(out[0], out[1]):
        np.testing.assert_array_equal(a, b)


def test_early_stop_follows_the_reference_rule():
    X = make_sparse(60, 400, 0.1, 41)
    W, H = init(60, 400, 3, 42)
    e = engine_for(X, 3)
    try:
        e.set_w(W); e.set_h(H)
        ferr, done = e.run(100000, early_stop=True)
        assert 3 <= done < 100000 and len(ferr) == done - 1
    finally:
        e.close()
    e = engine_for(X, 3)                      # the same run without the stop: the rule fires first at done - 1
    try:
        e.set_w(W); e.set_h(H)
        full, _ = e.run(done, early_stop=False)
    finally:
        e.close()
    np.testing.assert_array_equal(full[:done - 1], ferr)
    derr = np.abs(np.diff(full)) / 400
    fired = [i for i in range(2, done) if derr[i - 1] < O.EPS_CONV]
    assert fired and fired[0] == done - 1


def test_graph_replay_is_bit_identical():
    X = make_sparse(300, 777, 0.05, 51)
    W, H = init(300, 777, 10, 52)
    out = []
    for mode in ("auto", "off"):
        e = engine_for(X, 10)
        try:
            e.set_graph_mode(mode)
            e.set_w(W); e.set_h(H)
            f, _ = e.run(12, early_stop=False)
            out.append((e.get_w(np.float32), e.get_h(np.float32), f, e.graph_replays))
        finally:
            e.close()
    assert out[0][3] > 0 and out[1][3] == 0
    for a, b in zip(out[0][:3], out[1][:3]):
        np.testing.assert_array_equal(a, b)


def test_exact_fit_hands_over_to_the_direct_residual():
    """X = W* H* block-diagonal (sparse); from W*, H* the trace identity cancels, the context switches to the direct
    residual, which resolves the fp32 floor of the fit instead of the identity's sqrt(2e-7) ||X||."""
    d, n, k, nb = 2048, 8192, 8, 4
    rng = np.random.RandomState(61)
    Ws, Hs = np.zeros((d, k)), np.zeros((k, n))
    for b in range(nb):
        Ws[b * d // nb:(b + 1) * d // nb, 2 * b:2 * b + 2] = rng.uniform(0.5, 1.0, (d // nb, 2))
        Hs[2 * b:2 * b + 2, b * n // nb:(b + 1) * n // nb] = rng.uniform(0.5, 1.0, (2, n // nb))
    Ws, Hs = Ws.astype(np.float32).astype(np.float64), Hs.astype(np.float32).astype(np.float64)
    X = sps.csc_matrix(Ws.dot(Hs))
    e = engine_for(X, k)                      # auto: d * n * kp > 2^28 starts on the trace identity
    try:
        e.set_w(Ws); e.set_h(Hs)
        e.run(3, early_stop=False)
        f = e.frobenius()
    finally:
        e.close()
    xn = np.sqrt(X.multiply(X).sum())
    # the identity's value here is rounding noise of ~sqrt(2e-7) ||X|| or a clamped 0; the direct residual is the fp32
    # floor of W H, positive and far below that
    assert 0.0 < f < 1e-5 * xn, (f, xn)


def test_large_shape_against_scipy_restatement():
    d, n, k = 16384, 131072, 64
    X = make_sparse(d, n, 0.005, 71)
    W, H = init(d, n, k, 72)
    e = engine_for(X, k)
    try:
        e.set_w(W); e.set_h(H)
        e.run(3, early_stop=False)
        for _ in range(3):
            sp_update_w(X, W, H); sp_update_h(X, W, H)
        assert rel(e.get_w(), W) < TOL_WH and rel(e.get_h(), H) < TOL_WH
    finally:
        e.close()


def _csc_ok():
    X = make_sparse(20, 30, 0.2, 81)
    return X.indptr.astype(np.int64), X.indices.astype(np.int32), X.data


@pytest.mark.parametrize("rule", ["start", "decreasing", "end", "row_negative", "row_too_big", "row_order", "duplicate"])
def test_malformed_csc_is_rejected(rule):
    indptr, indices, vals = [a.copy() for a in _csc_ok()]
    c = int(np.argmax(np.diff(indptr) >= 2))              # a column with at least two entries
    a = int(indptr[c])
    if rule == "start":
        indptr[0] = 1
    elif rule == "decreasing":
        indptr[c + 1] = indptr[c] - 1
    elif rule == "end":
        indptr[-1] -= 1
    elif rule == "row_negative":
        indices[a] = -1
    elif rule == "row_too_big":
        indices[a] = 20
    elif rule == "row_order":
        indices[a], indices[a + 1] = indices[a + 1], indices[a]
    else:
        indices[a + 1] = indices[a]
    e = pymf_b200.Engine(20, 30, 3)
    try:
        with pytest.raises(pymf_b200._lib.PymfbError, match="malformed CSC"):
            e.upload_x_csc(indptr, indices, vals)
        e.upload_x_csc(*_csc_ok())                         # the context stays usable
        assert e.active_path == "sparse"
    finally:
        e.close()


def test_path_option_and_nndsvd_are_refused_and_dense_upload_switches_back():
    X = make_sparse(64, 256, 0.1, 91)
    e = engine_for(X, 4)
    try:
        for p in ("simt", "tc"):
            with pytest.raises(pymf_b200._lib.PymfbError):
                e.set_path(p)
        e.set_w(np.ones((64, 4))); e.set_h(np.ones((4, 256)))
        with pytest.raises(pymf_b200._lib.PymfbError):
            e.nndsvd()
        e.upload_x(X.toarray())
        assert e.active_path in ("simt", "tc")
        e.run(2)
    finally:
        e.close()


WORKER = r'''
import os, sys, numpy as np
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
import pymf_b200
from tests.test_sparse import make_sparse
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
X = make_sparse(%(d)d, %(n)d, 0.03, 101)
bounds = [int(round(%(n)d * r / float(world))) for r in range(world + 1)]
lo, hi = bounds[rank], bounds[rank + 1]
np.random.seed(5)
m = pymf_b200.NMF(X[:, lo:hi], num_bases=%(k)d, process_group=True, device=rank, sparse=True)
m.factorize(niter=%(niter)d)
np.savez(os.path.join(%(out)r, "r%%d.npz" %% rank), W=m.W, H=m.H, ferr=m.ferr, lo=lo, hi=hi)
dist.destroy_process_group()
'''


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def test_two_gpus_match_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d, n, k, niter = 700, 3000, 16, 8
    script = tmp_path / "worker.py"
    script.write_text(WORKER % dict(root=ROOT, d=d, n=n, k=k, niter=niter, out=str(tmp_path)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    X = make_sparse(d, n, 0.03, 101)
    np.random.seed(5)
    m = pymf_b200.NMF(X, num_bases=k, sparse=True)
    m.factorize(niter=niter)
    parts = [np.load(str(tmp_path / ("r%d.npz" % r_))) for r_ in range(2)]
    np.testing.assert_array_equal(parts[0]["W"], parts[1]["W"])
    for p in parts:
        assert rel(p["W"], m.W) < TOL_WH
        assert rel(p["H"], m.H[:, int(p["lo"]):int(p["hi"])]) < TOL_WH
        assert np.max(np.abs(p["ferr"] - m.ferr) / m.ferr) < TOL_FERR
