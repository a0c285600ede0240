"""NMF / BNMF / SNMF on torch sparse tensors (pymfb_upload_x_sparse_device): the canonical CSC built on the device gives
bit-identical results to the scipy route on the reference canonicalisation of tests/test_sparse_torch_host.py, every
validation rule is refused without a fault, and the upload leaves no device memory behind.  Needs a B200: `-m gpu`."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import pymf_b200
from oracle import nmf_oracle as O
from tests.test_sparse import TOL_FERR, TOL_WH, _free_port, init, rel
from tests.test_sparse_torch_host import as_layout, messy_coo, reference_of

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = torch.device("cuda", 0)


def messy(d, n, density, seed, dtype=torch.float32, empty=True):
    """messy_coo with explicit zeros and (empty=True) no entry in every 7th row and every 5th column, on the GPU."""
    t = messy_coo(d, n, density, seed, dup=0.05, zeros=3, dtype=dtype)
    idx, vals = t._indices(), t._values()
    if empty:
        keep = (idx[0] % 7 != 0) & (idx[1] % 5 != 0)
        idx, vals = idx[:, keep], vals[keep]
    return torch.sparse_coo_tensor(idx, vals, (d, n), check_invariants=False).to(CUDA)


def on_cuda(t):
    """The same tensor with its raw arrays on the GPU (no conversion, no coalescing)."""
    if t.layout == torch.sparse_coo:
        return torch.sparse_coo_tensor(t._indices().to(CUDA), t._values().to(CUDA), t.shape, check_invariants=False)
    if t.layout == torch.sparse_csr:
        return torch.sparse_csr_tensor(t.crow_indices().to(CUDA), t.col_indices().to(CUDA), t.values().to(CUDA),
                                       t.shape, check_invariants=False)
    return torch.sparse_csc_tensor(t.ccol_indices().to(CUDA), t.row_indices().to(CUDA), t.values().to(CUDA), t.shape,
                                   check_invariants=False)


def factorize(data, k, W0, H0, niter, cls="NMF", err_mode="auto"):
    m = getattr(pymf_b200, cls)(data, num_bases=k, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    m._ensure_engine().set_err_mode(err_mode)
    assert m._engine.active_path == "sparse"
    m.factorize(niter=niter)
    out = (m.W.copy(), m.H.copy(), m.ferr.copy())
    m._engine.close()
    return out


def assert_same_as_scipy_route(t, k, niter=6, cls="NMF", err_mode="auto", seed=3):
    ref = reference_of(t)
    W0, H0 = init(t.shape[0], t.shape[1], k, seed)
    got = factorize(t, k, W0, H0, niter, cls, err_mode)
    want = factorize(ref, k, W0, H0, niter, cls, err_mode)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)
    return got


def _combos():
    out = []
    for layout in ("coo", "csr", "csc"):
        for idt in ([torch.int64] if layout == "coo" else [torch.int32, torch.int64]):
            for vdt in (torch.float16, torch.bfloat16, torch.float32, torch.float64):
                out.append((layout, idt, vdt))
    return out


def _as(layout, coo, idt):
    if layout == "coo":
        return coo
    return on_cuda(as_layout(coo.cpu(), layout, idt, shuffle_rows=(layout == "csc"), seed=4))


@pytest.mark.parametrize("err_mode", ["trace", "direct"])
@pytest.mark.parametrize("layout,index_dtype,value_dtype", _combos(), ids=lambda v: str(v).replace("torch.", ""))
def test_bit_identical_to_the_scipy_route(monkeypatch, layout, index_dtype, value_dtype, err_mode):
    monkeypatch.setenv("PYMFB_SPARSE_PANEL", "64")
    t = _as(layout, messy(300, 777, 0.05, 11, dtype=value_dtype), index_dtype)
    assert_same_as_scipy_route(t, 10, err_mode=err_mode)


@pytest.mark.parametrize("case", ["nnz0", "d1", "n1", "all_duplicates"])
def test_edge_shapes(case):
    if case == "nnz0":
        t = torch.sparse_coo_tensor(torch.zeros(2, 0, dtype=torch.int64), torch.zeros(0), (40, 60)).to(CUDA)
    elif case == "d1":
        t = messy(1, 300, 0.3, 12, empty=False)
    elif case == "n1":
        t = messy(300, 1, 0.3, 13, empty=False)
    else:                                       # one entry repeated many times, in a long run
        idx = torch.tensor([[3] * 5000 + [1], [2] * 5000 + [0]])
        t = torch.sparse_coo_tensor(idx, torch.rand(5001, dtype=torch.float64), (8, 9), check_invariants=False).to(CUDA)
    for layout in ("coo", "csr", "csc"):
        assert_same_as_scipy_route(_as(layout, t, torch.int32), 3, niter=4)


@pytest.mark.parametrize("cls", ["BNMF", "SNMF"])
def test_bnmf_and_snmf(monkeypatch, cls):
    monkeypatch.setenv("PYMFB_SPARSE_PANEL", "128")
    t = messy(512, 2000, 0.05, 14)
    if cls == "SNMF":                           # signed data
        t = torch.sparse_coo_tensor(t._indices(), t._values() - 0.5, t.shape, check_invariants=False)
    for err_mode in ("trace", "direct"):
        assert_same_as_scipy_route(t, 32, niter=8, cls=cls, err_mode=err_mode)


def test_accuracy_against_the_oracle():
    t = messy(1000, 4096, 0.01, 15)
    Xd = reference_of(t).astype(np.float64).toarray()
    W, H = init(1000, 4096, 32, 16)
    m = pymf_b200.NMF(t, num_bases=32, sparse=True)
    m.W, m.H = W.copy(), H.copy()
    for i in range(10):
        m.factorize(niter=1)
        O.update_w(Xd, W, H)
        O.update_h(Xd, W, H)
        fr = O.frobenius_norm(Xd, W, H)
        assert rel(m.W, W) < TOL_WH and rel(m.H, H) < TOL_WH, i
        assert abs(m.ferr[0] - fr) < TOL_FERR * fr, (i, m.ferr[0], fr)


def test_cpu_tensor_and_repeated_uploads_are_bit_identical():
    t = messy(700, 3000, 0.03, 17)
    W0, H0 = init(700, 3000, 16, 18)
    a = factorize(t, 16, W0, H0, 5)
    b = factorize(t.cpu(), 16, W0, H0, 5)
    m = pymf_b200.NMF(t, num_bases=16, sparse=True)
    for _ in range(2):                           # the second run uploads the same uncoalesced tensor again
        m.data = t
        m.W, m.H = W0.copy(), H0.copy()
        m.factorize(niter=5)
        for x, y in zip(a, (m.W, m.H, m.ferr)):
            np.testing.assert_array_equal(x, y)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)


def _bad(layout, rule):
    """A 20 x 30 tensor (raw arrays on the GPU, invariants unchecked) that breaks `rule`; the expected message."""
    good = reference_of(messy(20, 30, 0.2, 19, empty=False))
    coo = good.tocoo()
    if layout == "coo":
        r, c = coo.row.astype(np.int64), coo.col.astype(np.int64)
        if rule == "row_negative":
            r[3] = -1
        elif rule == "row_too_big":
            r[3] = 20
        elif rule == "col_negative":
            c[3] = -1
        else:
            c[3] = 30
        t = torch.sparse_coo_tensor(torch.from_numpy(np.stack([r, c])).to(CUDA), torch.from_numpy(coo.data).to(CUDA),
                                    (20, 30), check_invariants=False)
        return t, "row index outside" if rule.startswith("row") else "column index outside"
    m = good.tocsr() if layout == "csr" else good
    ptr, idx = m.indptr.astype(np.int64).copy(), m.indices.astype(np.int64).copy()
    bound = 30 if layout == "csr" else 20
    o = int(np.argmax(np.diff(ptr) >= 2))
    if rule == "start":
        ptr[0] = 1
        msg = r"pointers\[0\] != 0"
    elif rule == "end":
        ptr[-1] -= 1
        msg = r"pointers\[last\] != nnz"
    elif rule == "decreasing":
        ptr[o + 1] = ptr[o] - 1
        msg = "pointers decrease"
    elif rule == "index_negative":
        idx[ptr[o]] = -1
        msg = "column index outside" if layout == "csr" else "row index outside"
    else:
        idx[ptr[o]] = bound
        msg = "column index outside" if layout == "csr" else "row index outside"
    p, i, v = (torch.from_numpy(x).to(CUDA) for x in (ptr, idx, m.data))
    make = torch.sparse_csr_tensor if layout == "csr" else torch.sparse_csc_tensor
    return make(p, i, v, (20, 30), check_invariants=False), msg


RULES = ([("coo", r) for r in ("row_negative", "row_too_big", "col_negative", "col_too_big")] +
         [(lay, r) for lay in ("csr", "csc") for r in ("start", "end", "decreasing", "index_negative", "index_too_big")])


@pytest.mark.parametrize("layout,rule", RULES, ids=["%s-%s" % r for r in RULES])
def test_malformed_input_is_refused_and_the_previous_x_stays(layout, rule):
    good = messy(20, 30, 0.2, 20, empty=False)
    W0, H0 = init(20, 30, 3, 21)
    want = factorize(good, 3, W0, H0, 4)
    m = pymf_b200.NMF(good, num_bases=3, sparse=True)
    m.W, m.H = W0.copy(), H0.copy()
    eng = m._ensure_engine()
    bad, msg = _bad(layout, rule)
    m.data = bad
    with pytest.raises(pymf_b200.PymfbError, match=msg):
        m.factorize(niter=1)
    assert eng.active_path == "sparse"
    eng.set_w(W0); eng.set_h(H0)                                    # still the previous X
    f, _ = eng.run(4)
    np.testing.assert_array_equal(f, want[2])
    np.testing.assert_array_equal(eng.get_w(), want[0])
    m.data = messy(20, 30, 0.3, 22, empty=False)                    # a good upload works
    m.factorize(niter=2)
    assert np.all(np.isfinite(m.ferr))


def test_inputs_untouched_switching_and_no_memory_left_behind():
    t = messy(2048, 8192, 0.02, 23, dtype=torch.float16)
    before = [x.clone() for x in (t._indices(), t._values())]
    ref = reference_of(t)
    W0, H0 = init(2048, 8192, 32, 24)
    m = pymf_b200.NMF(ref, num_bases=32, sparse=True)           # scipy -> torch -> scipy on one object
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=2)
    m.data = t
    m.factorize(niter=2)
    for x, y in zip(before, (t._indices(), t._values())):
        assert x.dtype == y.dtype and torch.equal(x, y)
    m.data = ref
    m.factorize(niter=2)
    eng = m._engine                                              # and dense data on the same context
    eng.upload_x(ref.toarray())
    assert eng.active_path in ("simt", "tc")
    eng.upload_x_sparse_device("coo", t._indices()[0], t._indices()[1], t._values().float())
    assert eng.active_path == "sparse"
    eng.set_w(W0); eng.set_h(H0)
    f, _ = eng.run(2)
    assert np.all(np.isfinite(f))
    eng.close()

    def free_after(data):
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        mm = pymf_b200.NMF(data, num_bases=32, sparse=True)
        mm.W, mm.H = W0.copy(), H0.copy()
        mm.factorize(niter=1)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        free = torch.cuda.mem_get_info(0)[0]
        mm._engine.close()
        return free

    f_scipy = free_after(ref)
    f_torch = free_after(t)
    assert abs(f_torch - f_scipy) < (4 << 20), (f_torch, f_scipy)


def test_large_uncoalesced_coo():
    d, n, k = 16384, 131072, 64
    t = messy_coo(d, n, 0.005, 25, dup=0.01).to(CUDA)
    assert_same_as_scipy_route(t, k, niter=3)


def test_wrong_device_is_refused():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    t = messy(20, 30, 0.2, 26).to(torch.device("cuda", 1))
    with pytest.raises(ValueError):
        pymf_b200.NMF(t, num_bases=3, sparse=True, device=0)
    m = pymf_b200.NMF(t, num_bases=3, sparse=True, device=1)
    m.factorize(niter=2)


WORKER = r'''
import os, sys, numpy as np
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
import pymf_b200
from tests.test_sparse_torch_host import messy_coo
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
t = messy_coo(%(d)d, %(n)d, 0.03, 101, dup=0.02)
bounds = [int(round(%(n)d * r / float(world))) for r in range(world + 1)]
lo, hi = bounds[rank], bounds[rank + 1]
idx, vals = t._indices(), t._values()
keep = (idx[1] >= lo) & (idx[1] < hi)
dev = torch.device("cuda", rank)
blk = torch.sparse_coo_tensor(torch.stack([idx[0][keep], idx[1][keep] - lo]).to(dev), vals[keep].to(dev),
                              (%(d)d, hi - lo), check_invariants=False)
other = blk.to(torch.device("cuda", 1 - rank))
try:
    pymf_b200.NMF(other, num_bases=%(k)d, process_group=True, device=rank, sparse=True)
    raise SystemExit("a tensor on another device was accepted")
except ValueError:
    pass
np.random.seed(5)
m = pymf_b200.NMF(blk, num_bases=%(k)d, process_group=True, device=rank, sparse=True)
m.factorize(niter=%(niter)d)
np.savez(os.path.join(%(out)r, "r%%d.npz" %% rank), W=m.W, H=m.H, ferr=m.ferr, lo=lo, hi=hi)
dist.destroy_process_group()
'''


def test_two_gpus_match_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    d, n, k, niter = 700, 3000, 16, 8
    script = tmp_path / "worker.py"
    script.write_text(WORKER % dict(root=ROOT, d=d, n=n, k=k, niter=niter, out=str(tmp_path)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    np.random.seed(5)
    m = pymf_b200.NMF(messy_coo(d, n, 0.03, 101, dup=0.02).to(CUDA), num_bases=k, sparse=True)
    m.factorize(niter=niter)
    parts = [np.load(str(tmp_path / ("r%d.npz" % r_))) for r_ in range(2)]
    np.testing.assert_array_equal(parts[0]["W"], parts[1]["W"])
    for p in parts:
        assert rel(p["W"], m.W) < TOL_WH
        assert rel(p["H"], m.H[:, int(p["lo"]):int(p["hi"])]) < TOL_WH
        assert np.max(np.abs(p["ferr"] - m.ferr) / m.ferr) < TOL_FERR
