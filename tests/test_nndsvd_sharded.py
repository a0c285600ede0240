"""NNDSVD on column-sharded data and with its passes over X on the tensor cores (pymfb_nndsvd, kernels_svd.cuh,
kernels_tc.cuh).  CPU: the planted shapes meet the preconditions of comparing an exact with an iterative SVD, and the
host layer of a sharded NNDSVD runs over gloo with an oracle-backed engine double.  GPU: two ranks on the CUDA-core
passes against the golden cases, one GPU and two ranks on the tensor-core passes against the closed-form oracle."""
import functools
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import cases, nmf_oracle as O
from tests._fake_engine import FakeEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL_WH = 1e-4
TOL_SIGMA = 1e-5
TOL_FERR = 1e-3
SWEEP_CAP = 100


def rel(a, b):
    b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


def planted(seed, d, n, k):
    """X = U diag(s) V^T + noise with m = k + 10 exact singular triplets: every u_i / v_i lives on its own random group
    of rows / columns (exactly orthogonal), is positive on 70 % of it for even i and 30 % for odd i (the sign choice of
    the second SVD is never close to a tie, and both branches occur), s_i = 100 * 0.985^i (1.5 % gaps), plus uniform
    zero-mean noise of amplitude 2e-3 (its singular values stay below 0.1, s_m > 14)."""
    rng = np.random.RandomState(seed)
    m = k + 10

    def factor(length):
        F = np.zeros((length, m))
        for i, g in enumerate(np.array_split(rng.permutation(length), m)):
            npos = int(round((0.7 if i % 2 == 0 else 0.3) * len(g)))
            sign = np.where(np.arange(len(g)) < npos, 1.0, -1.0)
            v = rng.uniform(0.5, 1.5, len(g)) * sign
            F[g, i] = v / np.linalg.norm(v)
        return F

    U, V = factor(d), factor(n)
    s = 100.0 * 0.985 ** np.arange(m)
    return (U * s).dot(V.T) + 2e-3 * (rng.random_sample((d, n)) - 0.5)


def closed_form(X, k):
    """NNDSVD of X from ONE exact SVD: the reference's second SVD of max(0, s u v^T) in closed form (the construction
    test_nndsvd.test_closed_form_of_the_second_svd pins to the reference).  Returns W, H, sigma, U, V."""
    U, S, V = O.svd_dense(X)
    W = np.zeros((X.shape[0], k)); H = np.zeros((k, X.shape[1]))
    W[:, 0] = np.sqrt(S[0, 0]) * np.abs(U[:, 0]); H[0] = np.sqrt(S[0, 0]) * np.abs(V[0])
    for i in range(1, k):
        u, v, s = U[:, i], V[i], S[i, i]
        up, un, vp, vn = np.maximum(u, 0), np.maximum(-u, 0), np.maximum(v, 0), np.maximum(-v, 0)
        a, b = (up, vp) if np.linalg.norm(up) * np.linalg.norm(vp) >= np.linalg.norm(un) * np.linalg.norm(vn) else (un, vn)
        s2 = s * np.linalg.norm(a) * np.linalg.norm(b)
        W[:, i] = np.sqrt(s2) * a / np.linalg.norm(a)
        H[i] = np.sqrt(s2) * b / np.linalg.norm(b)
    return W, H, np.diag(S)[:k + 1].copy(), U, V


# d * n > 2^24 (the tensor-core default), d not a multiple of 128, n odd; k covers the widths b' = 32, 64, 128, 256
PLANTED_TC = {"k16": (61, 1000, 16801, 16), "k40": (62, 1000, 16801, 40),
              "k100": (63, 1000, 16801, 100), "k120": (64, 1000, 16801, 120)}
PLANTED_2RANK = (65, 1000, 33603, 40)          # two shards of 16801 / 16802 columns: each above 2^24 elements


@functools.lru_cache(maxsize=None)
def planted_case(seed, d, n, k):
    X = planted(seed, d, n, k)
    W, H, sig, U, V = closed_form(X, k)
    return X, W, H, sig, U, V


@pytest.mark.parametrize("name", sorted(PLANTED_TC) + ["two_rank"])
def test_planted_shapes_are_comparable(name):
    """An exact and an iterative SVD agree on singular vectors (and on the sign choice of the second SVD) only where the
    leading k + 1 singular values are apart and |u+||v+| differs from |u-||v-|: both by at least 1 % here."""
    seed, d, n, k = PLANTED_TC[name] if name in PLANTED_TC else PLANTED_2RANK
    X, W, H, sig, U, V = planted_case(seed, d, n, k)
    assert d * n > 2 ** 24 and d % 128 != 0 and n % 2 == 1
    assert np.min((sig[:-1] - sig[1:]) / sig[:-1]) >= 0.01
    for i in range(1, k):
        u, v = U[:, i], V[i]
        a = np.linalg.norm(np.maximum(u, 0)) * np.linalg.norm(np.maximum(v, 0))
        b = np.linalg.norm(np.maximum(-u, 0)) * np.linalg.norm(np.maximum(-v, 0))
        assert abs(a - b) / max(a, b) >= 0.01, (i, a, b)
    assert W.min() >= 0 and H.min() >= 0


# ---------------------------------------------------------------------------------------------------------------
# CPU: the sharded host path over gloo
# ---------------------------------------------------------------------------------------------------------------
class NndsvdFakeEngine(FakeEngine):
    """FakeEngine plus nndsvd(): the sharded data flow with an exact SVD - X X^T summed over the ranks, V's columns
    from the local X, the |v+| / |v-| norms summed over the ranks, W replicated, H local."""

    def set_nndsvd_path(self, path):
        pass

    def nndsvd(self, max_iter=0, tol=0.0, extra_iter=-1):
        k = self.k
        vals, U = np.linalg.eigh(self._allreduce(self.X.dot(self.X.T)))
        idx = np.argsort(vals)[::-1][:k]
        s, U = np.sqrt(vals[idx]), U[:, idx]
        V = U.T.dot(self.X) / s[:, None]
        vn = self._allreduce(np.array([[np.sum(np.maximum(V[i], 0) ** 2), np.sum(np.maximum(-V[i], 0) ** 2)]
                                       for i in range(k)]))
        W, H = np.zeros((self.d, k)), np.zeros((k, self.n_local))
        W[:, 0] = np.sqrt(s[0]) * np.abs(U[:, 0]); H[0] = np.sqrt(s[0]) * np.abs(V[0])
        for i in range(1, k):
            up, un = np.maximum(U[:, i], 0), np.maximum(-U[:, i], 0)
            nup, nun, nvp, nvn = np.linalg.norm(up), np.linalg.norm(un), np.sqrt(vn[i, 0]), np.sqrt(vn[i, 1])
            pos = nup * nvp >= nun * nvn
            a, b, na, nb = (up, np.maximum(V[i], 0), nup, nvp) if pos else (un, np.maximum(-V[i], 0), nun, nvn)
            s2 = s[i] * na * nb
            W[:, i] = np.sqrt(s2) * a / na
            H[i] = np.sqrt(s2) * b / nb
        self.W, self.H = W, H
        self.nndsvd_path, self.nndsvd_change = "oracle", 0.0
        return s, 1


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _gloo_worker(rank, world, port, out):
    import torch.distributed as dist
    import pymf_b200
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        pymf_b200.NMF._engine_factory = NndsvdFakeEngine
        X = planted(71, 37, 101, 4)
        lo, hi = (0, 30) if rank == 0 else (30, 101)
        m = pymf_b200.NNDSVD(X[:, lo:hi], num_bases=4, process_group=True)
        m.factorize()
        f = pymf_b200.NMF(X[:, lo:hi], num_bases=4, process_group=True)
        f.W, f.H = m.W.copy(), m.H.copy()            # NMF updates an assigned array in place
        f.factorize(niter=5)
        np.savez(os.path.join(out, "n%d.npz" % rank), W=m.W, H=m.H, ferr=m.ferr, sigma=m.singular_values,
                 Wn=f.W, Hn=f.H, ferrn=f.ferr, lo=lo, hi=hi)
    finally:
        dist.destroy_process_group()


def test_sharded_nndsvd_host_path_over_gloo(tmp_path):
    import torch.multiprocessing as mp
    mp.spawn(_gloo_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    X = planted(71, 37, 101, 4)
    W, H, sig, _, _ = closed_form(X, 4)
    ferr = O.frobenius_norm(X, W, H)
    p0, p1 = [np.load(os.path.join(str(tmp_path), "n%d.npz" % r)) for r in range(2)]
    np.testing.assert_array_equal(p0["W"], p1["W"])
    np.testing.assert_array_equal(p0["sigma"], p1["sigma"])
    for p in (p0, p1):
        lo, hi = int(p["lo"]), int(p["hi"])
        assert p["H"].shape == (4, hi - lo)
        np.testing.assert_allclose(p["W"], W, rtol=1e-8, atol=1e-12)
        np.testing.assert_allclose(p["H"], H[:, lo:hi], rtol=1e-8, atol=1e-12)
        np.testing.assert_allclose(p["sigma"], sig[:4], rtol=1e-10)
        np.testing.assert_allclose(p["ferr"], [ferr], rtol=1e-9)         # the global error
    Wr, Hr = W.copy(), H.copy()
    fr = O.factorize(X, Wr, Hr, niter=5)
    np.testing.assert_array_equal(p0["Wn"], p1["Wn"])
    for p in (p0, p1):
        np.testing.assert_allclose(p["Wn"], Wr, rtol=1e-8, atol=1e-12)
        np.testing.assert_allclose(p["Hn"], Hr[:, int(p["lo"]):int(p["hi"])], rtol=1e-8, atol=1e-12)
        np.testing.assert_allclose(p["ferrn"], fr, rtol=1e-9)


# ---------------------------------------------------------------------------------------------------------------
# GPU, one device: the tensor-core passes
# ---------------------------------------------------------------------------------------------------------------
def _check_against(m, W, H, sig, X, k):
    assert np.max(np.abs(m.singular_values - sig[:k]) / sig[:k]) < TOL_SIGMA
    rw, rh = rel(m.W, W), rel(m.H, H)
    assert rw < TOL_WH and rh < TOL_WH, (rw, rh)
    f = O.frobenius_norm(X, W, H)
    assert abs(m.ferr[0] - f) / f < TOL_FERR
    assert m.W.min() >= 0 and m.H.min() >= 0
    return rw, rh


@pytest.mark.gpu
def test_gpu_nndsvd_tc_golden_case(golden_dir):
    import pymf_b200
    c = cases.NNDSVD_CASES["nndsvd_tc"]
    g = np.load(os.path.join(golden_dir, "nndsvd_tc.npz"))
    X = cases.build_nndsvd("nndsvd_tc")
    m = pymf_b200.NNDSVD(X, num_bases=c["k"], path="tc")
    m.factorize()
    assert m.svd_path == "tc" and m.svd_sweeps < SWEEP_CAP
    assert np.max(np.abs(m.singular_values - g["sigma"][:c["k"]]) / g["sigma"][:c["k"]]) < TOL_SIGMA
    assert rel(m.W, g["W"]) < TOL_WH and rel(m.H, g["H"]) < TOL_WH
    assert abs(m.ferr[0] - g["ferr"][0]) / g["ferr"][0] < TOL_FERR


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PLANTED_TC))
def test_gpu_nndsvd_tc_planted(name):
    import pymf_b200
    seed, d, n, k = PLANTED_TC[name]
    X, W, H, sig, _, _ = planted_case(seed, d, n, k)
    if k > 102:         # one GPU, b' = 256 > b: the default keeps the CUDA-core passes below d * n = 2^32
        m = pymf_b200.NNDSVD(X, num_bases=k)
        m.factorize()
        assert m.svd_path == "simt"
        _check_against(m, W, H, sig, X, k)
    m = pymf_b200.NNDSVD(X, num_bases=k, path="tc" if k > 102 else None)
    m.factorize()
    assert m.svd_path == "tc"                      # the default beyond d * n = 2^24
    assert m.svd_sweeps < SWEEP_CAP, m.svd_sweeps
    rw, rh = _check_against(m, W, H, sig, X, k)
    print(name, "sweeps", m.svd_sweeps, "change %.2e" % m._engine.nndsvd_change, "rel W %.2e rel H %.2e" % (rw, rh))


@pytest.mark.gpu
def test_gpu_nndsvd_tc_layouts_and_reruns_are_bit_identical():
    """A host numpy source (context-owned copy, panel-major) and a CUDA tensor bound in place (row-major) give the same
    bits, and so do two runs."""
    import torch
    import pymf_b200
    seed, d, n, k = PLANTED_TC["k40"]
    X = planted_case(seed, d, n, k)[0].astype(np.float32)
    runs = []
    for src in (X, X, torch.from_numpy(X).cuda()):
        m = pymf_b200.NNDSVD(src, num_bases=k)
        m.factorize()
        assert m.svd_path == "tc"
        runs.append((m.W.copy(), m.H.copy(), m.singular_values.copy(), m.svd_sweeps))
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            np.testing.assert_array_equal(a, b)


# ---------------------------------------------------------------------------------------------------------------
# GPU, two ranks over NCCL
# ---------------------------------------------------------------------------------------------------------------
WORKER = r'''
import os, sys, numpy as np
sys.path.insert(0, %(root)r)
import torch, torch.distributed as dist
import pymf_b200
from oracle import cases
from tests.test_nndsvd_sharded import planted
rank = int(os.environ["RANK"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
out = {}
for name, X, k, split, path in %(jobs)s:
    X = cases.build_nndsvd(name) if X is None else planted(*X)
    lo, hi = (0, split) if rank == 0 else (split, X.shape[1])
    shard = np.ascontiguousarray(X[:, lo:hi])
    m = pymf_b200.NNDSVD(shard, num_bases=k, process_group=True, device=rank, path=path)
    m.factorize()
    res = dict(W=m.W, H=m.H, ferr=m.ferr, sigma=m.singular_values, sweeps=m.svd_sweeps, lo=lo, hi=hi)
    res["tc"] = m.svd_path == "tc"
    if path == "simt":
        f = pymf_b200.NMF(shard, num_bases=k, process_group=True, device=rank)
        f.W, f.H = m.W.copy(), m.H.copy()
        f.factorize(niter=10)
        res.update(Wn=f.W, Hn=f.H, ferrn=f.ferr)
    out.update({"%%s__%%s" %% (name, key): val for key, val in res.items()})
np.savez(os.path.join(%(out)r, "r%%d.npz" %% rank), **out)
dist.destroy_process_group()
'''


def _two_ranks(tmp_path, jobs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(WORKER % dict(root=ROOT, jobs=repr(jobs), out=str(tmp_path)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()), str(script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    return [np.load(str(tmp_path / ("r%d.npz" % i))) for i in range(2)]


def _job(parts, name):
    return [{key.split("__", 1)[1]: p[key] for key in p.files if key.startswith(name + "__")} for p in parts]


def _replicas_agree(r0, r1):
    np.testing.assert_array_equal(r0["W"], r1["W"])
    np.testing.assert_array_equal(r0["sigma"], r1["sigma"])
    assert int(r0["sweeps"]) == int(r1["sweeps"])
    np.testing.assert_array_equal(r0["ferr"], r1["ferr"])


# uneven splits; nndsvd_small's first shard (20 columns) is narrower than the subspace block b = 32
SPLITS = {"nndsvd_small": 20, "nndsvd_wide": 700, "nndsvd_tall": 250, "nndsvd_tc": 1500}


@pytest.mark.gpu
def test_two_gpus_nndsvd_simt_matches_golden(tmp_path, golden_dir):
    jobs = [(name, None, cases.NNDSVD_CASES[name]["k"], SPLITS[name], "simt") for name in sorted(SPLITS)]
    parts = _two_ranks(tmp_path, jobs)
    for name in sorted(SPLITS):
        k = cases.NNDSVD_CASES[name]["k"]
        g = np.load(os.path.join(golden_dir, "%s.npz" % name))
        r0, r1 = _job(parts, name)
        _replicas_agree(r0, r1)
        assert not r0["tc"] and not r1["tc"]
        H = np.concatenate([r0["H"], r1["H"]], axis=1)
        assert np.max(np.abs(r0["sigma"] - g["sigma"][:k]) / g["sigma"][:k]) < TOL_SIGMA, name
        assert rel(r0["W"], g["W"]) < TOL_WH and rel(H, g["H"]) < TOL_WH, (name, rel(r0["W"], g["W"]), rel(H, g["H"]))
        assert abs(r0["ferr"][0] - g["ferr"][0]) / g["ferr"][0] < TOL_FERR, name
        assert r0["W"].min() >= 0 and H.min() >= 0
        # the sharded NMF warm-started from them
        np.testing.assert_array_equal(r0["Wn"], r1["Wn"])
        Hn = np.concatenate([r0["Hn"], r1["Hn"]], axis=1)
        assert rel(r0["Wn"], g["W_nmf10"]) < TOL_WH and rel(Hn, g["H_nmf10"]) < TOL_WH, name
        assert np.max(np.abs(r0["ferrn"] - g["ferr_nmf10"]) / g["ferr_nmf10"]) < TOL_FERR, name


@pytest.mark.gpu
def test_two_gpus_nndsvd_tc_matches_oracle(tmp_path):
    seed, d, n, k = PLANTED_2RANK
    split = n // 2
    parts = _two_ranks(tmp_path, [("planted", (seed, d, n, k), k, split, None)])
    X, W, H, sig, _, _ = planted_case(seed, d, n, k)
    r0, r1 = _job(parts, "planted")
    _replicas_agree(r0, r1)
    assert r0["tc"] and r1["tc"] and int(r0["sweeps"]) < SWEEP_CAP
    Hc = np.concatenate([r0["H"], r1["H"]], axis=1)
    assert np.max(np.abs(r0["sigma"] - sig[:k]) / sig[:k]) < TOL_SIGMA
    assert rel(r0["W"], W) < TOL_WH and rel(Hc, H) < TOL_WH, (rel(r0["W"], W), rel(Hc, H))
    f = O.frobenius_norm(X, W, H)
    assert abs(r0["ferr"][0] - f) / f < TOL_FERR
