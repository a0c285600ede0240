"""Parity of the CUDA path (through the C ABI / pymf_b200.NMF) against the oracle and the
committed reference trajectories.  Needs a B200: run with `-m gpu`.

Tolerances are BASELINE.json's: per-iteration W/H within 1e-4 relative Frobenius error of the
reference's float64 path, ferr within 1e-3 relative."""
import os

import numpy as np
import pytest

import pymf_b200
from oracle import cases, nmf_oracle as O

pytestmark = pytest.mark.gpu

TOL_WH = 1e-4
TOL_FERR = 1e-3


def rel(a, b):
    b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(np.asarray(a, dtype=np.float64) - b) / np.linalg.norm(b)


def paths_for(d, n, k):
    """Kernel families that must serve this shape ('tc' only where it applies)."""
    e = pymf_b200.Engine(d, n, k)
    try:
        X = np.zeros((d, n), dtype=np.float32)
        e.upload_x(X)
        auto = e.active_path
    finally:
        e.close()
    return ["simt"] if auto == "simt" else ["simt", "tc"]


@pytest.mark.parametrize("err_mode", ["trace", "direct"])
@pytest.mark.parametrize("name", sorted(cases.CASES))
def test_trajectory_matches_reference_golden(name, err_mode, golden_dir):
    """Single-step the engine and compare every kept iteration with the reference's output."""
    c = cases.CASES[name]
    g = np.load(os.path.join(golden_dir, "traj_%s.npz" % name))
    X, W0, H0 = cases.build(name)
    for path in paths_for(c["d"], c["n"], c["k"]):
        e = pymf_b200.Engine(c["d"], c["n"], c["k"], path=path)
        try:
            e.set_err_mode(err_mode)
            e.upload_x(X)
            e.set_w(W0)
            e.set_h(H0)
            ferr = np.zeros(c["niter"])
            ws = c.get("w_stride", 1)              # large-d fixtures keep every ws-th row of W + the full norms
            for i in range(c["niter"]):
                f, done = e.run(1, early_stop=False)
                ferr[i] = f[0]
                if (i + 1) in c["keep"]:
                    W = e.get_w()
                    assert rel(W[::ws], g["W_%d" % (i + 1)]) < TOL_WH, (name, path, i)
                    assert abs(np.linalg.norm(W) - g["normW"][i]) / g["normW"][i] < TOL_WH, (name, path, i)
                    assert rel(e.get_h(), g["H_%d" % (i + 1)]) < TOL_WH, (name, path, i)
            assert np.max(np.abs(ferr - g["ferr"]) / g["ferr"]) < TOL_FERR, (name, path)
            # Frobenius norms of W/H per iteration are not available from single-stepping only at
            # kept iterations; the final ones are checked through get_w/get_h above.
        finally:
            e.close()


def test_200_iteration_trajectory_on_the_tensor_path(golden_dir):
    """north_star: per-iteration W/H within 1e-4 over cfg2's 200 iterations.  The cfg2 column prefix
    (4096 x 2048, k = 32) on the tcgen05 path, run as multi-iteration enqueues (the product's code path:
    one pymfb_run per segment, A/B carried across iterations) against the reference's trajectory: ferr
    at every one of the 200 iterations, W/H at iterations 1, 50, 100 and 200."""
    c = cases.CASES["cfg2_prefix_200"]
    g = np.load(os.path.join(golden_dir, "traj_cfg2_prefix_200.npz"))
    X, W0, H0 = cases.build("cfg2_prefix_200")
    e = pymf_b200.Engine(c["d"], c["n"], c["k"], path="tc")
    try:
        e.set_err_mode("trace")
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        ferr, at, worst = [], 0, 0.0
        for stop in c["keep"]:
            f, done = e.run(stop - at, early_stop=False)
            assert done == stop - at
            ferr.extend(f)
            at = stop
            rw, rh = rel(e.get_w(), g["W_%d" % stop]), rel(e.get_h(), g["H_%d" % stop])
            worst = max(worst, rw, rh)
            assert rw < TOL_WH and rh < TOL_WH, (stop, rw, rh)
        assert e.active_path == "tc"
        ferr = np.array(ferr)
        assert ferr.shape == (200,)
        assert np.max(np.abs(ferr - g["ferr"]) / g["ferr"]) < TOL_FERR
        print("200-iteration tc trajectory: worst rel W/H %.2e, worst rel ferr %.2e"
              % (worst, np.max(np.abs(ferr - g["ferr"]) / g["ferr"])))
    finally:
        e.close()


@pytest.mark.parametrize("shape", [(16384, 2048, 128), (32768, 1024, 64), (16384, 1280, 32)])
def test_large_d_matches_live_oracle(shape):
    """cfg3's (d = 16384, k = 128) and cfg5's (d = 32768, k = 64) contraction depth against the float64
    oracle run live on the FULL factors (the committed cfg3_d / cfg5_d fixtures hold every 8th row of W):
    512 / 1024 MMA stages per column tile, i.e. 16 / 32 TMEM segments drained with RN adds."""
    d, n, k = shape
    X = O.gen_matrix(d + 1, d, n)
    W0 = O.gen_matrix(d + 2, d, k).astype(np.float64)
    H0 = O.gen_matrix(d + 3, k, n).astype(np.float64)
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=3, early_stop=False)
    e = pymf_b200.Engine(d, n, k, path="tc")
    try:
        e.set_err_mode("trace")
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        f, done = e.run(3, early_stop=False)
        rw, rh = rel(e.get_w(), Wr), rel(e.get_h(), Hr)
        assert rw < TOL_WH and rh < TOL_WH, (rw, rh)
        assert np.max(np.abs(f - fr) / fr) < TOL_FERR
        e.set_err_mode("direct")
        assert abs(e.frobenius() - fr[-1]) / fr[-1] < TOL_FERR
    finally:
        e.close()


@pytest.mark.parametrize("name", ["cfg1", "ragged", "k40"])
def test_multi_iteration_run_equals_single_stepping(name):
    """run(niter) (one enqueue, device-side loop state) == niter x run(1)."""
    c = cases.CASES[name]
    X, W0, H0 = cases.build(name)
    e1 = pymf_b200.Engine(c["d"], c["n"], c["k"])
    e2 = pymf_b200.Engine(c["d"], c["n"], c["k"])
    try:
        for e in (e1, e2):
            e.upload_x(X); e.set_w(W0); e.set_h(H0)
        f1, done = e1.run(12, early_stop=False)
        f2 = np.array([e2.run(1, early_stop=False)[0][0] for _ in range(12)])
        assert done == 12
        np.testing.assert_allclose(f1, f2, rtol=1e-5)
        assert rel(e1.get_w(), e2.get_w()) < 1e-5
        assert rel(e1.get_h(), e2.get_h()) < 1e-5
    finally:
        e1.close(); e2.close()


def test_reference_test_sequence_on_gpu(golden_dir):
    """tests/test_pymf.py:69,84-95 through pymf_b200.NMF on the GPU, value-for-value."""
    g = np.load(os.path.join(golden_dir, "ref_test_3x50.npz"))
    A = cases.ref_test_matrix()
    np.random.seed(cases.REF_TEST_INIT_SEED)
    m = pymf_b200.NMF(A, num_bases=4)
    m.factorize(show_progress=False, niter=20)
    assert m.ferr.shape == (20,)
    assert m.ferr[-1] / (A.shape[0] + A.shape[1]) < 0.1
    assert np.max(np.abs(m.ferr - g["ferr_20"]) / g["ferr_20"]) < TOL_FERR
    assert rel(m.W, g["W_20"]) < TOL_WH and rel(m.H, g["H_20"]) < TOL_WH
    m.factorize(compute_h=False)
    assert rel(m.W, g["W_a"]) < TOL_WH and rel(m.H, g["H_a"]) < TOL_WH
    assert abs(m.ferr[0] - g["ferr_a"][0]) / g["ferr_a"][0] < TOL_FERR
    m.factorize(compute_w=False)
    assert rel(m.H, g["H_b"]) < TOL_WH
    assert abs(m.ferr[0] - g["ferr_b"][0]) / g["ferr_b"][0] < TOL_FERR
    old = m.ferr.copy()
    m.factorize(compute_err=False)
    np.testing.assert_array_equal(m.ferr, old)
    assert rel(m.W, g["W_c"]) < TOL_WH and rel(m.H, g["H_c"]) < TOL_WH
    m.factorize(niter=20)
    assert rel(m.W, g["W_d"]) < TOL_WH and rel(m.H, g["H_d"]) < TOL_WH
    assert np.max(np.abs(m.ferr - g["ferr_d"]) / g["ferr_d"]) < TOL_FERR
    assert isinstance(m.W, np.ndarray) and m.W.dtype == np.float64


def test_frobenius_norm_matches_bruteforce():
    """Trace-identity error vs the oracle's direct ||X - WH|| (pymf/nmf.py:110)."""
    rng = np.random.RandomState(3)
    for (d, n, k) in [(64, 96, 8), (300, 1000, 40), (1000, 500, 10)]:
        X = rng.random_sample((d, n))
        m = pymf_b200.NMF(X, num_bases=k)
        m.W = rng.random_sample((d, k))
        m.H = rng.random_sample((k, n))
        want = O.frobenius_norm(X, m.W, m.H)
        assert abs(m.frobenius_norm() - want) / want < TOL_FERR
        for mode in ("trace", "direct"):
            m._engine.set_err_mode(mode)
            assert abs(m.frobenius_norm() - want) / want < TOL_FERR, mode


def test_early_stop_state_is_consistent():
    """Convergence on the 3x50 case: the stop index may differ from float64 (SURVEY 7.3), the
    state must be consistent: len(ferr) == iterations_done - 1, W/H are those of the last
    executed iteration, and the float64 oracle continued from them barely moves."""
    A = cases.ref_test_matrix()
    np.random.seed(cases.REF_TEST_INIT_SEED)
    W0, H0 = O.init_wh(3, 50, 4)
    e = pymf_b200.Engine(3, 50, 4)
    try:
        e.upload_x(A); e.set_w(W0); e.set_h(H0)
        ferr, done = e.run(100000, early_stop=True)
        assert 3 <= done < 100000 and len(ferr) == done - 1
        W, H = e.get_w(), e.get_h()
        # the engine's state equals `done` float64 iterations within tolerance
        Wr, Hr = W0.copy(), H0.copy()
        O.factorize(A, Wr, Hr, niter=done, early_stop=False)
        assert rel(W, Wr) < 5e-3 and rel(H, Hr) < 5e-3     # long run (thousand+ iterations)
        # near-exact fit: ferr ~ 1e-4 on ||A|| ~ 18, so allow the fp32 representation floor of W/H
        assert abs(O.frobenius_norm(A, W, H) - ferr[-1]) < TOL_FERR * ferr[-1] + 1e-6 * np.linalg.norm(A)
        # a second run continues from that state (warm start) and does not crash
        f2, d2 = e.run(3, early_stop=True)
        assert d2 == 3 and len(f2) == 3
    finally:
        e.close()


def test_hash_generator_matches_device():
    d, n, k = 70, 333, 5
    e = pymf_b200.Engine(d, n, k, n_global=n + 100, col0=60)
    try:
        e.gen_x(1234); e.gen_w(5); e.gen_h(6)
        W = e.get_w(np.float32); H = e.get_h(np.float32)
        np.testing.assert_array_equal(W, O.gen_matrix(5, d, k))
        np.testing.assert_array_equal(H, O.gen_matrix(6, k, n + 100, col0=60, ncols=n))
        # X is checked through one iteration against the oracle on the same block
        X = O.gen_matrix(1234, d, n + 100, col0=60, ncols=n).astype(np.float64)
        Wr, Hr = W.astype(np.float64), H.astype(np.float64)
        fr = O.factorize(X, Wr, Hr, niter=2, early_stop=False)
        f, _ = e.run(2, early_stop=False)
        assert rel(e.get_w(), Wr) < TOL_WH and rel(e.get_h(), Hr) < TOL_WH
        assert np.max(np.abs(f - fr) / fr) < TOL_FERR
    finally:
        e.close()


def test_device_tensor_input_is_borrowed():
    import torch
    rng = np.random.RandomState(1)
    X = rng.random_sample((128, 256)).astype(np.float32)
    xt = torch.from_numpy(X).cuda()
    np.random.seed(2)
    a = pymf_b200.NMF(xt, num_bases=16)
    a.factorize(niter=5)
    np.random.seed(2)
    b = pymf_b200.NMF(X, num_bases=16)
    b.factorize(niter=5)
    np.testing.assert_allclose(a.ferr, b.ferr, rtol=1e-5)
    Wr, Hr = None, None
    np.random.seed(2)
    Wr, Hr = O.init_wh(128, 256, 16)
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=5)
    assert rel(a.W, Wr) < TOL_WH and rel(a.H, Hr) < TOL_WH
    assert np.max(np.abs(a.ferr - fr) / fr) < TOL_FERR


def test_large_shape_properties():
    """Size-independent properties at a size the CPU oracle cannot single-step quickly:
    monotone non-increasing ferr (Lee-Seung), non-negativity, finite values, and the
    trace-identity error against a brute-force error on a sampled column block."""
    d, n, k = 4096, 32768, 32
    e = pymf_b200.Engine(d, n, k)
    try:
        e.gen_x(1234); e.gen_w(1235); e.gen_h(1236)
        ferr, done = e.run(10, early_stop=False)
        assert done == 10 and np.all(np.isfinite(ferr))
        assert np.all(np.diff(ferr) <= 1e-5 * ferr[:-1])
        W = e.get_w(); H = e.get_h()
        assert W.min() >= 0 and H.min() >= 0 and np.isfinite(W).all() and np.isfinite(H).all()
        # brute-force error on 2048 sampled columns, scaled comparison of the per-column mean
        cols = np.arange(0, n, n // 2048)[:2048]
        Xs = np.stack([O.hash_uniform(1234, np.arange(d, dtype=np.uint64) * np.uint64(n) + np.uint64(c))
                       for c in cols], axis=1).astype(np.float64)
        part = np.sum((Xs - W.dot(H[:, cols])) ** 2) / len(cols)
        full = ferr[-1] ** 2 / n
        assert abs(part - full) / full < 0.02
    finally:
        e.close()


@pytest.mark.parametrize("shape", [(4096, 262144, 32), (8192, 131072, 64), (16384, 65536, 128)])
def test_full_size_properties(shape):
    """BASELINE-sized shards (cfg2 in full; cfg4 / cfg3 at their d and k on a 4 GiB column shard), data
    generated on the device: Lee-Seung monotonicity, non-negativity, and the trace-identity error of
    the tensor-core path against the direct fp32/fp64 residual pass sqrt(sum((X - W H)^2))."""
    d, n, k = shape
    e = pymf_b200.Engine(d, n, k)
    try:
        e.set_err_mode("trace")
        e.gen_x(77); e.gen_w(78); e.gen_h(79)
        ferr, done = e.run(6, early_stop=False)
        assert e.active_path == "tc"
        assert done == 6 and np.all(np.isfinite(ferr))
        assert np.all(np.diff(ferr) <= 1e-5 * ferr[:-1])
        e.set_err_mode("direct")
        direct = e.frobenius()
        assert abs(direct - ferr[-1]) / direct < TOL_FERR, (direct, ferr[-1])
        W = e.get_w(np.float32)
        assert W.min() >= 0 and np.isfinite(W).all()
    finally:
        e.close()


@pytest.mark.parametrize("shape", [(256, 512, 32), (300, 1000, 40), (512, 640, 128), (1024, 4096, 64),
                                   (4096, 2048, 32), (200, 3000, 96), (130, 131, 17),
                                   (2048, 8192, 256), (2048, 8200, 200), (4096, 4100, 16), (1024, 16384, 512)])
def test_tensor_core_path_matches_fp32_path(shape):
    """tcgen05 3xTF32 kernels vs the fp32 CUDA-core kernels vs the float64 oracle, 3 iterations,
    including shapes whose d / n / k are not multiples of the tile sizes, k <= 16 padded to 32 and
    128 < k <= 512 run as blocks of 128 bases (both only on streaming-sized problems, d*n >= 2^24)."""
    d, n, k = shape
    rng = np.random.RandomState(d + n + k)
    X = rng.random_sample((d, n)).astype(np.float32)
    W0 = rng.random_sample((d, k))
    H0 = rng.random_sample((k, n))
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=3, early_stop=False)
    res = {}
    for path in ("simt", "tc"):
        e = pymf_b200.Engine(d, n, k, path=path)
        try:
            e.set_err_mode("trace")
            e.upload_x(X); e.set_w(W0); e.set_h(H0)
            f, done = e.run(3, early_stop=False)
            assert e.active_path == path
            res[path] = (e.get_w(), e.get_h(), f)
        finally:
            e.close()
        W, H, f = res[path]
        assert rel(W, Wr) < TOL_WH, (path, rel(W, Wr))
        assert rel(H, Hr) < TOL_WH, (path, rel(H, Hr))
        assert np.max(np.abs(f - fr) / fr) < TOL_FERR, path
    # the two kernel families agree far below the tolerance (3xTF32 ~ fp32 accuracy)
    assert rel(res["tc"][0], res["simt"][0]) < 2e-5
    assert rel(res["tc"][1], res["simt"][1]) < 2e-5


@pytest.mark.parametrize("shape", [(512, 4096 + 40, 32), (1000, 2000, 64), (700, 1157, 50)])
def test_ss_kernels_serve_small_k_when_forced(shape, monkeypatch):
    """The SS kernels (both operands from shared memory, three rings; the k >= 96 default) also instantiate for 32 and 64 bases
    (PYMFB_TC_FORCE_SS=1, used for A/B runs against the TS kernels): float64 oracle parity over 5 iterations."""
    d, n, k = shape
    monkeypatch.setenv("PYMFB_TC_FORCE_SS", "1")
    rng = np.random.RandomState(d + n + k)
    X = rng.random_sample((d, n)).astype(np.float32)
    W0 = rng.random_sample((d, k))
    H0 = rng.random_sample((k, n))
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=5, early_stop=False)
    e = pymf_b200.Engine(d, n, k, path="tc")
    try:
        e.set_err_mode("trace")
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        f, _ = e.run(5, early_stop=False)
        W, H = e.get_w(), e.get_h()
    finally:
        e.close()
    assert rel(W, Wr) < TOL_WH and rel(H, Hr) < TOL_WH
    assert np.max(np.abs(f - fr) / fr) < TOL_FERR


@pytest.mark.parametrize("shape", [(512, 4096, 32), (1000, 5000, 20), (4096, 8192, 32), (300, 1100, 32),
                                   (256, 40000, 32), (200, 50001, 20), (64, 131072, 32)])
def test_fused_one_pass_kernel_matches_two_pass(shape, monkeypatch):
    """kernels_fused.cuh (H update + X.H^T + H.H^T with X read once) vs the two-pass tensor-core
    kernels vs the float64 oracle; PYMFB_FUSED forces / disables the fused kernel.  d <= 256 (one row slab: the
    shapes where the one-pass kernel is the default) included."""
    d, n, k = shape
    rng = np.random.RandomState(d + n)
    X = rng.random_sample((d, n)).astype(np.float32)
    W0 = rng.random_sample((d, k)); H0 = rng.random_sample((k, n))
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=4, early_stop=False)
    res = {}
    for fused in ("0", "1"):
        monkeypatch.setenv("PYMFB_FUSED", fused)
        e = pymf_b200.Engine(d, n, k, path="tc")
        try:
            e.set_err_mode("trace")
            e.upload_x(X); e.set_w(W0); e.set_h(H0)
            f, done = e.run(4, early_stop=False)
            res[fused] = (e.get_w(), e.get_h(), f)
        finally:
            e.close()
        W, H, f = res[fused]
        assert rel(W, Wr) < TOL_WH and rel(H, Hr) < TOL_WH, (fused, rel(W, Wr), rel(H, Hr))
        assert np.max(np.abs(f - fr) / fr) < TOL_FERR, fused
    assert rel(res["1"][0], res["0"][0]) < 2e-5 and rel(res["1"][1], res["0"][1]) < 2e-5


def test_200_iteration_trajectory_on_the_one_pass_kernel():
    """The one-pass kernel is the default at d <= 256, k <= 32, d n > 2^24 (no knob set here).  Its W^T X chain truncates
    while its G H (k_gh_ratio) rounds to nearest, so the chain length sets a scale drift per iteration (DESIGN 5.1,
    "Segments"): W / H must stay within 1e-4 of the float64 oracle over 200 iterations."""
    d, n, k = 256, 65536 + 128, 32
    X = O.gen_matrix(81, d, n)
    W0 = O.gen_matrix(82, d, k).astype(np.float64)
    H0 = O.gen_matrix(83, k, n).astype(np.float64)
    Wr, Hr = W0.copy(), H0.copy()
    e = pymf_b200.Engine(d, n, k)
    try:
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        e.set_err_mode("trace")
        at = 0
        for stop in (50, 100, 200):
            f, done = e.run(stop - at, early_stop=False)
            assert done == stop - at
            O.factorize(X.astype(np.float64), Wr, Hr, niter=stop - at, compute_err=False, early_stop=False)
            at = stop
            rw, rh = rel(e.get_w(), Wr), rel(e.get_h(), Hr)
            assert rw < TOL_WH and rh < TOL_WH, (stop, rw, rh)
        print("200-iteration one-pass trajectory: rel W %.2e, rel H %.2e" % (rw, rh))
    finally:
        e.close()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_pinned_ingest_equals_pageable_ingest(dtype):
    """X from page-locked memory (direct DMA, pymfb_upload_x fast path) gives the same device
    matrix as the pageable staging ring: identical trajectories, incl. a strided row view and a
    row count that spans several fp64 staging chunks."""
    d, n, k = 300, 70001, 8                       # 300 x 70001 f64 = 168 MB > 2 x 64 MB staging chunks
    rng = np.random.RandomState(5)
    base = pymf_b200.pinned_empty((d, n + 13), dtype)
    base[...] = rng.random_sample((d, n + 13))
    Xp = base[:, 5:5 + n]                         # strided view of pinned memory (ld = n + 13)
    Xh = np.array(Xp)                             # pageable dense copy
    W0 = rng.random_sample((d, k)); H0 = rng.random_sample((k, n))
    out = []
    for X, want_direct in ((Xp, True), (Xh, False)):
        m = pymf_b200.NMF(X, num_bases=k)
        m.W, m.H = W0.copy(), H0.copy()
        # one H update touches every element of X and has no atomics: bit-exact on identical device data
        m.factorize(niter=1, compute_w=False, compute_err=False)
        assert m._engine.last_upload_pinned == want_direct
        h1 = m.H.copy()
        m.W, m.H = W0.copy(), H0.copy()
        m.factorize(niter=3)
        out.append((h1, m.W.copy(), m.H.copy(), m.ferr.copy()))
    np.testing.assert_array_equal(out[0][0], out[1][0])
    assert rel(out[0][1], out[1][1]) < 2e-6 and rel(out[0][2], out[1][2]) < 2e-6   # fp32 atomics order only
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(Xh.astype(np.float64), Wr, Hr, niter=3)
    assert rel(out[0][1], Wr) < TOL_WH and rel(out[0][2], Hr) < TOL_WH
    assert np.max(np.abs(out[0][3] - fr) / fr) < TOL_FERR


def test_factors_download_in_place_into_pinned_arrays():
    d, n, k = 128, 1024, 16
    rng = np.random.RandomState(6)
    X = rng.random_sample((d, n))
    W = pymf_b200.pinned_empty((d, k), np.float64); W[...] = rng.random_sample((d, k))
    H = pymf_b200.pinned_empty((k, n), np.float32); H[...] = rng.random_sample((k, n))
    Wr, Hr = W.copy(), H.astype(np.float64)
    m = pymf_b200.NMF(X, num_bases=k)
    m.W, m.H = W, H
    m.factorize(niter=4)
    assert m.W is W and m.H is H                  # identity kept, values written in place
    O.factorize(X, Wr, Hr, niter=4)
    assert rel(W, Wr) < TOL_WH and rel(H, Hr) < TOL_WH


@pytest.mark.parametrize("flags", [(True, True, True), (True, True, False), (False, True, True), (True, False, True),
                                   (False, True, False)])
@pytest.mark.parametrize("shape", [(200, 333, 7), (256, 1024, 32)])
def test_graph_replay_equals_plain_launches(shape, flags):
    """Launch-bound problems replay two iterations per CUDA graph launch (pymfb.cu graph_build); the
    results are those of the plain launch sequence (up to the atomic summation order of the X.H^T flush)."""
    d, n, k = shape
    cw, ch, ce = flags
    X = O.gen_matrix(41, d, n)
    W0 = O.gen_matrix(42, d, k).astype(np.float64)
    H0 = O.gen_matrix(43, k, n).astype(np.float64)
    res = {}
    for mode in ("off", "auto"):
        e = pymf_b200.Engine(d, n, k)
        try:
            e.set_graph_mode(mode)
            e.upload_x(X); e.set_w(W0); e.set_h(H0)
            f1, done1 = e.run(11, compute_w=cw, compute_h=ch, compute_err=ce, early_stop=False)
            f2, done2 = e.run(6, compute_w=cw, compute_h=ch, compute_err=ce, early_stop=False)   # cached graph
            assert done1 == 11 and done2 == 6
            res[mode] = (e.get_w(), e.get_h(), np.concatenate([f1, f2]), e.graph_replays, e.frobenius())
        finally:
            e.close()
    assert res["off"][3] == 0 and res["auto"][3] == 4 + 1          # (11 - 3) // 2 and (6 - 3) // 2 replays
    assert rel(res["auto"][0], res["off"][0]) < 1e-5 and rel(res["auto"][1], res["off"][1]) < 1e-5
    if ce:
        np.testing.assert_allclose(res["auto"][2], res["off"][2], rtol=1e-5)
    assert abs(res["auto"][4] - res["off"][4]) <= 1e-5 * res["off"][4]
    # and against the oracle
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=17, compute_w=cw, compute_h=ch, compute_err=ce, early_stop=False)
    assert rel(res["auto"][0], Wr) < TOL_WH and rel(res["auto"][1], Hr) < TOL_WH
    if ce:
        f = res["auto"][2]
        frr = np.concatenate([fr[:11], fr[11:17]])
        assert np.max(np.abs(f - frr) / frr) < TOL_FERR


def test_graph_replay_keeps_early_stop_semantics(golden_dir):
    """The reference's 3x50 case stops early (pymf/nmf.py:198-202); the device-side stop flag also ends a
    replayed run: same iteration count and ferr length with and without graphs."""
    A = cases.ref_test_matrix()
    out = {}
    for mode in ("off", "auto"):
        np.random.seed(cases.REF_TEST_INIT_SEED)
        W0, H0 = O.init_wh(3, 50, 4)
        e = pymf_b200.Engine(3, 50, 4)
        try:
            e.set_graph_mode(mode)
            e.upload_x(A); e.set_w(W0); e.set_h(H0)
            ferr, done = e.run(5000)
            out[mode] = (len(ferr), done, e.get_w(), ferr, e.graph_replays)
        finally:
            e.close()
    assert out["auto"][4] > 0
    assert out["auto"][1] == len(out["auto"][3]) + 1 or out["auto"][1] == 5000
    # fp32 round-off moves the exact stopping index a little from run to run (atomics); the state must be consistent
    assert abs(out["auto"][0] - out["off"][0]) <= max(5, 0.05 * out["off"][0])
    assert rel(out["auto"][2], out["off"][2]) < 1e-3


def test_c_abi_reports_errors_instead_of_crashing():
    """Error convention of include/pymfb.h: non-zero return + pymfb_last_error(), never an exception or a crash."""
    import ctypes as C
    from pymf_b200 import _lib
    lib = _lib.load()
    ctx = C.c_void_p()
    assert lib.pymfb_create(C.byref(ctx), 0, 0, 10, 10, 0, 2) != 0 and b"bad shape" in lib.pymfb_last_error()
    assert lib.pymfb_create(C.byref(ctx), 99, 8, 8, 8, 0, 2) != 0 and b"out of range" in lib.pymfb_last_error()
    e = pymf_b200.Engine(16, 200, 3)
    try:
        with pytest.raises(pymf_b200.PymfbError, match="no data bound"):
            e.run(1)
        e.upload_x(np.random.RandomState(0).random_sample((16, 200)))
        with pytest.raises(pymf_b200.PymfbError, match="W and H must be set"):
            e.run(1)
        with pytest.raises(ValueError):
            e.set_w(np.zeros((5, 3)))
        with pytest.raises(pymf_b200.PymfbError, match="tcgen05 path not available"):
            e.set_path("tc")                       # d = 16 is below the tensor path's minimum
        e.set_path("auto")
        with pytest.raises(pymf_b200.PymfbError, match="bad penalty"):
            e.set_penalty(-1.0, 0.0)
        assert lib.pymfb_upload_x(e._ctx, None, 0, 200) != 0 and b"null" in lib.pymfb_last_error()
        e.set_w(np.ones((16, 3))); e.set_h(np.ones((3, 200)))
        f, done = e.run(2)
        assert done == 2 and np.all(np.isfinite(f))
        assert e.run(0)[1] == 0                    # niter = 0 is a no-op
    finally:
        e.close()


@pytest.mark.parametrize("shape", [(1024, 128 * 33, 64), (700, 128 * 9 + 5, 20)])
def test_cta_pair_h_update_kernel_is_bit_identical(shape, monkeypatch):
    """Opt-in CTA-pair (tcgen05 cta_group::2) H-update kernel (PYMFB_TS2=1, kernels_ts2.cuh): same MMAs in the same
    order as the single-CTA kernel, so one H update must be bit-identical - odd tile count (virtual OOB tile), ragged n."""
    d, n, k = shape
    out = []
    for ts2 in (False, True):
        if ts2:
            monkeypatch.setenv("PYMFB_TS2", "1")
        else:
            monkeypatch.delenv("PYMFB_TS2", raising=False)
        e = pymf_b200.Engine(d, n, k, path="tc")
        try:
            e.gen_x(1); e.gen_w(2); e.gen_h(3)
            e.run(1, compute_w=False, compute_h=True, compute_err=False, early_stop=False)
            H = e.get_h(np.float32)
            f, _ = e.run(2, early_stop=False)
            out.append((H, f))
        finally:
            e.close()
    np.testing.assert_array_equal(out[0][0], out[1][0])
    np.testing.assert_allclose(out[0][1], out[1][1], rtol=1e-6)


@pytest.mark.parametrize("shape", [(1024, 128 * 33, 128), (700, 128 * 9 + 5, 100), (2048, 128 * 100 + 17, 256)])
def test_cta_pair_ss_h_update_kernel_is_bit_identical(shape, monkeypatch):
    """Opt-in CTA-pair SS H-update kernel (PYMFB_TC2=1, kernels_tc2.cuh; 128-wide blocks of bases): one tcgen05.mma.cta_group::2
    covers the tiles of both CTAs with the same per-tile MMA chain as k_h_update_tc, so one H update must be bit-identical -
    odd tile count (virtual out-of-bounds tile), ragged n and d, k below the padded width, two blocks of bases."""
    d, n, k = shape
    out = []
    for tc2 in (False, True):
        if tc2:
            monkeypatch.setenv("PYMFB_TC2", "1")
        else:
            monkeypatch.delenv("PYMFB_TC2", raising=False)
        e = pymf_b200.Engine(d, n, k, path="tc")
        try:
            e.gen_x(1); e.gen_w(2); e.gen_h(3)
            e.run(1, compute_w=False, compute_h=True, compute_err=False, early_stop=False)
            H = e.get_h(np.float32)
            f, _ = e.run(2, early_stop=False)
            out.append((H, f))
        finally:
            e.close()
    np.testing.assert_array_equal(out[0][0], out[1][0])
    np.testing.assert_array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("shape", [(1024, 128 * 33, 64), (700, 128 * 9 + 5, 20), (2048 + 40, 128 * 12, 32)])
def test_ts_h_update_kernel_variants_are_bit_identical(shape, monkeypatch):
    """The TS H-update kernels (k <= 64) exist in four schedules - 32-row stages with separate commits (PYMFB_TS_RS=1, the
    k = 64 default), two MMA-issuing warps (2), 32- and 64-row stages with one commit per stage (32 / 64; 64 is the
    k <= 32 default).  They issue the same MMAs in the same order over the same segments, so H after one update and the
    errors of two further iterations must be bit-identical - ragged d (rows beyond the matrix are zero-filled by TMA),
    ragged n, k below the padded width."""
    d, n, k = shape
    out = []
    for rs in ("1", "2", "32", "64"):
        monkeypatch.setenv("PYMFB_TS_RS", rs)
        e = pymf_b200.Engine(d, n, k, path="tc")
        try:
            e.gen_x(1); e.gen_w(2); e.gen_h(3)
            e.run(1, compute_w=False, compute_h=True, compute_err=False, early_stop=False)
            H = e.get_h(np.float32)
            f, _ = e.run(2, early_stop=False)
            out.append((H, f))
        finally:
            e.close()
    for o in out[1:]:
        np.testing.assert_array_equal(out[0][0], o[0])
        np.testing.assert_array_equal(out[0][1], o[1])


@pytest.mark.parametrize("shape,path", [((1000, 500, 10), "simt"), ((512, 4096, 32), "tc"), ((1024, 4096, 128), "tc"),
                                        ((300, 3000, 40), "tc"), ((256, 65536 + 128, 32), "tc"), ((150, 120000, 20), "tc")])
def test_runs_are_bit_reproducible(shape, path):
    """The column splits of X H^T / H H^T are combined in a fixed order (partial copies, no atomics), so
    two runs of the same problem in one process give bit-identical W, H and ferr - also on the d <= 256, k <= 32 shapes
    that run the one-pass kernel by default (one copy of [A | B] per CTA group, summed in group order)."""
    d, n, k = shape
    X = O.gen_matrix(71, d, n)
    W0 = O.gen_matrix(72, d, k).astype(np.float64)
    H0 = O.gen_matrix(73, k, n).astype(np.float64)
    out = []
    for _ in range(2):
        e = pymf_b200.Engine(d, n, k, path=path)
        try:
            e.upload_x(X); e.set_w(W0); e.set_h(H0)
            f, done = e.run(9, early_stop=False)
            out.append((e.get_w(np.float32), e.get_h(np.float32), f))
        finally:
            e.close()
    np.testing.assert_array_equal(out[0][0], out[1][0])
    np.testing.assert_array_equal(out[0][1], out[1][1])
    np.testing.assert_array_equal(out[0][2], out[1][2])
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=9, early_stop=False)
    assert rel(out[0][0], Wr) < TOL_WH and rel(out[0][1], Hr) < TOL_WH
    assert np.max(np.abs(out[0][2] - fr) / fr) < TOL_FERR


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_panel_streamed_ingest_equals_in_memory_ingest(dtype, monkeypatch):
    """An h5py-like source (only `.shape`, `.dtype`, slicing) is ingested in column panels data[:, c0:c1] through two
    page-locked panel buffers (pymfb_upload_x_panel); the device matrix, hence the trajectory, is the one of the
    in-memory upload - ragged last panel, fp64 panels cast on the device."""
    import pymf_b200.engine as eng_mod
    from tests.test_host_logic import RecordingSource
    d, n, k = 300, 5000, 8
    rng = np.random.RandomState(8)
    X = rng.random_sample((d, n)).astype(dtype)
    W0 = rng.random_sample((d, k)); H0 = rng.random_sample((k, n))
    orig = eng_mod.panel_ranges
    monkeypatch.setattr(eng_mod, "panel_ranges", lambda d_, n_, isz, pb=0: orig(d_, n_, isz, d * isz * 640))
    src = RecordingSource(X)
    out = []
    for data in (src, X):
        m = pymf_b200.NMF(data, num_bases=k)
        m.W, m.H = W0.copy(), H0.copy()
        m.factorize(niter=1, compute_w=False, compute_err=False)      # one H update: no split combine, bit-exact
        h1 = m.H.copy()
        m.W, m.H = W0.copy(), H0.copy()
        m.factorize(niter=4)
        out.append((h1, m.W.copy(), m.H.copy(), m.ferr.copy()))
    assert len(src.reads) == 8 and src.widest_read() == 640            # 7 x 640 + 520 columns
    for a, b in zip(out[0], out[1]):
        np.testing.assert_array_equal(a, b)
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=4)
    assert rel(out[0][1], Wr) < TOL_WH and rel(out[0][2], Hr) < TOL_WH
    assert np.max(np.abs(out[0][3] - fr) / fr) < TOL_FERR


def test_trace_identity_hands_over_to_the_direct_residual_when_it_cancels():
    """Near-exact low-rank data at a size where the error normally comes from the trace identity (d n k > 2^28):
    once ferr^2 drops below 1e-3 ||X||^2 the identity has lost its digits; the library flags it, takes no early-stop
    decision from such a value, and measures the error directly (pymf/nmf.py:110 as written) from the next call on."""
    d, n, k, r = 2048, 8192, 32, 4
    rng = np.random.RandomState(1)
    X = (rng.random_sample((d, r)).dot(rng.random_sample((r, n))) + 1e-4 * rng.random_sample((d, n))).astype(np.float32)
    W0 = rng.random_sample((d, k)); H0 = rng.random_sample((k, n))
    m = pymf_b200.NMF(X, num_bases=k)
    m.W, m.H = W0.copy(), H0.copy()
    m.factorize(niter=150)
    xx = float(np.sum(X.astype(np.float64) ** 2))
    assert m.ferr[-1] ** 2 < 1e-3 * xx                        # deep in the cancelling regime
    assert len(m.ferr) == 150                                   # no noise-driven early stop
    W, H = m.W.copy(), m.H.copy()
    true = O.frobenius_norm(X.astype(np.float64), W, H)
    assert abs(m.frobenius_norm() - true) / true < TOL_FERR    # measured directly now
    m.factorize(niter=3)
    Wr, Hr = W.copy(), H.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=3)
    assert np.max(np.abs(m.ferr - fr) / fr) < TOL_FERR


@pytest.mark.parametrize("shape", [(300, 1000, 20), (512, 4100, 32), (1024, 2500, 128), (256, 3000, 64)])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_panel_major_x_equals_row_major_x(shape, dtype, monkeypatch):
    """Wide context-owned matrices are stored panel-major (column panels of 4096 columns, common.cuh) so that a TMA
    box stays inside one page; PYMFB_XPANEL=7 forces 128-column panels on a small matrix.  Every reader of X (both
    kernel families, ||X||^2, the direct residual, the column sums, NNDSVD) and every ingest path (pinned, pageable,
    h5py-like panels) must see the same matrix: one H update is bit-identical, trajectories match the oracle."""
    from tests.test_host_logic import RecordingSource
    d, n, k = shape
    rng = np.random.RandomState(n)
    X = rng.random_sample((d, n)).astype(dtype)
    W0 = rng.random_sample((d, k)); H0 = rng.random_sample((k, n))
    Xp = pymf_b200.pinned_empty((d, n), dtype); Xp[...] = X
    Wr, Hr = W0.copy(), H0.copy()
    fr = O.factorize(X.astype(np.float64), Wr, Hr, niter=3, early_stop=False)
    res = {}
    for layout in ("0", "7"):
        monkeypatch.setenv("PYMFB_XPANEL", layout)
        for path in ("simt", "tc"):
            for src_name, data in (("pageable", X), ("pinned", Xp), ("panels", RecordingSource(X))):
                m = pymf_b200.NMF(data, num_bases=k, path=path)
                m.W, m.H = W0.copy(), H0.copy()
                m.factorize(niter=1, compute_w=False, compute_err=False)
                h1 = m.H.copy()
                m.W, m.H = W0.copy(), H0.copy()
                m._engine.set_err_mode("trace")
                m.factorize(niter=3)
                f_trace = m.ferr.copy()
                m._engine.set_err_mode("direct")
                f_direct = m.frobenius_norm()
                res[(layout, path, src_name)] = (h1, m.W.copy(), m.H.copy(), f_trace, f_direct)
                assert rel(m.W, Wr) < TOL_WH and rel(m.H, Hr) < TOL_WH, (layout, path, src_name)
                assert np.max(np.abs(f_trace - fr) / fr) < TOL_FERR and abs(f_direct - fr[-1]) / fr[-1] < TOL_FERR
    for path in ("simt", "tc"):
        ref = res[("0", path, "pageable")]
        for key, val in res.items():
            if key[1] == path:
                np.testing.assert_array_equal(val[0], ref[0], err_msg=str(key))     # one H update: bit-identical
                np.testing.assert_array_equal(val[1], ref[1], err_msg=str(key))     # deterministic combine: W too
                np.testing.assert_array_equal(val[3], ref[3], err_msg=str(key))
    # NNDSVD reads X through the same layout
    monkeypatch.setenv("PYMFB_XPANEL", "0")
    a = pymf_b200.NNDSVD(X, num_bases=min(k, 8)); a.factorize()
    monkeypatch.setenv("PYMFB_XPANEL", "7")
    b = pymf_b200.NNDSVD(X, num_bases=min(k, 8)); b.factorize()
    np.testing.assert_array_equal(a.W, b.W)
    np.testing.assert_array_equal(a.H, b.H)
