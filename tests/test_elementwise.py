"""Every update pass, element by element, against the float64 update on the same float32 inputs.

The other parity tests measure the relative Frobenius error of the whole W and H.  On parts-based data most entries of
W and H are near zero, and a kernel can be badly wrong on exactly those entries while the large ones carry the norm.
This file holds each pass to a per-element bound instead.

Contract
--------
Error model: each contraction of a pass (C = W^T X, D = G H with G = W^T W, A = X H^T, W B with B = H H^T) is a sum of
products, and its computed value obeys the standard forward error bound of a dot product,

    |C_hat - C| <= gamma * (|W|^T |X|)          elementwise, and the same form for D, A and W B.

The reference is the float64 update of ``oracle/nmf_oracle.py`` applied to the inputs AFTER rounding them to float32,
so that input rounding does not count as kernel error.  One tolerance, TAU = 1e-5, stands for gamma in every kernel
family (honest kernels sit near 1e-6; the failures this file was written against sit at 1e-2 and above):

* NMF and BNMF: every operand is non-negative, so |W|^T |X| = C and every term of the ratio is a sum of non-negative
  terms.  Each element of the new H (and the new W) is within TAU relative of its reference:
  |h_hat - h| <= TAU * max(|h|, FLOOR).
* SNMF (``snmf_ratio``): C = W^T X is signed.  With E = |W|^T |X| + 2 (|W|^T |W|) H (H >= 0), the device's
  num = c+ + (G- H) and den = c- + (G+ H) + 1e-9 each lie within TAU * E of the reference: |c_hat+ - c+| <= |c_hat - c|
  <= TAU |W|^T|X|; G_hat+- is within TAU |W|^T|W| of G+- and the product with H adds TAU (|W|^T|W|) H once more.  The
  new h = h_old * sqrt(num / den) therefore lies in
      [h_old * sqrt(max(num - TAU E, 0) / (den + TAU E)),  h_old * sqrt((num + TAU E) / max(den - TAU E, 0))]
  widened by 8 float32 ulps for the epilogue's own divide, square root and multiply.
* The error ||X - W H||: in the direct form and in the trace form ||X||^2 - 2 <W, A> + <G, B> alike, the computed
  square is within TAU * S of the reference, S = sum (|X| + |W| |H|)^2, so |f_hat - f| <= TAU * S / (f_hat + f).
* FLOOR = 1e-30: below it a reference value is compared in absolute terms (TAU * FLOOR).  No data set here drives a
  pass near it: the smallest non-zero reference values are about 1e-16.

Each pass is isolated through the public Engine API: one H update is set_w, set_h, run(1, compute_w=False,
compute_err=False); one W update is run(1, compute_h=False, compute_err=False) (the X H^T / H H^T bootstrap pass on the
current H, then k_update_w); the error is frobenius() in direct and in trace mode.  The one-pass kernel has no H-only
mode: it runs when A and B of the new H are needed, so it is checked through one and two full iterations in trace
mode, the second W update consuming its A and B.

Data families (seeded, generated here): uniform (the control); parts-based with exact zeros; parts-based near
convergence (floors of 1e-9 on W, 1e-7 on X and H); columns of X scaled by 2^u, u uniform in [-20, 20]; zero rows and
columns of X and an all-zero basis of W.  Shapes are ragged (d = 1000, n = 1300: neither a multiple of 32 nor of 128,
11 column tiles) and k sits below its padded width wherever the kernel family allows it.
"""
import zlib

import numpy as np
import pytest
import scipy.sparse as sp

import pymf_b200
from oracle import nmf_oracle as O

pytestmark = pytest.mark.gpu

TAU = 1e-5
FLOOR = 1e-30
ULP32 = 2.0 ** -24

D, N = 1000, 1300
FAMILIES = ["uniform", "parts_zero", "parts_floor", "colscale", "zeros"]

# (id, k, path, environment): one entry per kernel family / schedule (DESIGN.md 11 lists the knobs).  The tensor-core
# path serves padded widths of 32..128 in steps of 32 and 256 / 384 / 512 only: k = 16 is not a tensor-core shape (the
# 64-row TS kernel is taken at k = 20, 24, 32), and the two-block SS case is k = 240 (k = 200 would pad to 224).
DENSE_CASES = [
    ("simt-k20", 20, "simt", {}),
    ("simt-k64", 64, "simt", {}),
    ("tsr64-k24", 24, "tc", {}),
    ("tsr64-k20", 20, "tc", {}),
    ("tsr64-k32", 32, "tc", {}),
    ("ts-k20-rs1", 20, "tc", {"PYMFB_TS_RS": "1"}),
    ("ts-k20-rs32", 20, "tc", {"PYMFB_TS_RS": "32"}),
    ("ts-k50", 50, "tc", {}),
    ("ts-k64", 64, "tc", {}),
    ("ts-k50-rs1", 50, "tc", {"PYMFB_TS_RS": "1"}),
    ("ts-k50-rs2", 50, "tc", {"PYMFB_TS_RS": "2"}),
    ("ts-k50-rs32", 50, "tc", {"PYMFB_TS_RS": "32"}),
    ("ts-k50-rs64", 50, "tc", {"PYMFB_TS_RS": "64"}),
    ("ts2-k20", 20, "tc", {"PYMFB_TS2": "1"}),
    ("ts2-k64", 64, "tc", {"PYMFB_TS2": "1"}),
    ("ss-forced-k32", 32, "tc", {"PYMFB_TC_FORCE_SS": "1"}),
    ("ss-forced-k64", 64, "tc", {"PYMFB_TC_FORCE_SS": "1"}),
    ("ss-k96", 96, "tc", {}),
    ("ss-k128", 128, "tc", {}),
    ("ss-k240", 240, "tc", {}),
    ("ss-k256", 256, "tc", {}),
    ("ss-k512", 512, "tc", {}),
    ("tc2-k128", 128, "tc", {"PYMFB_TC2": "1"}),
]
CASE = {c[0]: c for c in DENSE_CASES}
# the epilogues of the penalised / semi-NMF ratios on the CUDA-core, TS and SS families
VARIANT_CASES = ["simt-k20", "tsr64-k20", "ts-k50", "ts-k64", "ss-forced-k32", "ss-k128", "ss-k240"]
ERROR_CASES = ["simt-k20", "tsr64-k20", "ts-k64", "ss-k128", "ss-k512"]


# --------------------------------------------------------------------------- data
def make_data(family, d, n, k, seed):
    """float32 X (d x n), W (d x k), H (k x n) of one data family."""
    rng = np.random.RandomState(seed)
    if family in ("uniform", "colscale", "zeros"):
        X, W, H = rng.random_sample((d, n)), rng.random_sample((d, k)), rng.random_sample((k, n))
        if family == "colscale":
            X *= 2.0 ** rng.uniform(-20.0, 20.0, size=n)[None, :]
        elif family == "zeros":
            X[rng.choice(d, max(1, d // 20), replace=False), :] = 0.0
            X[:, rng.choice(n, max(1, n // 20), replace=False)] = 0.0
            W[:, k // 2] = 0.0
    else:
        # k disjoint row blocks ("parts"), basis j lives on block j; each column holds 1-3 parts, and its column of H
        # is non-zero on those parts plus one other basis (a factorisation still in progress), whose C is exactly 0
        blk = np.repeat(np.arange(k), [len(b) for b in np.array_split(np.arange(d), k)])
        member = np.zeros((k, n), dtype=bool)
        hmask = np.zeros((k, n), dtype=bool)
        for c in range(n):
            parts = rng.choice(k, rng.randint(1, 4), replace=False)
            member[parts, c] = True
            hmask[parts, c] = True
            hmask[rng.choice(np.setdiff1d(np.arange(k), parts)), c] = True
        X = rng.random_sample((d, n)) * member[blk, :]
        W = rng.random_sample((d, k)) * (blk[:, None] == np.arange(k)[None, :])
        H = rng.random_sample((k, n)) * hmask
        if family == "parts_floor":
            X += 1e-7 * rng.random_sample((d, n))
            W = np.where(W == 0.0, 1e-9, W)
            H = np.where(H == 0.0, 1e-7, H)
    return X.astype(np.float32), W.astype(np.float32), H.astype(np.float32)


def f64(*arrays):
    return [np.asarray(a, dtype=np.float64) for a in arrays]


# --------------------------------------------------------------------------- checks
def assert_within(got, ref, bound, what):
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got - ref)
    bad = ~(err <= bound)
    if bad.any():
        rel = err / np.maximum(np.abs(ref), FLOOR)
        i = np.unravel_index(np.argmax(np.where(bad, rel, -1.0)), ref.shape)
        raise AssertionError("%s: %d of %d elements outside the bound; worst relative error %.3g at %s "
                             "(got %.9g, reference %.9g, bound %.3g)"
                             % (what, int(bad.sum()), bad.size, rel[i], i, got[i], ref[i], bound[i]))


def assert_rel(got, ref, what):
    assert_within(got, ref, TAU * np.maximum(np.abs(ref), FLOOR), what)


def assert_snmf_h(got, X, W, H, what):
    """The interval of the module docstring around the float64 snmf_update_h."""
    C = W.T @ X
    G = W.T @ W
    Gp, Gn = (np.abs(G) + G) / 2.0, (np.abs(G) - G) / 2.0
    E = np.abs(W).T @ np.abs(X) + 2.0 * (np.abs(W).T @ np.abs(W)) @ H
    num = np.maximum(C, 0.0) + Gn @ H
    den = np.maximum(-C, 0.0) + Gp @ H + O.EPS_DENOM
    ref = O.snmf_update_h(X, W, H.copy())
    assert np.all(H >= 0.0)
    lo = H * np.sqrt(np.maximum(num - TAU * E, 0.0) / (den + TAU * E)) * (1.0 - 8 * ULP32)
    with np.errstate(divide="ignore", invalid="ignore"):
        r_hi = np.where(den - TAU * E > 0.0, np.sqrt((num + TAU * E) / (den - TAU * E)), np.inf)
    hi = np.where(H == 0.0, 0.0, H * r_hi) * (1.0 + 8 * ULP32)
    assert np.all((lo <= ref) & (ref <= hi))
    got = np.asarray(got, dtype=np.float64)
    assert_within(got, (lo + hi) / 2.0, (hi - lo) / 2.0 + TAU * FLOOR, what)


def assert_ferr(got, X, W, H, what):
    ref = O.frobenius_norm(X, W, H)
    S = np.sum((np.abs(X) + np.abs(W) @ np.abs(H)) ** 2)
    bound = TAU * S / (got + ref) if got + ref > 0 else 0.0
    assert abs(got - ref) <= bound, "%s: ferr %.12g, reference %.12g, bound %.3g" % (what, got, ref, bound)


# --------------------------------------------------------------------------- engine helpers
def engine(monkeypatch, case, d=D, n=N, env=None):
    _, k, path, cenv = CASE[case] if isinstance(case, str) else case
    for key, val in dict(cenv, **(env or {})).items():
        monkeypatch.setenv(key, val)
    return pymf_b200.Engine(d, n, k, path=path)


def h_pass(e, X, W, H):
    e.set_w(W); e.set_h(H)
    e.run(1, compute_w=False, compute_err=False, early_stop=False)
    return e.get_h()


def w_pass(e, X, W, H):
    e.set_w(W); e.set_h(H)
    e.run(1, compute_h=False, compute_err=False, early_stop=False)
    return e.get_w()


def seed_of(*parts):
    return zlib.crc32("/".join(str(p) for p in parts).encode()) % (2 ** 31)


# --------------------------------------------------------------------------- NMF passes, dense
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("case", [c[0] for c in DENSE_CASES])
def test_h_update(case, family, monkeypatch):
    k = CASE[case][1]
    X, W, H = make_data(family, D, N, k, seed_of("h", family, k))
    e = engine(monkeypatch, case)
    try:
        e.upload_x(X)
        got = h_pass(e, X, W, H)
        assert e.active_path == CASE[case][2]
    finally:
        e.close()
    X, W, H = f64(X, W, H)
    assert_rel(got, O.update_h(X, W, H.copy()), "H update, %s, %s" % (case, family))


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("case", [c[0] for c in DENSE_CASES])
def test_w_update(case, family, monkeypatch):
    k = CASE[case][1]
    X, W, H = make_data(family, D, N, k, seed_of("w", family, k))
    e = engine(monkeypatch, case)
    try:
        e.upload_x(X)
        got = w_pass(e, X, W, H)
    finally:
        e.close()
    X, W, H = f64(X, W, H)
    assert_rel(got, O.update_w(X, W.copy(), H), "W update, %s, %s" % (case, family))


@pytest.mark.parametrize("mode", ["direct", "trace"])
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("case", ERROR_CASES)
def test_frobenius(case, family, mode, monkeypatch):
    k = CASE[case][1]
    X, W, H = make_data(family, D, N, k, seed_of("f", family, k))
    e = engine(monkeypatch, case)
    try:
        e.set_err_mode(mode)
        e.upload_x(X); e.set_w(W); e.set_h(H)
        got = e.frobenius()
    finally:
        e.close()
    assert_ferr(got, *f64(X, W, H), what="ferr (%s), %s, %s" % (mode, case, family))


# --------------------------------------------------------------------------- one-pass kernel
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("d,k", [(200, 20), (256, 32), (512, 32), (512, 24)])
def test_one_pass_kernel(d, k, family, monkeypatch):
    """PYMFB_FUSED=1: iteration 1 = bootstrap X H^T, W update, one-pass H update (+ its A, B), trace error; iteration 2's
    W update consumes the one-pass kernel's A and B.  Each pass against the float64 update of the device's inputs."""
    X, W0, H0 = make_data(family, d, N, k, seed_of("fused", family, d, k))
    e = engine(monkeypatch, ("fused", k, "tc", {"PYMFB_FUSED": "1"}), d=d)
    try:
        e.set_err_mode("trace")
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        Xd = f64(X)[0]
        W, H = f64(W0, H0)
        for it in (1, 2):
            f, _ = e.run(1, early_stop=False)
            Wn, Hn = e.get_w(np.float32), e.get_h(np.float32)
            tag = "iteration %d, d=%d k=%d, %s" % (it, d, k, family)
            assert_rel(Wn, O.update_w(Xd, W.copy(), H), "W update, " + tag)
            Wn64 = f64(Wn)[0]
            assert_rel(Hn, O.update_h(Xd, Wn64, H.copy()), "one-pass H update, " + tag)
            W, H = Wn64, f64(Hn)[0]
            assert_ferr(f[0], Xd, W, H, "ferr (trace), " + tag)
    finally:
        e.close()


# --------------------------------------------------------------------------- BNMF / SNMF epilogues
@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("case", VARIANT_CASES)
def test_bnmf_passes(case, family, monkeypatch):
    k = CASE[case][1]
    lam = {"W": 0.05, "H": 0.08}
    X, W, H = make_data(family, D, N, k, seed_of("bnmf", family, k))
    e = engine(monkeypatch, case)
    try:
        e.upload_x(X)
        e.set_penalty(lam["W"], lam["H"], 1.0, 1.0)
        gh = h_pass(e, X, W, H)
        gw = w_pass(e, X, W, H)
    finally:
        e.close()
    X, W, H = f64(X, W, H)
    assert_rel(gh, O.bnmf_update_h(X, W, H.copy(), dict(lam)), "BNMF H update, %s, %s" % (case, family))
    assert_rel(gw, O.bnmf_update_w(X, W.copy(), H, dict(lam)), "BNMF W update, %s, %s" % (case, family))


@pytest.mark.parametrize("family", FAMILIES + ["signed"])
@pytest.mark.parametrize("case", VARIANT_CASES)
def test_snmf_h_update(case, family, monkeypatch):
    k = CASE[case][1]
    X, W, H = make_data("uniform" if family == "signed" else family, D, N, k, seed_of("snmf", family, k))
    if family == "signed":           # X and W of both signs, as semi-NMF allows
        X, W = (X - np.float32(0.3)), (W - np.float32(0.3))
    e = engine(monkeypatch, case)
    try:
        e.set_variant("snmf")
        e.upload_x(X)
        got = h_pass(e, X, W, H)
    finally:
        e.close()
    assert_snmf_h(got, *f64(X, W, H), what="SNMF H update, %s, %s" % (case, family))


# --------------------------------------------------------------------------- sparse passes
@pytest.mark.parametrize("panel", [None, "256"])
@pytest.mark.parametrize("k", [32, 64, 128, 600])
@pytest.mark.parametrize("family", FAMILIES[1:])
def test_sparse_passes(family, k, panel, monkeypatch):
    """k_h_update_csc and k_xht_csr on X stored as CSC (families 3-5 are dense as a matrix: every column has more than
    512 non-zeros, which takes the split-column branch of the H update)."""
    X, W, H = make_data(family, D, N, k, seed_of("sparse", family, k))
    if panel:
        monkeypatch.setenv("PYMFB_SPARSE_PANEL", panel)
    m = sp.csc_matrix(X)
    m.sort_indices()
    e = pymf_b200.Engine(D, N, k)
    try:
        e.upload_x_csc(m.indptr, m.indices, m.data)
        assert e.active_path == "sparse"
        gh = h_pass(e, X, W, H)
        gw = w_pass(e, X, W, H)
    finally:
        e.close()
    X, W, H = f64(X, W, H)
    tag = "k=%d, %s, panel %s" % (k, family, panel)
    assert_rel(gh, O.update_h(X, W, H.copy()), "sparse H update, " + tag)
    assert_rel(gw, O.update_w(X, W.copy(), H), "sparse W update, " + tag)


# --------------------------------------------------------------------------- what a user sees
TRAJ_ITERS = 100
# An entry of H (or W) changes each iteration by a ratio whose numerator and denominator each carry at most TAU of
# relative error in the H update and again in the W update that feeds it: (1 + TAU)^4 per iteration, so after
# TRAJ_ITERS iterations a small entry lies within a factor (1 + TAU)^(4 * TRAJ_ITERS) ~ 1.004 of the oracle's.
# ASSUMPTION, not a derived bound: this counts only the errors of the entry's own ratios.  The deviations of the
# other entries of W and H also enter C and D of the next pass; the factor assumes that this coupling does not
# amplify them (near convergence the large entries sit at a fixed point of the update, which damps it).  A float32
# numpy restatement of the same 100 iterations stays within 2e-4 on these entries, against 4e-3 allowed here.
TRAJ_FACTOR = (1.0 + TAU) ** (4 * TRAJ_ITERS)
SMALL = 1e-6                         # "small": below this fraction of the largest entry of its column


@pytest.mark.parametrize("k,path", [(32, "tc"), (64, "tc"), (32, "simt")])
def test_small_entries_stay_small_over_100_iterations(k, path):
    """Parts-based data near convergence, 100 iterations from the same start against the float64 oracle: the entries the
    oracle holds below SMALL of their column's maximum (the zeros a user reads off a parts-based factorisation) must
    stay within TRAJ_FACTOR of the oracle's value."""
    X, W0, H0 = make_data("parts_floor", D, N, k, seed_of("traj", k))
    e = pymf_b200.Engine(D, N, k, path=path)
    try:
        e.upload_x(X); e.set_w(W0); e.set_h(H0)
        _, done = e.run(TRAJ_ITERS, compute_err=False, early_stop=False)
        assert done == TRAJ_ITERS
        Wg, Hg = e.get_w(), e.get_h()
    finally:
        e.close()
    Xd, Wr, Hr = f64(X, W0, H0)
    O.factorize(Xd, Wr, Hr, niter=TRAJ_ITERS, compute_err=False, early_stop=False)
    checked = 0
    for name, got, ref in (("W", Wg, Wr), ("H", Hg, Hr)):
        small = ref < SMALL * ref.max(axis=0, keepdims=True)
        checked += int(small.sum())
        bound = np.where(small, (TRAJ_FACTOR - 1.0) * np.maximum(ref, FLOOR), np.inf)
        assert_within(got, ref, bound, "small entries of %s after %d iterations, k=%d %s" % (name, TRAJ_ITERS, k, path))
    assert checked > 0
