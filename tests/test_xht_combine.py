"""The X H^T column splits of a large k = 128 problem are summed in a fixed order (DESIGN 5.8).

At 16384 x 524288, k = 128 the X H^T pass runs 37 column splits of 448 chunks, whose partial copies (310 MB) fit the
1 GiB budget of the ordered combine.  With tasks capped at ~4 K columns the same shape made 147 splits (1.23 GB of
copies) and fell back to fp32 atomics, so two runs differed in the last bits.  X (32 GiB) is generated on the device;
the host fp64 oracle of test_gpu_parity.py does not scale to it, so the error computed from A = X H^T by the trace
identity is checked against the direct residual instead.
"""
import numpy as np
import pytest

import pymf_b200

pytestmark = pytest.mark.gpu

TAU = 1e-5     # the per-element tolerance of tests/test_elementwise.py


def _run(d, n, k, niter):
    e = pymf_b200.Engine(d, n, k, path="tc")
    try:
        e.set_err_mode("trace")
        e.gen_x(51); e.gen_w(52); e.gen_h(53)
        f, done = e.run(niter, early_stop=False)
        assert done == niter
        W, H = e.get_w(np.float32), e.get_h(np.float32)
        e.set_err_mode("direct")
        f_direct = e.frobenius()
        return W, H, f, f_direct
    finally:
        e.close()


def test_large_k128_xht_splits_are_bit_reproducible():
    d, n, k = 16384, 524288, 128
    W1, H1, f1, fd1 = _run(d, n, k, 3)
    W2, H2, f2, fd2 = _run(d, n, k, 3)
    np.testing.assert_array_equal(W1, W2)
    np.testing.assert_array_equal(H1, H2)
    np.testing.assert_array_equal(f1, f2)
    # Trace form ||X||^2 - 2 <W, A> + <G, B> against ||X - W H|| as written: each is within TAU * S / (f_hat + f) of the
    # exact error, S = sum (|X| + |W| |H|)^2 (test_elementwise.py).  Everything is non-negative, so
    # S = ||X + W H||^2 <= (||X - W H|| + 2 ||W H||)^2, with ||W H||^2 = <W^T W, H H^T>.
    W64, H64 = W1.astype(np.float64), H1.astype(np.float64)
    wh = float(np.sqrt(np.sum((W64.T @ W64) * (H64 @ H64.T))))
    S = (fd1 + 2.0 * wh) ** 2
    assert abs(f1[-1] - fd1) <= 2.0 * TAU * S / (f1[-1] + fd1), (f1[-1], fd1)
