"""Time the sparse passes (NMF(..., sparse=True), DESIGN 5.9) at user-sized shapes on one GPU.

    python profiles/sparse_scale.py --out profiles/sparse_scale.json

Data, generated on the device with torch's seeded generator and handed to the library as host CSC arrays:
column c holds counts[c] rows drawn uniformly with replacement (duplicates dropped), values U(0, 1].  counts[c] is
Poisson(density * d), or, for "power-law" shapes, density * d * n * w_c / sum(w) with w_c = rank^-0.9 over a shuffled
column order (capped at d).

Per shape: the upload (host clock around upload_x_csc: copy, validation, CSR build); iterations/s (CUDA events around
N enqueued full iterations after a warm-up, ending in a synchronise); the two pass slots of pymfb_kernel_timing_read
(0: the H update with its G H launch, 1: X H^T + H H^T); in a separate run under torch.profiler the per-kernel device
time, which separates the dense k x k x n launches (k_gh_*, k_ltr_partial_simt + k_sum_partials on H^T) from the
sparse ones; achieved bytes/s of the two slots against the model 16 nnz + 8 kp n_local (X read in both formats, H read
and written once), next to a measured device-to-device copy rate.  The cfg2 density sweep also times the dense path on
the same matrix (bound as a device array).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import pymf_b200  # noqa: E402

SHAPES = [("text_k64", 1 << 17, 1 << 20, 0.0005, False, 64), ("text_k128", 1 << 17, 1 << 20, 0.0005, False, 128),
          ("cell_k32", 1 << 15, 1 << 19, 0.03, True, 32)]
DENSITIES = [0.005, 0.02, 0.05, 0.10, 0.20]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def make_csc(d, n, density, power_law, seed):
    """(indptr int64, indices int32, values float32) host arrays of the recipe in the module docstring."""
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    if power_law:
        w = 1.0 / torch.arange(1, n + 1, device=dev, dtype=torch.float64) ** 0.9
        counts = torch.clamp(torch.round(w / w.sum() * density * d * n), max=d).long()
        counts = counts[torch.randperm(n, generator=g, device=dev)]
    else:
        counts = torch.poisson(torch.full((n,), density * d, device=dev, dtype=torch.float32), generator=g).long()
    cols = torch.repeat_interleave(torch.arange(n, device=dev, dtype=torch.int64), counts)
    key = torch.unique(cols * d + torch.randint(0, d, (cols.numel(),), generator=g, device=dev))
    del cols
    indices = (key % d).to(torch.int32)
    indptr = torch.searchsorted(key // d, torch.arange(n + 1, device=dev, dtype=torch.int64))
    vals = 1.0 - torch.rand(key.numel(), generator=g, device=dev)
    del key
    return indptr.cpu().numpy(), indices.cpu().numpy(), vals.cpu().numpy()


def copy_rate():
    a = torch.empty(1 << 29, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 10 * 2 * a.numel() * 4 / (e0.elapsed_time(e1) * 1e-3)


def time_iters(e, niter):
    e.gen_w(1); e.gen_h(2)
    e.enqueue(3); e.sync()
    ev0, ev1 = e.event(), e.event()
    e.record(ev0)
    e.enqueue(niter)
    e.record(ev1)
    e.sync()
    return niter / (e.elapsed_ms(ev0, ev1) * 1e-3)


def kernel_split(e, niter):
    from torch.profiler import ProfilerActivity, profile
    e.gen_w(1); e.gen_h(2)
    e.enqueue(2); e.sync()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        e.enqueue(niter)
        e.sync()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.key.startswith("void pymfb"):
            name = ev.key.split("(")[0].replace("void ", "")
            out[name] = out.get(name, 0.0) + ev.device_time_total / 1e3 / niter        # ms per iteration
    return out


def run_sparse(d, n, k, csc, niter):
    indptr, indices, vals = csc
    nnz = int(indices.size)
    e = pymf_b200.Engine(d, n, k)
    try:
        t0 = time.perf_counter()
        e.upload_x_csc(indptr, indices, vals)
        upload_s = time.perf_counter() - t0
        rate = time_iters(e, niter)
        e.kernel_timing(True)
        e.enqueue(niter); e.sync()
        s0, _ = e.kernel_timing_read(0)
        s1, _ = e.kernel_timing_read(1)
        e.kernel_timing(False)
        split = kernel_split(e, 3)
        model = 16.0 * nnz + 8.0 * k * n              # kp = k at these shapes (multiples of 32)
        dense_kkn = sum(v for kname, v in split.items() if "k_gh" in kname or "k_ltr_partial" in kname or "k_sum_partials" in kname)
        return {"nnz": nnz, "upload_s": upload_s, "it_per_s": rate, "h_update_ms": s0, "xht_hht_ms": s1,
                "dense_kkn_ms": dense_kkn, "kernels_ms": split, "model_bytes": model,
                "achieved_GBps": model / ((s0 + s1) * 1e-3) / 1e9}
    finally:
        e.close()


def run_dense(d, n, k, csc, niter):
    indptr, indices, vals = csc
    dev = torch.device("cuda")
    X = torch.zeros(d, n, dtype=torch.float32, device=dev)
    ip = torch.from_numpy(indptr).to(dev)
    cols = torch.repeat_interleave(torch.arange(n, device=dev), ip[1:] - ip[:-1])
    X[torch.from_numpy(indices).to(dev).long(), cols] = torch.from_numpy(vals).to(dev)
    e = pymf_b200.Engine(d, n, k)
    try:
        e.bind_x_device(X.data_ptr(), X.stride(0), keepalive=X)
        return {"path": e.active_path, "it_per_s": time_iters(e, niter)}
    finally:
        e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--niter", type=int, default=20)
    a = ap.parse_args()
    res = {"meta": gpu_info(), "copy_GBps": copy_rate() / 1e9, "shapes": []}
    print(json.dumps(res["meta"]), flush=True)
    for name, d, n, dens, pl, k in SHAPES:
        csc = make_csc(d, n, dens, pl, 7)
        r = {"name": name, "d": d, "n": n, "k": k, "density": dens, "power_law": pl}
        r.update(run_sparse(d, n, k, csc, a.niter))
        print(json.dumps(r), flush=True)
        res["shapes"].append(r)
        del csc
    d, n, k = 4096, 262144, 32
    for dens in DENSITIES:
        csc = make_csc(d, n, dens, False, 8)
        r = {"name": "cfg2_%g" % dens, "d": d, "n": n, "k": k, "density": dens, "power_law": False}
        r.update(run_sparse(d, n, k, csc, a.niter))
        r["dense"] = run_dense(d, n, k, csc, a.niter)
        print(json.dumps(r), flush=True)
        res["shapes"].append(r)
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
