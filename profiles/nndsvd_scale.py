"""Time NNDSVD.factorize() at user-sized shapes, CUDA-core passes against tensor-core passes (DESIGN 5.7).

    python profiles/nndsvd_scale.py --out profiles/nndsvd_scale.json                      # one GPU
    torchrun --nproc-per-node=N profiles/nndsvd_scale.py --dist --out profiles/nndsvd_scale_nN.json

Data: the planted-low-rank recipe of oracle.cases.build_nndsvd, generated on the device with torch's seeded generator:
X = Ws Hs + 0.02 U[0,1) with Ws = U * (U < 0.5) * scale (d x r), Hs = U * (U < 0.5) (r x n), r = k + 16 and
scale_i = 0.75^(4 i / r): the leading k + 1 singular values stand above the noise (uniform data has a flat spectrum and
would time the sweep cap, not the method) and within 1e3 of the largest (the Cholesky of Y^T Y drops directions below
that, kernels_svd.cuh).  Under torchrun every rank builds its own columns of one d x n matrix.

Per run: a warm-up factorize() of a fresh object, then one timed factorize() (host clock ending in a device
synchronise).  The two pass families alternate in the same process, twice.  Reported: seconds, sweeps, ms per sweep and
the X bytes two passes stream per sweep over the time of a sweep; the outputs of the two families compared (rel W,
rel H, sigma); the settled sweep-to-sweep change of the Ritz values (25 sweeps, no stop).
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

SHAPES_1GPU = [("cfg2", 4096, 262144, 32), ("cfg4_k64", 8192, 524288, 64), ("cfg4_k128", 8192, 524288, 128),
               ("cfg3_shard_n8", 16384, 131072, 128), ("below_2^24", 1024, 8192, 32)]
SHAPES_DIST = [("cfg3", 16384, 1 << 20, 128)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        name, power = [s.strip() for s in q[torch.cuda.current_device()].split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def planted_x(d, n, k, seed, col0=0, n_loc=None):
    """Columns [col0, col0 + n_loc) of the planted d x n matrix, built on the current device."""
    n_loc = n if n_loc is None else n_loc
    dev = torch.device("cuda", torch.cuda.current_device())
    r = k + 16
    g = torch.Generator(device=dev).manual_seed(seed)
    scale = torch.tensor(0.75 ** (4.0 * np.arange(r) / r), dtype=torch.float32, device=dev)
    Ws = torch.rand(d, r, generator=g, device=dev) * (torch.rand(d, r, generator=g, device=dev) < 0.5) * scale
    Hs = torch.empty(r, n_loc, device=dev)
    for c0 in range(0, n, 1 << 18):                      # the same draws on every rank: keep the local columns
        w = min(1 << 18, n - c0)
        blk = torch.rand(r, w, generator=g, device=dev) * (torch.rand(r, w, generator=g, device=dev) < 0.5)
        lo, hi = max(c0, col0), min(c0 + w, col0 + n_loc)
        if lo < hi:
            Hs[:, lo - col0:hi - col0] = blk[:, lo - c0:hi - c0]
    gn = torch.Generator(device=dev).manual_seed(seed + 1 + col0)
    X = torch.rand(d, n_loc, generator=gn, device=dev).mul_(0.02)
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    X.addmm_(Ws, Hs)
    torch.backends.cuda.matmul.allow_tf32 = prev
    del Ws, Hs
    torch.cuda.synchronize()
    return X


def one_run(X, k, path, dist_kw):
    m = pymf_b200.NNDSVD(X, num_bases=k, path=path, **dist_kw)
    m.factorize()                                        # warm-up: engine, plan, first touch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.factorize()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    res = dict(path=m.svd_path, seconds=sec, sweeps=int(m.svd_sweeps), ms_per_sweep=1e3 * sec / max(1, m.svd_sweeps),
               change_at_stop=float(m._engine.nndsvd_change))
    out = (m.W.copy(), m.H.copy(), m.singular_values.copy())
    return m, res, out


def rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def measure(name, d, n, k, dist_kw, rank=0, world=1):
    n_loc = [n // world + (1 if r < n % world else 0) for r in range(world)]
    col0 = sum(n_loc[:rank])
    X = planted_x(d, n, k, seed=2024, col0=col0, n_loc=n_loc[rank])
    bytes_sweep = 2.0 * d * n_loc[rank] * 4
    runs, outs = [], {}
    for rep in range(2):
        for path in ("simt", "tc"):
            m, res, out = one_run(X, k, path, dist_kw)
            res["x_GBps_per_sweep"] = bytes_sweep / (res["ms_per_sweep"] * 1e-3) / 1e9
            res["rep"] = rep
            runs.append(res)
            outs.setdefault(path, out)
            del m
    W0, H0, s0 = outs["simt"]
    W1, H1, s1 = outs["tc"]
    cmp = dict(rel_W=rel(W1, W0), rel_H_local=rel(H1, H0), max_rel_sigma=float(np.max(np.abs(s1 - s0) / s0)))
    settled = {}
    for path in ("simt", "tc"):                          # sweep-to-sweep change once the basis has settled
        m = pymf_b200.NNDSVD(X, num_bases=k, path=path, **dist_kw)
        m.factorize()
        m._engine.nndsvd(max_iter=25, tol=1e-30)
        settled[path] = float(m._engine.nndsvd_change)
        del m
    default = pymf_b200.NNDSVD(X, num_bases=k, **dist_kw)
    default.factorize()
    best = {p: min(r["seconds"] for r in runs if r["path"] == p) for p in ("simt", "tc")}
    del X
    torch.cuda.empty_cache()
    return dict(shape=name, d=d, n=n, k=k, world=world, n_local=n_loc[rank], default_path=default.svd_path,
                x_bytes_per_sweep=bytes_sweep, runs=runs, best_s=best, tc_speedup=best["simt"] / best["tc"],
                simt_vs_tc=cmp, settled_change_25_sweeps=settled)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--dist", action="store_true", help="under torchrun: column-sharded over all ranks")
    ap.add_argument("--only", default=None, help="comma-separated shape names")
    a = ap.parse_args()
    rank, world, dist_kw = 0, 1, {}
    if a.dist:
        import torch.distributed as dist
        rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
        dist_kw = dict(process_group=True, device=torch.cuda.current_device())
    shapes = SHAPES_DIST if a.dist else SHAPES_1GPU
    if a.only:
        shapes = [s for s in shapes if s[0] in a.only.split(",")]
    info = gpu_info()
    info["recipe"] = "X = Ws Hs + 0.02 U[0,1), r = k + 16, scale_i = 0.75^(4 i / r), torch seed 2024 (see docstring)"
    results = []
    for name, d, n, k in shapes:
        r = measure(name, d, n, k, dist_kw, rank, world)
        r.update(info)
        results.append(r)
        if rank == 0:
            print(json.dumps(dict(shape=name, world=world, best_s=r["best_s"], tc_speedup=round(r["tc_speedup"], 2),
                                  sweeps=[x["sweeps"] for x in r["runs"]], default=r["default_path"],
                                  cmp=r["simt_vs_tc"], settled=r["settled_change_25_sweeps"])), flush=True)
    if rank == 0:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)
    if a.dist:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
