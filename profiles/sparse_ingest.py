"""Time the upload of sparse X (DESIGN 5.9) by route, on the two user-sized shapes of profiles/sparse_scale.py.

    python profiles/sparse_ingest.py --out profiles/sparse_ingest.json

Per shape the same matrix (the recipe of sparse_scale.make_csc) goes through four routes into one engine:
  coo    torch COO arrays on the device, uncoalesced: entries shuffled, plus about 1 % duplicate entries (a copy of a
         random 1 % of the entries, with the values split so the sums equal the matrix)  -> upload_x_sparse_device
  csr    torch CSR arrays on the device (int64)                                           -> upload_x_sparse_device
  csc    torch CSC arrays on the device (int64)                                           -> upload_x_sparse_device
  scipy  the host route of NMF(..., sparse=True): tocsc(copy=True), sum_duplicates(), upload_x_csc
Every timing is a host clock around the call, ending in a device synchronise.  Each route is warmed up once, then the
routes alternate for --rounds rounds and the best time is kept.  Peak device memory of a device route: the lowest
free memory (cudaMemGetInfo, sampled by a second thread every ~0.2 ms during the call) below the free memory before
the call, which covers the previous X being replaced only after the new one is built; the increase left after the call
is reported next to it.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import scipy.sparse as sps
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
import pymf_b200  # noqa: E402
from sparse_scale import gpu_info, make_csc  # noqa: E402

SHAPES = [("text_k64", 1 << 17, 1 << 20, 0.0005, False, 64), ("cell_k32", 1 << 15, 1 << 19, 0.03, True, 32)]


def device_inputs(d, n, csc, seed):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(seed)
    indptr, indices, vals = (torch.from_numpy(a).to(dev) for a in csc)
    nnz = indices.numel()
    cols = torch.repeat_interleave(torch.arange(n, device=dev), indptr[1:] - indptr[:-1])
    rows = indices.long()
    out = {"csc": (indptr, indices.long(), vals)}                  # int64 pointers and rows
    order = torch.argsort(rows * n + cols)                          # CSR: by (row, column)
    out["csr"] = (torch.searchsorted(rows[order], torch.arange(d + 1, device=dev)), cols[order].contiguous(),
                  vals[order].contiguous())
    dup = torch.randperm(nnz, generator=g, device=dev)[:nnz // 100]
    v = vals.clone()
    v[dup] *= 0.5
    r, c, v = torch.cat([rows, rows[dup]]), torch.cat([cols, cols[dup]]), torch.cat([v, v[dup]])
    perm = torch.randperm(r.numel(), generator=g, device=dev)
    out["coo"] = (r[perm].contiguous(), c[perm].contiguous(), v[perm].contiguous())
    del order, perm, r, c, v, cols, rows
    torch.cuda.synchronize()
    return out


class FreeSampler(object):
    def __init__(self):
        self.low, self.stop = None, False

    def run(self):
        while not self.stop:
            f = torch.cuda.mem_get_info()[0]
            self.low = f if self.low is None else min(self.low, f)
            time.sleep(0.0002)


def time_device(e, layout, arrays):
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info()[0]
    s = FreeSampler()
    th = threading.Thread(target=s.run)
    th.start()
    t0 = time.perf_counter()
    e.upload_x_sparse_device(layout, *arrays)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    s.stop = True
    th.join()
    free1 = torch.cuda.mem_get_info()[0]
    return dt, free0 - min(s.low, free1), free0 - free1


def time_scipy(e, X):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m = X.tocsc(copy=True)
    m.sum_duplicates()
    e.upload_x_csc(np.ascontiguousarray(m.indptr, dtype=np.int64), np.ascontiguousarray(m.indices, dtype=np.int32),
                   np.ascontiguousarray(m.data))
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    res = {"meta": gpu_info(), "rounds": a.rounds, "shapes": []}
    print(json.dumps(res["meta"]), flush=True)
    for name, d, n, dens, pl, k in SHAPES:
        csc = make_csc(d, n, dens, pl, 7)
        X = sps.csc_matrix((csc[2], csc[1], csc[0]), shape=(d, n))
        dev = device_inputs(d, n, csc, 8)
        e = pymf_b200.Engine(d, n, k)
        times = {r: [] for r in ("coo", "csr", "csc", "scipy")}
        peak, left = {}, {}
        try:
            for rnd in range(a.rounds + 1):                        # round 0 is the warm-up
                for route in ("coo", "csr", "csc", "scipy"):
                    if route == "scipy":
                        dt = time_scipy(e, X)
                    else:
                        dt, pk, lf = time_device(e, route, dev[route])
                        peak[route] = max(peak.get(route, 0), pk)
                        left[route] = lf
                    if rnd > 0:
                        times[route].append(dt)
        finally:
            e.close()
        r = {"name": name, "d": d, "n": n, "k": k, "density": dens, "power_law": pl, "nnz": int(csc[1].size),
             "coo_entries": int(dev["coo"][0].numel()),
             "best_s": {k_: min(v) for k_, v in times.items()}, "all_s": times,
             "peak_extra_bytes": peak, "bytes_left_after_upload": left}
        print(json.dumps(r), flush=True)
        res["shapes"].append(r)
        del dev, X, csc
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
