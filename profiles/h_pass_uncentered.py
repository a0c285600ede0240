"""Cost of the uncentered TS H-update pass (k <= 64, DESIGN 5.1) against the centered one it replaced.

    python profiles/h_pass_uncentered.py --old-lib path/to/parent/libpymfb.so --out profiles/h_pass_uncentered.json

The old library is a build of the parent commit (centered operands, 8-stage segments); the new one is this tree's
(uncentered operands, C drained every 64 rows).  Each (library, shape) measurement runs in a process of its own
(PYMFB_LIB selects the build), the two libraries alternating, so that both see the same box in the same minutes.
Per measurement, on device-generated data (gen_x / gen_w / gen_h, X far larger than L2):
the H pass (pymfb_kernel_timing slot 0, averaged over H-only iterations after a warm-up) and iterations/s of the full
iteration (W update, H update, trace-identity error; CUDA events around the enqueued iterations).
The card's name and power limit are read in the same call.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = [("cfg2", 4096, 262144, 32, 600, 300), ("cfg4_k64", 8192, 524288, 64, 150, 100)]


def child(d, n, k, h_iters, iters):
    sys.path.insert(0, ROOT)
    import pymf_b200
    e = pymf_b200.Engine(d, n, k, path="tc")
    e.set_err_mode("trace")
    e.gen_x(1); e.gen_w(2); e.gen_h(3)
    e.run(3, early_stop=False)
    e.kernel_timing(True)
    e.enqueue(h_iters, compute_w=False, compute_err=False)
    e.sync()
    h_ms, h_cnt = e.kernel_timing_read(0)
    e.kernel_timing(False)
    e.enqueue(5)
    ev0, ev1 = e.event(), e.event()
    e.record(ev0)
    e.enqueue(iters)
    e.record(ev1)
    e.sync()
    ms = e.elapsed_ms(ev0, ev1)
    e.close()
    print(json.dumps({"h_pass_ms": h_ms, "h_pass_count": h_cnt, "it_per_s": iters / (ms / 1e3), "ms_per_iter": ms / iters}))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old-lib", required=True)
    ap.add_argument("--new-lib", default=os.path.join(ROOT, "pymf_b200", "libpymfb.so"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", required=True)
    ap.add_argument("--child", nargs=5, type=int, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(*a.child)
        return
    res = {"gpu": gpu_info(), "runs": []}
    for rep in range(a.reps):
        for name, d, n, k, h_iters, iters in SHAPES:
            for which, lib in (("old_centered", a.old_lib), ("new_uncentered", a.new_lib)):
                env = dict(os.environ, PYMFB_LIB=os.path.abspath(lib))
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--old-lib", a.old_lib, "--out", a.out,
                                      "--child", str(d), str(n), str(k), str(h_iters), str(iters)],
                                     env=env, capture_output=True, text=True, check=True).stdout
                r = dict(json.loads(out.strip().splitlines()[-1]), rep=rep, shape=name, d=d, n=n, k=k, code=which)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
    summary = {}
    for name, *_ in SHAPES:
        for which in ("old_centered", "new_uncentered"):
            rs = [r for r in res["runs"] if r["shape"] == name and r["code"] == which]
            summary["%s/%s" % (name, which)] = {
                "h_pass_ms": [round(r["h_pass_ms"], 4) for r in rs], "it_per_s": [round(r["it_per_s"], 1) for r in rs]}
    res["summary"] = summary
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
