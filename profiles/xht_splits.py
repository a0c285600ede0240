"""X H^T column splits without the 4 K-column cap, with L2 eviction priorities (DESIGN 5.1, 5.8).

    PYMFB_OUT=build_exp/libpymfb_parent.so pymf_b200/csrc/build.sh        # in a checkout of the parent commit
    python profiles/xht_splits.py --arm parent=build_exp/libpymfb_parent.so \\
        --arm parent_det=build_exp/libpymfb_parent.so:PYMFB_DETERMINISTIC=1 \\
        --arm new=pymf_b200/libpymfb.so --out profiles/xht_splits.json

Each --arm is NAME=LIBRARY[:VAR=VALUE,...]: a build of the library (PYMFB_LIB selects it) and the environment it runs
under.  The arms of the recorded run:
  parent        the parent commit: X H^T tasks capped at ~4 K columns (cfg3: 256 splits), over the 1 GiB budget of
                the partial copies on cfg3, cfg5 and cfg4 k >= 256, so fp32 atomics into a cleared P there;
  parent_det    the same build with PYMFB_DETERMINISTIC=1 (cfg3: 256 copies, 2.15 GB): the ordered combine on the
                short splits, which separates "no atomics" from "long splits + L2 priorities";
  new           no cap (cfg3: 37 splits), X loaded evict_first, [H_hi ; H_lo] evict_last in both X H^T kernels;
  new_h_normal  the same with the [H_hi ; H_lo] loads unhinted (default priority) in both kernels.
profiles/xht_splits_ts.json repeats the k <= 64 workloads with 5 runs per arm: parent; `new` = k_xht_ts with X
evict_first and H unhinted; `ts_x_plain` = k_xht_ts with neither hint.  This tree is `new` of xht_splits.json for
k_xht_tc (k >= 96: cfg3, cfg4 k >= 128) and `ts_x_plain` of xht_splits_ts.json for k_xht_ts (k <= 64: cfg2, cfg4 k = 64,
cfg5); each kernel serves only its own workloads.
Each (arm, workload) measurement runs in a process of its own, the arms alternating in a rotated order per repetition,
so that all see the same box in the same minutes.  Per measurement, on device-generated data (gen_x / gen_w / gen_h,
X far larger than L2): ms per full iteration (W update, H update, error; CUDA events around the enqueued iterations),
the H pass and the X H^T pass (pymfb_kernel_timing slots 0 and 1: the X H^T slot covers its launches and the ordered
sum of the copies, not the clear of P), the median SM clock over the timed window (NVML) and ||X - W H|| afterwards.
The card's name and power limit are read in the same call.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# name, d, n, k, timed iterations (each window ~0.5-1 s)
WORKLOADS = [("cfg3", 16384, 1 << 20, 128, 20), ("cfg2", 4096, 262144, 32, 400), ("cfg4k64", 8192, 524288, 64, 100),
             ("cfg4k128", 8192, 524288, 128, 60), ("cfg4k256", 8192, 524288, 256, 30), ("cfg4k512", 8192, 524288, 512, 20),
             ("cfg5", 32768, 524288, 64, 30)]


class Clock(threading.Thread):
    def __init__(self):
        threading.Thread.__init__(self, daemon=True)
        import pynvml
        pynvml.nvmlInit()
        self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(0)
        self.samples, self.stop = [], threading.Event()

    def run(self):
        while not self.stop.is_set():
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            self.stop.wait(0.01)


def child(d, n, k, iters):
    sys.path.insert(0, ROOT)
    import pymf_b200
    e = pymf_b200.Engine(d, n, k, path="tc")
    e.gen_x(1234); e.gen_w(1235); e.gen_h(1236)
    e.enqueue(5)
    e.sync()
    clk = Clock()
    e.kernel_timing(True)
    ev0, ev1 = e.event(), e.event()
    clk.start()
    e.record(ev0)
    e.enqueue(iters)
    e.record(ev1)
    e.sync()
    clk.stop.set(); clk.join()
    ms = e.elapsed_ms(ev0, ev1)
    h_ms, _ = e.kernel_timing_read(0)
    x_ms, _ = e.kernel_timing_read(1)
    e.kernel_timing(False)
    ferr = e.frobenius()
    e.close()
    print(json.dumps({"ms_per_step": ms / iters, "h_update_ms": h_ms, "xht_ms": x_ms,
                      "sm_clock_median_mhz": statistics.median(clk.samples) if clk.samples else None, "ferr": ferr}))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def parse_arm(s):
    name, rest = s.split("=", 1)
    lib, _, envs = rest.partition(":")
    env = dict(kv.split("=", 1) for kv in envs.split(",") if kv)
    return name, os.path.abspath(lib), env


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", action="append", default=[], help="NAME=LIBRARY[:VAR=VALUE,...]")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(w[0] for w in WORKLOADS))
    ap.add_argument("--out", required=True)
    ap.add_argument("--child", nargs=4, type=int, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(*a.child)
        return
    if not a.arm:
        ap.error("at least one --arm is needed")
    arms = [parse_arm(s) for s in a.arm]
    wls = [w for w in WORKLOADS if w[0] in a.workloads.split(",")]
    res = {"gpu": gpu_info(), "arms": {nm: {"lib": os.path.relpath(lib, ROOT), "env": env} for nm, lib, env in arms},
           "runs": []}
    for rep in range(a.reps):
        for name, d, n, k, iters in wls:
            for i in range(len(arms)):
                arm, lib, extra = arms[(i + rep) % len(arms)]
                env = dict(os.environ, PYMFB_LIB=lib, **extra)
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--out", a.out,
                                    "--child", str(d), str(n), str(k), str(iters)], env=env, capture_output=True, text=True)
                if p.returncode != 0:
                    sys.exit("%s on %s failed:\n%s" % (arm, name, p.stderr[-3000:]))
                r = dict(json.loads(p.stdout.strip().splitlines()[-1]), rep=rep, workload=name, d=d, n=n, k=k, arm=arm)
                print(json.dumps(r), flush=True)
                res["runs"].append(r)
    summary = {}
    for name, *_ in wls:
        for arm, _, _ in arms:
            rs = [r for r in res["runs"] if r["workload"] == name and r["arm"] == arm]
            summary["%s/%s" % (name, arm)] = {key: [None if r[key] is None else round(r[key], 3) for r in rs]
                                              for key in ("ms_per_step", "h_update_ms", "xht_ms", "sm_clock_median_mhz")}
            summary["%s/%s" % (name, arm)]["ferr"] = [r["ferr"] for r in rs]
    res["summary"] = summary
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
