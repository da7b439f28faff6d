"""Cost of a rescan: host wall time of kvg_rescan_pci against kvg_scan_pci on the same snapshot (10,000 and
1,000,000 records), of kvg_rescan_mdev against kvg_scan_mdev (65,536 mdevs), and the device time of the two diff
kernels (rescan_merge, rescan_keys) from the per-kernel timing pass.

Every tick's snapshot is seeded churn over the oracle generator: gen_pci(0, N) with a seeded 0.1 % of the
records hidden (records appear and disappear between ticks), a few driver flips and a few numa / group rewrites
(moves); mdevs the same over gen_mdev.  Snapshots are host arrays, as the plugin passes them.  One JSON object on
stdout (and to --out), with the card's name and power limit read in the same run.

    python tools/time_rescan.py [--ticks 200] [--out profiles/time_rescan.json]
"""
import argparse
import ctypes as C
import gzip
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "kubevirt-gpu-device-plugin_b200")]
import kvgpu  # noqa: E402
from oracle import oracle as O  # noqa: E402


def churn_pci(base, t, frac=0.001):
    rng = np.random.default_rng(1000 + t)
    keep = rng.random(len(base)) >= frac
    recs = base.copy()
    k = max(1, len(base) // 5000)
    flip = rng.choice(len(base), k, replace=False)
    recs["driver"][flip] = np.where(recs["driver"][flip] == 1, 3, 1)
    mv = rng.choice(len(base), k, replace=False)
    recs["numa"][mv[: k // 2 + 1]] ^= 1
    recs["iommu_group"][mv[k // 2:]] += 7
    return np.ascontiguousarray(recs[keep])


def churn_mdev(base, t, n_types, frac=0.001):
    rng = np.random.default_rng(2000 + t)
    keep = rng.random(len(base)) >= frac
    recs = base.copy()
    k = max(1, len(base) // 5000)
    mv = rng.choice(len(base), 3 * k, replace=False)
    recs["parent_numa"][mv[:k]] ^= 1
    recs["parent"][mv[k:2 * k]] += 1
    recs["type_idx"][mv[2 * k:]] = rng.integers(0, n_types, k)
    return np.ascontiguousarray(recs[keep])


def pct(xs, p):
    return float(np.percentile(np.asarray(xs) * 1e6, p))


def wall(fn, ticks):
    """host wall time per call (each call ends in a device synchronise: the result is on the host)"""
    out = []
    for t in range(ticks):
        t0 = time.perf_counter()
        fn(t)
        out.append(time.perf_counter() - t0)
    return out


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ticks", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    text = gzip.open(os.path.join(ROOT, "tests", "golden", "pci.ids.gz"), "rb").read()
    ids = O.nv_ids(text)
    res = {"card": card(), "ticks": args.ticks, "unit": "us", "pci": {}, "mdev": {}, "kernels_us": {}}
    ctx = kvgpu.Context(0)
    ctx.pciids_load(text)
    lib, h = kvgpu.load(), ctx.handle
    for n in (10_000, 1_000_000):
        base = O.gen_pci(0, n, ids, 16)
        snaps = [churn_pci(base, t) for t in range(min(args.ticks, 50))]
        S = len(snaps)
        for t in range(5):                                 # warm-up: both shapes, both entry points
            ctx.rescan_pci(snaps[t % S])
            ctx.scan_pci(snaps[t % S])
        # the raw C calls: the Python result copies are not part of what a caller of the C-ABI pays
        pr, sr = C.POINTER(kvgpu._lib.PciRescanC)(), C.POINTER(kvgpu._lib.PciResultC)()

        def rescan(t):
            s = snaps[t % S]
            assert lib.kvg_rescan_pci(h, s.ctypes.data, len(s), C.byref(pr)) == 0
            lib.kvg_result_free(pr)

        def scan(t):
            s = snaps[t % S]
            assert lib.kvg_scan_pci(h, s.ctypes.data, len(s), C.byref(sr)) == 0
            lib.kvg_result_free(sr)
        # alternate the two in blocks so that both see the same host and device conditions
        tr, ts = [], []
        for blk in range(0, args.ticks, 10):
            tr += wall(lambda t: rescan(blk + t), 10)
            ts += wall(lambda t: scan(blk + t), 10)
        res["pci"][str(n)] = {"rescan_p50": pct(tr, 50), "rescan_p99": pct(tr, 99),
                              "scan_p50": pct(ts, 50), "scan_p99": pct(ts, 99)}
        ctx.set_kernel_timing(True)
        per = {}
        for t in range(10):
            ctx.rescan_pci(snaps[t % S])
            for name, ms in ctx.kernel_times():
                if name.startswith("rescan_"):
                    per.setdefault(name, []).append(ms * 1e3)
        ctx.set_kernel_timing(False)
        res["kernels_us"]["pci_%d" % n] = {k: float(np.median(v)) for k, v in per.items()}
    types = O.gen_type_names(256)
    mbase = O.gen_mdev(0, 65_536)
    msnaps = [churn_mdev(mbase, t, 256) for t in range(min(args.ticks, 50))]
    S = len(msnaps)
    for t in range(5):
        ctx.rescan_mdev(msnaps[t % S], types)
        ctx.scan_mdev(msnaps[t % S], types)
    td, keep = ctx._type_dict(types)
    mr, ms_ = C.POINTER(kvgpu._lib.MdevRescanC)(), C.POINTER(kvgpu._lib.MdevResultC)()

    def mrescan(t):
        s = msnaps[t % S]
        assert lib.kvg_rescan_mdev(h, s.ctypes.data, len(s), C.byref(td), C.byref(mr)) == 0
        lib.kvg_result_free(mr)

    def mscan(t):
        s = msnaps[t % S]
        assert lib.kvg_scan_mdev(h, s.ctypes.data, len(s), C.byref(td), C.byref(ms_)) == 0
        lib.kvg_result_free(ms_)
    tr, ts = [], []
    for blk in range(0, args.ticks, 10):
        tr += wall(lambda t: mrescan(blk + t), 10)
        ts += wall(lambda t: mscan(blk + t), 10)
    res["mdev"]["65536"] = {"rescan_p50": pct(tr, 50), "rescan_p99": pct(tr, 99), "scan_p50": pct(ts, 50),
                            "scan_p99": pct(ts, 99)}
    ctx.set_kernel_timing(True)
    per = {}
    for t in range(10):
        ctx.rescan_mdev(msnaps[t % S], types)
        for name, ms in ctx.kernel_times():
            if name.startswith("rescan_"):
                per.setdefault(name, []).append(ms * 1e3)
    ctx.set_kernel_timing(False)
    res["kernels_us"]["mdev_65536"] = {k: float(np.median(v)) for k, v in per.items()}
    ctx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
