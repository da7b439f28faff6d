#!/usr/bin/env python3
"""bench.py — the discovery-scan benchmark (contract: see the task statement / DESIGN.md §Measurement).

  python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--records R] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input:
  parse the full utils/pci.ids image (1,536,458 B) into the name table  +  classify / compact /
  bucket R synthetic PCI records (default 1,000,000 = BASELINE.json configs[1]).
N > 1 (torchrun, one rank per GPU): every rank owns R records (weak scaling), classifies its shard, keeps
its survivors (its part of bdfToIommuMap) and sends every survivor once per map to the owner of its key
(stores into the owners' peer windows over NVLink; --exchange nccl for the fallback); every rank buckets
the keys it owns.  Before anything is timed every rank checks its part of the result against a numpy
restatement of the oracle ("parity" in the JSON line; a mismatch aborts the run).

value   records/s with inputs resident in HBM (CUDA events on the launching stream, L2 flushed
        between steps, max over ranks)
e2e     the same metric through the reference-facing C-ABI calls (kvg_pciids_load + kvg_scan_pci)
        with PINNED HOST buffers in and host results out, copies inside the timed region

--dump-outputs DIR writes the result of the last timed step, as a caller of the scan receives it, to
DIR/<name>.npy (float64, one file per array; N > 1: every rank its own part, prefixed rank<r>_).  The
inputs depend on the arguments only, so two builds can be compared array for array.
"""
import argparse
import gzip
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "kubevirt-gpu-device-plugin_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "PCI device records classified/sec (pci.ids parse + classify + bucket per step)"
GROUP_BITS_FOR = lambda n: max(1, int(np.ceil(np.log2(max(2, n // 2)))))


def load_pciids() -> bytes:
    return gzip.open(os.path.join(ROOT, "tests", "golden", "pci.ids.gz"), "rb").read()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4)
                          if r[2 + i].lower().startswith("active")})
        csv_path = os.environ.get("KVG_CLOCKS_CSV")   # evidence: the raw samples behind the medians
        if csv_path:
            try:
                with open(csv_path, "w") as f:
                    f.write(self.Q + "\n")
                    for r in self.rows:
                        f.write(",".join(r) + "\n")
            except OSError:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_baseline(text, ids, sample, threads):
    """Oracle port timed on this box's host cores (checker code used as the CPU yardstick only)."""
    from oracle import oracle as O
    recs = O.gen_pci(0, sample, ids, GROUP_BITS_FOR(sample))
    ta, sa, _ = O.bench_faithful(recs, text)
    tb, sb, _ = O.bench_threads(recs, text, threads)
    assert sa == sb
    return {"value": sample / ta, "unit": "records/s", "cores": 1, "kind": "port",
            "sample": "%d synthetic PCI records + one getDeviceName pci.ids scan per distinct "
                      "device id (faithful-cost restatement of device_plugin.go:187-247,371-438, "
                      "logging off), %.2f s" % (sample, ta),
            "best_effort_mt": {"value": sample / tb, "unit": "records/s", "cores": threads,
                               "seconds": tb,
                               "what": "parse-once + %d threads + counting/radix merge" % threads},
            "host_cores": os.cpu_count()}


def _expect_survivors(recs):
    """numpy restatement of the classification (device_plugin.go:201-244) on the oracle generator's records:
    survivors in Walk order as (addr, iommu_group, device, numa)."""
    alive = (recs["vendor"] == 0x10de) & ((recs["flags"] & 15) == 0) & ((recs["driver"] == 1) | (recs["driver"] == 2))
    s = recs[alive]
    numa = np.where(((s["flags"] & 16) != 0) | (s["numa"] < 0), 0, s["numa"]).astype(np.uint16)
    return s["addr"], s["iommu_group"], s["device"], numa


def _check_members(got, exp, sel, what):
    addr, grp, dev, numa = exp
    ok = (len(got) == int(sel.sum()) and np.array_equal(got["addr"], addr[sel]) and
          np.array_equal(got["iommu_group"], grp[sel]) and np.array_equal(got["device"], dev[sel]) and
          np.array_equal(got["numa"], numa[sel]))
    if not ok:
        raise AssertionError("parity: %s differ from the CPU restatement" % what)


def _check_ordering(members, field, keys, off, perm, what):
    k = members[field].astype(np.int64)
    order = np.argsort(k, kind="stable")
    uk, first = np.unique(k[order], return_index=True)
    if not (np.array_equal(keys.astype(np.int64), uk) and np.array_equal(off[:-1].astype(np.int64), first) and
            int(off[-1]) == len(k) and np.array_equal(perm.astype(np.int64), order)):
        raise AssertionError("parity: %s ordering differs from a stable sort" % what)


def check_parity(ctx, sharded, rank, world, n, ids, gbits, text, O):
    """Exact check of THIS run's output before anything is timed.  N = 1: the fetched result of kvg_dev_scan_pci;
    N > 1: this rank's part of the sharded scan — its shard's survivors, and ALL members of the device ids /
    iommu groups it owns (key % N == rank), both orderings — against a numpy group-by of the same synthetic
    records (oracle generator) over ALL shards.  Raises on the first difference."""
    exp = _expect_survivors(O.gen_pci(0, n * world, ids, gbits))
    addr, grp, dev, numa = exp
    if sharded is None:
        res = ctx.dev_scan_pci_fetch()
        _check_members(res.survivors, exp, np.ones(len(addr), bool), "survivors")
        dev_res = grp_res = res
    else:
        res = sharded.fetch()
        lo = np.searchsorted(addr, rank * n), np.searchsorted(addr, (rank + 1) * n)   # addr == Walk index here
        sel = np.zeros(len(addr), bool)
        sel[lo[0]:lo[1]] = True
        _check_members(res.local, exp, sel, "rank %d shard survivors" % rank)
        _check_members(res.dev.survivors, exp, dev.astype(np.int64) % world == rank, "rank %d owned deviceMap members" % rank)
        _check_members(res.grp.survivors, exp, grp.astype(np.int64) % world == rank, "rank %d owned iommuMap members" % rank)
        dev_res, grp_res = res.dev, res.grp
    _check_ordering(dev_res.survivors, "device", dev_res.dev_keys, dev_res.dev_off, dev_res.dev_perm, "deviceMap")
    _check_ordering(grp_res.survivors, "iommu_group", grp_res.grp_keys, grp_res.grp_off, grp_res.grp_perm, "iommuMap")
    for k in range(0, len(dev_res.dev_keys), max(1, len(dev_res.dev_keys) // 48)):   # the name join, sampled
        key = b"%04x" % int(dev_res.dev_keys[k])
        if dev_res.name_at(int(dev_res.dev_name_slot[k])) != O.get_device_name(text, key):
            raise AssertionError("parity: resource name of device id %s differs from the oracle" % key.decode())
    return {"status": "ok", "checked": ("survivor list, both orderings (keys, offsets, stable permutation) and a "
                                        "sample of joined names" if sharded is None else
                                        "this rank's shard survivors, all members of the keys it owns, both "
                                        "orderings and a sample of joined names; every rank checks its own part"),
            "against": "numpy group-by of the oracle generator's records + oracle getDeviceName",
            "survivors_global": int(len(addr))}


DUMP_BYTES = 60_000_000   # array data of one --dump-outputs run: under 64 MB with the .npy headers


def result_arrays(res, prefix="", maps=("dev", "grp")):
    """The arrays of a PciResult: one per survivor field, the orderings of `maps`, and with the device-id
    ordering the name slots and the name pool they point into."""
    out = {prefix + "survivors_" + f: res.survivors[f] for f in res.survivors.dtype.names}
    for m in maps:
        for f in ("keys", "off", "perm") + (("name_slot",) if m == "dev" else ()):
            out["%s%s_%s" % (prefix, m, f)] = getattr(res, "%s_%s" % (m, f))
    if "dev" in maps:
        out[prefix + "name_pool"] = np.frombuffer(res.name_pool, dtype=np.uint8)
    return out


def last_step_arrays(ctx, sharded, rank):
    """What the last scan handed its caller: the fetched result (N = 1), or this rank's part of the sharded
    result (its shard's survivors and the members and orderings of the keys it owns)."""
    if sharded is None:
        return result_arrays(ctx.dev_scan_pci_fetch())
    res = sharded.fetch()
    out = {"local_" + f: res.local[f] for f in res.local.dtype.names}
    out.update(result_arrays(res.dev, "devmap_", ("dev",)))
    out.update(result_arrays(res.grp, "grpmap_", ("grp",)))
    return {"rank%d_%s" % (rank, k): v for k, v in out.items()}


def dump_outputs(out_dir, arrays, budget):
    """One float64 .npy per array (exact for every integer the scan returns).  Past `budget` bytes in all,
    every array keeps the same fraction of its elements, at indices drawn from a fixed seed, so two builds
    that compute the same result write the same files."""
    os.makedirs(out_dir, exist_ok=True)
    total = 8 * sum(a.size for a in arrays.values())
    keep = budget / total if total > budget else 1.0
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float64)
        if keep < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm (oracle port; the Go binary cannot be
    built in this image) on the host cores, bounded sample per step."""
    if rank != 0:
        return
    from oracle import oracle as O
    text = load_pciids()
    ids = O.nv_ids(text)
    sample = min(args.records, args.ref_sample) if args.ref_sample else args.records
    recs = O.gen_pci(0, sample, ids, GROUP_BITS_FOR(sample))
    for _ in range(min(args.warmup, 1)):
        O.bench_faithful(recs, text)
    times = []
    for _ in range(args.steps):
        t, _, _ = O.bench_faithful(recs, text)
        times.append(t)
    tot = sum(times)
    value = sample * len(times) / tot
    tb, _, _ = O.bench_threads(recs, text, os.cpu_count() or 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "records/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u32 (byte + integer)", "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[1]: full pci.ids (1,536,458 B) name lookups + %d synthetic PCI "
                               "records per step%s" % (sample, "" if sample == args.records else
                                                       " (bounded sample of %d)" % args.records),
                   "records_per_step": sample, "same_config_as_gpu_arm": sample == args.records},
        "cpu_baseline": {"value": value, "unit": "records/s", "cores": 1, "kind": "port",
                         "sample": "%d records/step x %d steps, faithful-cost C restatement of the "
                                   "Go scan (single goroutine in the reference => 1 thread)" % (
                                       sample, len(times)),
                         "best_effort_mt": {"value": sample / tb, "cores": os.cpu_count()},
                         "host_cores": os.cpu_count()},
        "e2e": {"value": value, "unit": "records/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--records", type=int, default=1_000_000, help="PCI records per rank per step")
    ap.add_argument("--ref-sample", type=int, default=0,
                    help="records per step of the reference arm (0 = the full --records workload: same config)")
    ap.add_argument("--cpu-sample", type=int, default=200_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config-3 / config-5 legs")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: transport of the exchange by owner — stores into the owners' peer windows over NVLink "
                         "(default), or the NCCL fallback a deployment without peer access gets")
    ap.add_argument("--config4", action="store_true",
                    help="run the config-4 leg (12 M PCI + 0.5 M mdev records per rank) at any N > 1, not only at N = 8")
    ap.add_argument("--big-records", type=int, default=1 << 24,
                    help="records for the HBM-bound roofline leg (N=1 only; 0 disables)")
    ap.add_argument("--big-files", type=int, default=256,
                    help="pci.ids images for the HBM-bound parse roofline leg (0 disables)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU scan's result; the reference arm has none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import kvgpu
    from oracle import oracle as O  # generator twin + cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    text = load_pciids()
    ids = O.nv_ids(text)
    n = args.records
    gbits = GROUP_BITS_FOR(n * world)
    hbm_peak, peak_src = peaks()

    ctx = kvgpu.Context(local_rank)
    ext = torch.cuda.ExternalStream(ctx.stream, device=local_rank)

    # ---- inputs resident in HBM
    pad = ctx.text_pad(len(text))
    h_text = np.full(pad + 16, 10, dtype=np.uint8)
    h_text[:len(text)] = np.frombuffer(text, dtype=np.uint8)
    d_text = torch.from_numpy(h_text).cuda()
    d_recs = torch.empty(max(n, 1) * 16, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    ctx.dev_gen_pci(d_recs.data_ptr(), rank * n, n, ids, gbits)
    ctx.dev_pciids_parse(d_text.data_ptr(), len(text), pad + 16, 1)

    sharded = None
    if world > 1:
        def bcast(b, src):
            t = torch.zeros(128, dtype=torch.uint8, device="cuda")
            if rank == src:
                t.copy_(torch.frombuffer(bytearray(b), dtype=torch.uint8))
            dist.broadcast(t, src)
            return bytes(t.cpu().numpy().tobytes())
        def allgather(b):
            t = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
            outs = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(outs, t)
            return [bytes(o.cpu().numpy().tobytes()) for o in outs]
        use_p2p = args.exchange == "p2p"
        run_c4 = not args.no_extra and (world == 8 or args.config4)
        c4_pci, c4_mdev = (12_000_000, 500_000) if run_c4 else (0, 0)
        sharded = kvgpu.ShardedScan(ctx, rank, world, bcast, allgather if use_p2p else None,
                                    max(n, c4_pci, 2 * c4_mdev) + 1)

    def step():
        ctx.dev_pciids_parse(d_text.data_ptr(), len(text), pad + 16, 1)
        if sharded:
            sharded.scan_device_shard(d_recs.data_ptr(), n)
        else:
            ctx.dev_scan_pci(d_recs.data_ptr(), n)

    def sync_all():
        ctx.dev_scan_pci_count()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        ctx.dev_flush_l2()
        step()
    sync_all()
    S, KD, G = ctx.dev_scan_pci_count()
    # ---- parity of what is about to be timed (every rank checks its own part; a mismatch aborts the run)
    parity = check_parity(ctx, sharded, rank, world, n, ids, gbits, text, O)
    if world > 1:
        flags = [None] * world
        dist.all_gather_object(flags, parity["status"])
        assert all(f == "ok" for f in flags)

    # ---- timed region: K steps, CUDA events on the launching stream, L2 flushed between steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    evs = []
    sync_all()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.dev_flush_l2()  # untimed: outside the event bracket
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(ext)
        step()
        e1.record(ext)
        evs.append((e0, e1))
    sync_all()
    t_wall = time.perf_counter() - t_wall0
    launches = ctx.launch_count - launches0 - args.steps  # minus the flush fills
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step_arrays(ctx, sharded, rank), DUMP_BYTES // world)
    if world > 1:
        t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms = float(t.item())
    ms_per_step = dev_ms / args.steps
    value = n * world / (ms_per_step * 1e-3)

    # ---- per-kernel times (separate pass, events around every launch) -> roofline
    ctx.set_kernel_timing(True)
    per = {}
    passes = max(3, min(args.steps, 10))
    for _ in range(passes):
        ctx.dev_flush_l2()
        ctx.set_kernel_timing(True)
        step()
        for name, ms in ctx.kernel_times():
            per.setdefault(name, []).append(ms)
    ctx.set_kernel_timing(False)
    ksum = {k: sum(v) / passes for k, v in per.items()}          # ms per step per kernel name
    kavg = {k: sum(v) / len(v) for k, v in per.items()}          # ms per launch
    nl = {k: len(v) / passes for k, v in per.items()}            # launches per step
    S, KD, G = ctx.dev_scan_pci_count()
    info = ctx.pciids_info()
    # members each ordering sorts on this rank: all survivors (N = 1) or the members of the owned keys
    S_ord = S if not sharded else parity["survivors_global"] // world
    import ctypes as _C
    _np, _sh, _bt = _C.c_uint32(), (_C.c_uint32 * 4)(), (_C.c_uint32 * 4)()
    kvgpu.load().kvg_debug_radix_plan((1 << int(gbits)) - 1 if gbits else max(n // 2, 1), 32,
                                      8 if n >= (8 << 20) else 11, _C.byref(_np), _sh, _bt)
    grp_passes = max(1, int(_np.value))
    # IMPLEMENTATION bytes per step of every kernel family (what this implementation moves; the CONTRACT
    # figure of SURVEY.md 8(d), 16 N + 24 S per scan, is reported separately as whole_scan_contract)
    algo = {
        "pciids_parse": len(text) + 16 * ((len(text) + 4095) // 4096),   # text once + one 16-byte summary per span
        "classify_compact": 16 * n + 16 * S,                   # every record read, every survivor written
        "order_hist": 4 * S_ord * 2 + 8 * S_ord * (1 + (grp_passes - 1)),
        "order_scatter": 16 * S_ord * (2 + grp_passes),        # 8 B read + 8 B written per pair per pass
        "order_final": (8 * S_ord + 4 * S_ord) * 2 + 8 * (KD + G),
        "shard_send": 16 * S * 3,                              # survivors read, one record stored per ordering
        "classify_send": 16 * n + 16 * S * 3,                  # records read; survivor stored locally + once per ordering
        "shard_gather": 2 * 32 * S_ord,                        # window regions -> dense owned lists
    }
    main_kernels = [k for k in algo if k in ksum]
    dominant = max(main_kernels, key=lambda k: ksum.get(k, 0.0))
    step_ms = sum(ksum.values())

    def roof(name, nbytes, ms, launches_per_step=1):
        ach = nbytes / (ms * 1e-3) / 1e9 if ms else 0.0
        return {"kernel": name, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                "frac": ach / hbm_peak, "traffic": None, "algorithmic_bytes": nbytes,
                "avg_launch_ms": ms / launches_per_step, "peak_source": peak_src}
    # DRAM traffic per launch from the committed ncu --set full captures (never measured here: a
    # number taken under a profiler is not a bench number, and ncu is not run by bench.py)
    try:
        ncu_traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
    except (OSError, ValueError):
        ncu_traffic = {}

    def traffic_for(key):
        t = ncu_traffic.get(key)
        return t["bytes_per_launch"] if t else None
    roofline = roof(dominant, algo[dominant], ksum[dominant], nl[dominant])
    if n == 1_000_000:
        roofline["traffic"] = traffic_for(dominant + "@config2")
        roofline["traffic_note"] = "per launch, from profiles/r02_ncu_traffic.json (ncu --set full capture of the same kernel and size)"
    roofline["share_of_step"] = ksum[dominant] / step_ms
    roofline["note"] = ("dominant kernel FAMILY of the step at this config (all its launches; per-kernel event timing "
                        "adds ~5 us per launch, so shares are indicative); at 1 M records every kernel is "
                        "latency-bound — the HBM-bound fractions are in roofline_hbm_bound")
    # the contract figure: bytes that MUST move for one scan (every record read once, every survivor written
    # once, two 4-byte permutation entries per survivor) over the time the whole scan takes
    scan_ms = sum(v for k, v in ksum.items() if not k.startswith("pciids"))
    contract = 16 * n + 24 * S
    roofline["whole_scan_contract"] = {"bytes": contract, "scan_ms_sum_of_kernels": scan_ms,
                                       "GBps": contract / (scan_ms * 1e-3) / 1e9 if scan_ms else None,
                                       "frac": contract / (scan_ms * 1e-3) / 1e9 / hbm_peak if scan_ms else None,
                                       "what": "(16 N + 24 S) / sum of the scan's kernel times at THIS config (latency-bound)"}
    kernel_rooflines = {k: {"ms_per_step": ksum[k], "share": ksum[k] / step_ms, "launches_per_step": nl[k],
                            "GBps": algo[k] / (ksum[k] * 1e-3) / 1e9, "frac": algo[k] / (ksum[k] * 1e-3) / 1e9 / hbm_peak}
                        for k in main_kernels}

    # ---- HBM-bound legs (inputs larger than L2): the >=70 % target is judged here
    roofline_big = {}
    if world == 1 and args.big_records:
        nb = args.big_records
        big = torch.empty(nb * 16, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        ctx.dev_gen_pci(big.data_ptr(), 0, nb, ids, GROUP_BITS_FOR(nb))
        for _ in range(3):
            ctx.dev_scan_pci(big.data_ptr(), nb)
        ts, packs, offs = [], [], []
        for _ in range(5):
            ctx.set_kernel_timing(True)
            ctx.dev_scan_pci(big.data_ptr(), nb)
            kt = ctx.kernel_times()
            d = {}
            for k, v in kt:
                d.setdefault(k, []).append(v)
            ts.append(d["classify_compact"][0])
            packs.append(d.get("pack_survivors", [0.0])[0])
            offs.append(d.get("tile_offsets", [0.0])[0])
            tot_ms = sum(v for _, v in kt)
        # the same scan WITHOUT per-kernel events (programmatic dependent launch on): the honest whole-scan time
        ctx.set_kernel_timing(False)
        evs2 = []
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            ctx.dev_scan_pci(big.data_ptr(), nb)
            e1.record(ext)
            evs2.append((e0, e1))
        Sb = ctx.dev_scan_pci_count()[0]
        whole_ms = sum(a.elapsed_time(b) for a, b in evs2) / len(evs2)
        cl = sum(ts) / len(ts)
        r = roof("classify_compact", 16 * nb + 16 * Sb, cl)
        comp_ms = cl + sum(packs) / len(packs) + sum(offs) / len(offs)
        r.update({"records": nb, "survivors": Sb, "whole_scan_ms": whole_ms,
                  "whole_scan_ms_sum_of_event_timed_kernels": tot_ms,
                  "whole_scan_records_per_s": nb / (whole_ms * 1e-3),
                  "compaction": {"what": "classify + tile offsets + pack = filter + STABLE compaction (the ragged "
                                         "classify kernel alone is the `achieved` figure above)",
                                 "ms": comp_ms, "GBps": (16 * nb + 16 * Sb) / (comp_ms * 1e-3) / 1e9,
                                 "frac": (16 * nb + 16 * Sb) / (comp_ms * 1e-3) / 1e9 / hbm_peak},
                  "whole_scan_contract": {"bytes": 16 * nb + 24 * Sb,
                                          "GBps": (16 * nb + 24 * Sb) / (whole_ms * 1e-3) / 1e9,
                                          "frac": (16 * nb + 24 * Sb) / (whole_ms * 1e-3) / 1e9 / hbm_peak}})
        r["traffic"] = traffic_for("classify_compact@%d" % nb)
        roofline_big["classify_compact"] = r
        del big
    if world == 1 and args.big_files:
        nf = args.big_files
        stride = pad + 16
        bigt = d_text[:stride].repeat(nf)
        torch.cuda.synchronize()
        c2 = kvgpu.Context(local_rank)
        for _ in range(3):
            c2.dev_pciids_parse(bigt.data_ptr(), len(text), stride, nf)
        ts, fam = [], []
        for _ in range(5):
            c2.set_kernel_timing(True)
            c2.dev_pciids_parse(bigt.data_ptr(), len(text), stride, nf)
            kt = dict(c2.kernel_times())
            ts.append(kt["pciids_parse"])
            fam.append(kt["pciids_parse"] + kt.get("pciids_resolve", 0.0))
        c2.set_kernel_timing(False)
        ent = c2.pciids_info()["n_entries"]
        spans = (len(text) + 4095) // 4096
        r = roof("pciids_parse", nf * (len(text) + 16 * spans), sum(ts) / len(ts))
        fam_ms = sum(fam) / len(fam)
        r.update({"images": nf, "text_bytes": nf * len(text), "entries_image0": ent,
                  "parse_GBps_text_only": nf * len(text) / (sum(ts) / len(ts) * 1e-3) / 1e9,
                  "scan_plus_resolve": {"ms": fam_ms, "GBps": nf * len(text) / (fam_ms * 1e-3) / 1e9,
                                        "frac": nf * len(text) / (fam_ms * 1e-3) / 1e9 / hbm_peak,
                                        "what": "k_pciids_scan + k_pciids_resolve_finalize (the lines of the NVIDIA "
                                                "block are recorded by the resolve pass)"}})
        r["traffic"] = traffic_for("pciids_parse@%d" % nf)
        roofline_big["pciids_parse"] = r
        c2.close()
        del bigt

    # ---- BASELINE.json configs 3 and 5 (extra keys; the headline stays config 2)
    extra = {}
    if world == 1 and not args.no_extra:
        import ctypes as C
        lib = kvgpu.load()
        # config 3: 65,536 mdev UUIDs over 256 raw type names (128 labels), 2,048 parents
        m = 65536
        mrecs = torch.from_numpy(np.frombuffer(O.gen_mdev(0, m).tobytes(), dtype=np.uint8).copy()).pin_memory()
        types = O.gen_type_names(256)
        td, keep = ctx._type_dict(types)
        def mdev_step():
            res = C.POINTER(kvgpu._lib.MdevResultC)()
            rc = lib.kvg_scan_mdev(ctx.handle, mrecs.data_ptr(), m, C.byref(td), C.byref(res))
            assert rc == 0
            s_ = int(res.contents.n_survivors)
            lib.kvg_result_free(res)
            return s_
        for _ in range(5):
            ms_ = mdev_step()
        t0 = time.perf_counter()
        for _ in range(50):
            mdev_step()
        tm = (time.perf_counter() - t0) / 50
        extra["config3_mdev"] = {"mdevs": m, "raw_types": 256, "survivors": ms_, "ms_per_scan_e2e": tm * 1e3,
                                 "mdevs_per_s_e2e": m / tm,
                                 "what": "kvg_scan_mdev: pinned host records in, host result out (labels, "
                                         "256 exact-prefix name lookups, 2 orderings)"}
        # config 5: 10,000 devices re-scanned at 1 kHz; 0.1 % of the records flip per tick
        hn = 10_000
        hrecs = torch.from_numpy(np.frombuffer(O.gen_pci(0, hn, ids, 12).tobytes(), dtype=np.uint8).copy()).pin_memory()
        hview = np.frombuffer(hrecs.numpy(), dtype=kvgpu.PCI_REC)
        rng = np.random.default_rng(5)
        lib.kvg_health_reset(ctx.handle)
        lat = []
        ticks = 10_000
        period = 1e-3
        t_next = time.perf_counter()
        for tick in range(ticks + 50):
            flip = rng.integers(0, hn, 10)
            hview["driver"][flip] = rng.integers(0, 5, 10)
            t0 = time.perf_counter()                        # snapshot is in the pinned buffer
            res = C.POINTER(kvgpu._lib.HealthDeltaC)()
            rc = lib.kvg_health_rescan(ctx.handle, hrecs.data_ptr(), hn, C.byref(res))
            dt = time.perf_counter() - t0                   # delta list visible to the host
            assert rc == 0
            lib.kvg_result_free(res)
            if tick >= 50:
                lat.append(dt)
            t_next += period
            while time.perf_counter() < t_next:
                pass
        lat = np.array(lat) * 1e6
        extra["config5_health_rescan"] = {"devices": hn, "poll_hz": 1000, "ticks": ticks,
                                          "p50_us": float(np.percentile(lat, 50)),
                                          "p99_us": float(np.percentile(lat, 99)),
                                          "max_us": float(lat.max()),
                                          "what": "host wall time from snapshot-in-pinned-buffer to "
                                                  "transition list on the host (H2D 160 KB + K6 + D2H)"}

    # ---- SURVEY.md 8(f)2: Allocate re-validation = one tiny batch through kvg_scan_pci; latency per request size
    if world == 1 and not args.no_extra:
        import ctypes as C
        lib = kvgpu.load()
        reval = {}
        for k in (1, 2, 4, 8, 16):
            rr = np.zeros(k, dtype=kvgpu.PCI_REC)
            for i in range(k):
                rr[i] = (i, 0x10de, 0, i // 2, 1, 0, 0)          # what BatchRevalidator builds: driver pinned, index mode
            hr = torch.from_numpy(np.frombuffer(rr.tobytes(), dtype=np.uint8).copy()).pin_memory()
            lat = []
            for it in range(1050):
                t0 = time.perf_counter()
                res = C.POINTER(kvgpu._lib.PciResultC)()
                rc = lib.kvg_scan_pci(ctx.handle, hr.data_ptr(), k, C.byref(res))
                dt = time.perf_counter() - t0
                assert rc == 0 and res.contents.n_survivors == k
                lib.kvg_result_free(res)
                if it >= 50:
                    lat.append(dt)
            lat = np.array(lat) * 1e6
            reval[str(k)] = {"p50_us": float(np.percentile(lat, 50)), "p99_us": float(np.percentile(lat, 99))}
        extra["allocate_revalidation"] = {"devices_per_request": reval, "requests_per_size": 1000,
                                          "what": "host wall time of one kvg_scan_pci batch of the size an Allocate request "
                                                  "re-checks (pinned records in, result block out): classify + both "
                                                  "orderings + fetch"}

    # ---- BASELINE.json config 4 as stated: mixed passthrough + vGPU, 100 M records over 8 GPUs
    if world > 1 and run_c4:
        c4_types = O.gen_type_names(256)
        d4 = torch.empty(c4_pci * 16, dtype=torch.uint8, device="cuda")
        m4 = torch.empty(c4_mdev * 32, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        ctx.dev_gen_pci(d4.data_ptr(), rank * c4_pci, c4_pci, ids, GROUP_BITS_FOR(c4_pci * world))
        ctx.dev_gen_mdev(m4.data_ptr(), rank * c4_mdev, c4_mdev)

        def c4_step():
            sharded.scan_device_shard(d4.data_ptr(), c4_pci)
            sharded.scan_device_mdev_shard(m4.data_ptr(), c4_mdev, c4_types)
        for _ in range(2):
            c4_step()
        sync_all()
        # size-independent properties of the sharded result (the exact check ran at the headline size)
        sharded.scan_device_shard(d4.data_ptr(), c4_pci)          # a fetch returns the LAST scan's result
        r4 = sharded.fetch()
        sharded.scan_device_mdev_shard(m4.data_ptr(), c4_mdev, c4_types)
        q4 = sharded.fetch_mdev()
        cnt = torch.tensor([len(r4.local), len(r4.dev.survivors), len(r4.grp.survivors), len(q4.local),
                            len(q4.by_type.survivors), len(q4.by_parent.survivors)], dtype=torch.int64, device="cuda")
        dist.all_reduce(cnt)
        cnt = [int(x) for x in cnt.tolist()]
        assert cnt[0] == cnt[1] == cnt[2] and cnt[3] == cnt[4] == cnt[5], cnt   # every survivor has exactly one owner per map
        assert np.all(r4.dev.survivors["device"].astype(np.int64) % world == rank)
        assert np.all(r4.grp.survivors["iommu_group"].astype(np.int64) % world == rank)
        assert np.all(np.diff(r4.local["addr"].astype(np.int64)) > 0) and np.all(np.diff(r4.dev.survivors["addr"].astype(np.int64)) > 0)
        _check_ordering(r4.dev.survivors, "device", r4.dev.dev_keys, r4.dev.dev_off, r4.dev.dev_perm, "config 4 deviceMap")
        _check_ordering(r4.grp.survivors, "iommu_group", r4.grp.grp_keys, r4.grp.grp_off, r4.grp.grp_perm, "config 4 iommuMap")
        _check_ordering(q4.by_type.survivors, "type_key", q4.by_type.type_keys, q4.by_type.type_off, q4.by_type.type_perm, "config 4 vGpuMap")
        _check_ordering(q4.by_parent.survivors, "parent", q4.by_parent.par_keys, q4.by_parent.par_off, q4.by_parent.par_perm, "config 4 gpuVgpuMap")
        del r4, q4
        evs4 = []
        sync_all()
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(ext)
            c4_step()
            e1.record(ext)
            evs4.append((e0, e1))
        sync_all()
        t4 = torch.tensor([sum(a.elapsed_time(b) for a, b in evs4) / len(evs4)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t4, op=dist.ReduceOp.MAX)
        t4 = float(t4.item())
        per_rank_bytes = 16 * c4_pci + 24 * (cnt[0] // world) + 32 * c4_mdev + 24 * (cnt[3] // world)
        extra["config4_sharded_100M"] = {
            "records_total": (c4_pci + c4_mdev) * world, "pci_per_rank": c4_pci, "mdev_per_rank": c4_mdev,
            "pci_survivors_total": cnt[0], "mdev_survivors_total": cnt[3], "ms_per_scan_max_over_ranks": t4,
            "records_per_s": (c4_pci + c4_mdev) * world / (t4 * 1e-3),
            "per_rank_contract_GBps": per_rank_bytes / (t4 * 1e-3) / 1e9,
            "per_rank_contract_frac": per_rank_bytes / (t4 * 1e-3) / 1e9 / hbm_peak,
            "nvlink_out_bytes_per_rank": 2 * 16 * (cnt[0] // world) + 2 * 32 * (cnt[3] // world),
            "exchange": sharded.mode, "parity": "properties: one owner per survivor and map (all-reduced counts), "
            "key % world == rank, Walk order inside every list, both orderings == stable sort, on every rank"}
        del d4, m4

    # ---- end to end through the reference-facing calls: pinned host in, host results out
    e2e = None
    if world == 1:
        p_text = torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()).pin_memory()
        p_recs = torch.empty(max(n, 1) * 16, dtype=torch.uint8).pin_memory()
        p_recs.numpy()[:n * 16] = np.frombuffer(O.gen_pci(0, n, ids, gbits).tobytes(), dtype=np.uint8)
        recs_np = np.frombuffer(p_recs.numpy()[:n * 16], dtype=kvgpu.PCI_REC)
        import ctypes as C
        lib = kvgpu.load()

        def e2e_step():
            rc = lib.kvg_pciids_load(ctx.handle, p_text.data_ptr(), len(text))
            assert rc == 0, rc
            res = C.POINTER(kvgpu._lib.PciResultC)()
            rc = lib.kvg_scan_pci(ctx.handle, recs_np.ctypes.data, n, C.byref(res))
            assert rc == 0, rc
            r = res.contents
            nbytes = (int(r.n_survivors) * (16 + 4 + 4) + int(r.n_dev_keys) * 10 +
                      int(r.n_groups) * 8 + int(r.name_pool_len))
            surv = int(r.n_survivors)
            lib.kvg_result_free(res)
            return nbytes, surv
        for _ in range(max(3, args.warmup)):
            d2h, s_e2e = e2e_step()
        assert s_e2e == (S if not sharded else s_e2e)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            d2h, _ = e2e_step()
        te = time.perf_counter() - t0
        # what the link itself does on this box (pinned <-> device, same buffers): the e2e floor
        dev_tmp = torch.empty_like(p_recs, device="cuda")
        host_tmp = torch.empty_like(p_recs).pin_memory()
        bw = {}
        for name, dst, src_ in (("h2d", dev_tmp, p_recs), ("d2h", host_tmp, dev_tmp)):
            dst.copy_(src_, non_blocking=True)
            torch.cuda.synchronize()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(5):
                dst.copy_(src_, non_blocking=True)
            b_.record()
            torch.cuda.synchronize()
            bw[name] = 5 * p_recs.numel() / (a.elapsed_time(b_) * 1e-3) / 1e9
        del dev_tmp, host_tmp
        e2e = {"value": n * args.steps / te, "unit": "records/s", "ms_per_step": 1e3 * te / args.steps,
               "h2d_bytes_per_step": len(text) + 16 * n, "d2h_bytes_per_step": d2h,
               "pcie_measured_GBps": {k: round(v, 1) for k, v in bw.items()},
               "pcie_floor_ms": {"h2d_only": 1e3 * (len(text) + 16 * n) / (bw["h2d"] * 1e9),
                                 "h2d_plus_d2h_serial": 1e3 * ((len(text) + 16 * n) / (bw["h2d"] * 1e9) +
                                                               d2h / (bw["d2h"] * 1e9))},
               "timing": "host wall clock around kvg_pciids_load + kvg_scan_pci (pinned host buffers "
                         "in, pinned host result out)"}
    else:
        # N > 1: per-rank pinned shard in, gathered result out on every rank
        p_recs = torch.empty(max(n, 1) * 16, dtype=torch.uint8).pin_memory()
        p_recs.numpy()[:n * 16] = np.frombuffer(O.gen_pci(rank * n, n, ids, gbits).tobytes(), dtype=np.uint8)
        p_text = torch.from_numpy(np.frombuffer(text, dtype=np.uint8).copy()).pin_memory()
        lib = kvgpu.load()

        import ctypes as C

        def e2e_step():
            rc = lib.kvg_pciids_load(ctx.handle, p_text.data_ptr(), len(text))      # pinned: copy + parse enqueued
            assert rc == 0
            with torch.cuda.stream(ext):                                           # the rank's shard: async, same stream
                d_recs[:n * 16].copy_(p_recs[:n * 16], non_blocking=True)
            sharded.scan_device_shard(d_recs.data_ptr(), n)
            res = C.POINTER(kvgpu._lib.PciShardResultC)()
            rc = lib.kvg_dev_scan_pci_shard_fetch(ctx.handle, C.byref(res))        # THIS rank's parts -> host
            assert rc == 0
            r = res.contents
            out = (int(r.n_local), int(r.n_dev_members), int(r.n_grp_members), int(r.n_dev_keys), int(r.n_groups))
            lib.kvg_result_free(res)
            return out
        for _ in range(3):
            r = e2e_step()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            r = e2e_step()
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        te = float(te.item())
        e2e = {"value": n * world * args.steps / te, "unit": "records/s",
               "ms_per_step": 1e3 * te / args.steps,
               "h2d_bytes_per_step": len(text) + 16 * n,
               "d2h_bytes_per_step": int(16 * (r[0] + r[1] + r[2]) + 4 * (r[1] + r[2]) + 10 * r[3] + 8 * r[4]),
               "timing": "host wall clock, max over ranks; per rank: pinned shard in, its parts of the result out"}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_baseline(text, ids, min(n, args.cpu_sample), os.cpu_count() or 1)
        line = {
            "metric": METRIC, "value": value, "unit": "records/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/u32 (byte + integer)", "data": "synthetic",
            "config": {"workload": "BASELINE.json configs[1]: full utils/pci.ids (%d B, %d lines) parse "
                                   "+ %d synthetic PCI records per GPU per step%s" % (
                                       len(text), info["n_lines"], n,
                                       "" if world == 1 else ", range-sharded over %d GPUs, every survivor sent to the "
                                       "owner of its key once per map (%s), maps partitioned by key" % (
                                           world, "stores into the owners' peer windows over NVLink"
                                           if sharded.mode == "p2p" else "NCCL allgatherv + local select")),
                       "exchange": None if world == 1 else sharded.mode,
                       "records_per_gpu": n, "survivors": S, "device_ids": KD, "iommu_groups": G,
                       "iommu_group_order": "bijective scramble of i>>1 (group_bits=%d)" % gbits,
                       "l2": "flushed between timed steps (192 MiB fill, outside the event bracket)",
                       "wall_s_timed_loop_incl_flush": t_wall},
            "pciids_parse_GBps": len(text) / (kavg.get("pciids_parse", 0) * 1e-3) / 1e9 if kavg.get("pciids_parse") else None,
            "parity": parity,
            "roofline": roofline,
            "kernel_rooflines": kernel_rooflines,
            "roofline_hbm_bound": roofline_big,
            "kernel_ms_per_step": ksum,
            "cpu_baseline": cpu,
            "other_configs": extra,
            "e2e": e2e,
            "gpu_launches": launches,
            "clocks": clocks,
        }
        print(json.dumps(line))
    # free torch tensors before the context (and its stream) goes away — pinned ones too: the host allocator
    # records an event on every stream a pinned block was used on when the block is freed
    del d_recs, d_text, p_recs, p_text
    import gc
    gc.collect()
    torch.cuda.synchronize()
    if sharded:
        sharded.close()
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
