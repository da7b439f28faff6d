"""GPU: kvg_rescan_pci / kvg_rescan_mdev against the oracle.  Expected deltas come from the oracle's maps of the
previous and the current snapshot (canonical dumps parsed into dicts and diffed); the embedded scan must equal
Context.scan_pci / scan_mdev byte for byte; baseline resets, input checks, a seeded churn sequence, and
DiscoveryScan.rediscover() on a mutated sysfs tree."""
import os

import numpy as np
import pytest

import conftest  # noqa: F401
import kvgpu
import util
from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def text():
    return util.pciids_text()


@pytest.fixture(scope="module")
def ids(text):
    return O.nv_ids(text)


@pytest.fixture
def ctx(text):
    with kvgpu.Context(0) as c:
        c.pciids_load(text)
        yield c


# ---- the oracle side ---------------------------------------------------------------------------------------------
def parse_dump(dump: bytes) -> dict:
    """canonical dump -> {tag: {key: [member line, ...]}} (B: {addr: group})"""
    out = {t: {} for t in "DIBVG"}
    cur = None
    for line in dump.decode("latin-1").splitlines():
        if line.startswith("  "):
            cur.append(line.strip())
            continue
        parts = line.split(" ")
        if parts[0] == "B":
            out["B"][parts[1]] = parts[2]
        else:
            cur = out[parts[0]].setdefault(parts[1], [])
    return out


def oracle_pci(recs, text):
    om = O.Maps()
    om.create_iommu_device_map_flat(recs)
    return parse_dump(om.dump(text))


def oracle_mdev(recs, types, text):
    om = O.Maps()
    om.create_vgpu_id_map_flat(recs, types)
    return parse_dump(om.dump(text))


def dict_diff(old: dict, new: dict):
    return (sorted(set(new) - set(old)), sorted(set(old) - set(new)),
            sorted(k for k in set(old) & set(new) if old[k] != new[k]))


def keyed(d: dict, f) -> dict:
    return {f(k): v for k, v in d.items()}


def pci_survivors(p: dict) -> dict:
    """addr -> (device, group, numa) from the D and B sections"""
    out = {}
    for dev, members in p["D"].items():
        for m in members:
            addr, numa = m.split(" ")
            out[kvgpu.parse_bdf(addr)] = (int(dev, 16), int(p["B"][addr]), int(numa))
    return out


def mdev_survivors(p: dict, canon: dict) -> dict:
    """uuid -> (canonical type, parent, numa) from the V and G sections"""
    parent = {u: kvgpu.parse_bdf(g) for g, us in p["G"].items() for u in us}
    out = {}
    for label, members in p["V"].items():
        for m in members:
            u, numa = m.split(" ")
            out[u] = (canon[label], parent[u], int(numa))
    return out


def surv_diff(old: dict, new: dict):
    return (sorted(set(new) - set(old)), sorted(set(old) - set(new)),
            sorted(k for k in set(old) & set(new) if old[k] != new[k]))


def check_pci(r, prev, cur):
    got_keys = [(list(d.added), list(d.removed), list(d.changed)) for d in (r.dev, r.grp)]
    want_keys = [dict_diff(keyed(prev["D"], lambda k: int(k, 16)), keyed(cur["D"], lambda k: int(k, 16))),
                 dict_diff(keyed(prev["I"], int), keyed(cur["I"], int))]
    assert got_keys == [tuple(map(list, w)) for w in want_keys]
    a, rm, mv = surv_diff(pci_survivors(prev), pci_survivors(cur))
    s = r.scan.survivors["addr"]
    assert s[r.added].tolist() == a and r.removed["addr"].tolist() == rm and s[r.moved].tolist() == mv


def canon_of(res) -> dict:
    return {res.labels[i].decode("latin-1"): int(res.type_canon[i]) for i in range(len(res.labels))}


def check_mdev(r, prev, cur):
    canon = canon_of(r.scan)
    got_keys = [(list(d.added), list(d.removed), list(d.changed)) for d in (r.type, r.parent)]
    want_keys = [dict_diff(keyed(prev["V"], canon.get), keyed(cur["V"], canon.get)),
                 dict_diff(keyed(prev["G"], kvgpu.parse_bdf), keyed(cur["G"], kvgpu.parse_bdf))]
    assert got_keys == [tuple(map(list, w)) for w in want_keys]
    a, rm, mv = surv_diff(mdev_survivors(prev, canon), mdev_survivors(cur, canon))
    u = [kvgpu.format_uuid(x) for x in r.scan.survivors["uuid"]]
    assert [u[i] for i in r.added] == a and [u[i] for i in r.moved] == mv
    assert [kvgpu.format_uuid(x) for x in r.removed["uuid"]] == rm


def same_pci(a, b):
    for f in ("survivors", "dev_keys", "dev_off", "dev_perm", "dev_name_slot", "grp_keys", "grp_off", "grp_perm"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    assert a.name_pool == b.name_pool and a.n_records == b.n_records


def same_mdev(a, b):
    for f in ("survivors", "type_keys", "type_off", "type_perm", "type_canon", "par_keys", "par_off", "par_perm"):
        assert getattr(a, f).tobytes() == getattr(b, f).tobytes(), f
    assert a.labels == b.labels and a.type_names == b.type_names


# ---- seeded churn --------------------------------------------------------------------------------------------------
def churn_pci(base, t, frac=0.001):
    rng = np.random.default_rng(1000 + t)
    n = len(base)
    if n == 0:
        return base
    keep = rng.random(n) >= frac                      # records appear and disappear
    recs = base.copy()
    k = max(1, n // 5000)
    flip = rng.choice(n, k, replace=False)            # driver flips
    recs["driver"][flip] = np.where(recs["driver"][flip] == 1, 3, 1)
    mv = rng.choice(n, k, replace=False)              # numa / group rewrites
    recs["numa"][mv[: k // 2 + 1]] ^= 1
    recs["iommu_group"][mv[k // 2:]] += 7
    return recs[keep]


def churn_mdev(base, t, n_types, frac=0.001):
    rng = np.random.default_rng(2000 + t)
    n = len(base)
    keep = rng.random(n) >= frac
    recs = base.copy()
    k = max(1, n // 5000)
    mv = rng.choice(n, 3 * k, replace=False)
    recs["parent_numa"][mv[:k]] ^= 1
    recs["parent"][mv[k:2 * k]] += 1
    recs["type_idx"][mv[2 * k:]] = rng.integers(0, n_types, k)
    return recs[keep]


# ---- tests ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [0, 1, 10_000, 1_000_000])
def test_pci_scan_is_identical_and_first_call_reports_everything_added(ctx, text, ids, n):
    recs = O.gen_pci(0, n, ids, 16)
    r = ctx.rescan_pci(recs)
    same_pci(r.scan, ctx.scan_pci(recs))
    assert not r.had_baseline
    assert r.added.tolist() == list(range(len(r.scan.survivors))) and len(r.removed) == 0 and len(r.moved) == 0
    assert r.dev.added.tolist() == r.scan.dev_keys.tolist() and r.grp.added.tolist() == r.scan.grp_keys.tolist()
    check_pci(r, oracle_pci(recs[:0], text), oracle_pci(recs, text))
    # the next tick: churn crosses the same path (>= 128 Ki records: the pipelined host copy)
    nxt = churn_pci(recs, 1)
    r2 = ctx.rescan_pci(nxt)
    assert r2.had_baseline
    same_pci(r2.scan, ctx.scan_pci(nxt))
    if n >= 10_000:
        check_pci(r2, oracle_pci(recs, text), oracle_pci(nxt, text))


def test_mdev_65536_with_an_appended_dictionary(ctx, text):
    types = O.gen_type_names(256)
    recs = O.gen_mdev(0, 65_536)
    r = ctx.rescan_mdev(recs, types)
    same_mdev(r.scan, ctx.scan_mdev(recs, types))
    assert not r.had_baseline and r.type.added.tolist() == r.scan.type_keys.tolist()
    more = O.gen_type_names(300)
    assert more[:256] == types
    nxt = churn_mdev(recs, 1, 300)
    r2 = ctx.rescan_mdev(nxt, more)
    same_mdev(r2.scan, ctx.scan_mdev(nxt, more))
    check_mdev(r2, oracle_mdev(recs, types, text), oracle_mdev(nxt, more, text))


def test_resets(ctx, text, ids):
    recs = O.gen_pci(0, 5000, ids, 16)
    ctx.rescan_pci(recs)
    assert ctx.rescan_pci(recs).had_baseline
    r = ctx.rescan_pci(recs)
    assert len(r.added) == 0 and len(r.dev.changed) == 0 and len(r.grp.added) == 0
    ctx.rescan_reset()
    r = ctx.rescan_pci(recs)
    assert not r.had_baseline and len(r.added) == len(r.scan.survivors)
    ctx.pciids_load(text)                             # names may change: the baseline goes
    r = ctx.rescan_pci(recs)
    assert not r.had_baseline and len(r.added) == len(r.scan.survivors)
    # the other calls leave the baseline alone
    ctx.scan_pci(O.gen_pci(7, 3000, ids, 16))
    ctx.health_rescan(recs)
    assert ctx.rescan_pci(recs).had_baseline


def test_non_ascending_snapshot_is_refused_and_keeps_the_baseline(ctx, text, ids):
    recs = O.gen_pci(0, 20_000, ids, 16)
    ctx.rescan_pci(recs)
    bad = recs.copy()
    bad[[100, 15000]] = bad[[15000, 100]]
    with pytest.raises(kvgpu.KvgError) as e:
        ctx.rescan_pci(bad)
    assert e.value.rc == -1
    nxt = churn_pci(recs, 3)
    r = ctx.rescan_pci(nxt)                           # diffed against `recs`, not against the refused snapshot
    check_pci(r, oracle_pci(recs, text), oracle_pci(nxt, text))


def test_non_extending_dictionary_is_refused(ctx):
    types = O.gen_type_names(256)
    recs = O.gen_mdev(0, 4096)
    ctx.rescan_mdev(recs, types)
    for other in (types[:200], [types[1], types[0]] + types[2:], types[:10] + [b"X"] + types[11:]):
        with pytest.raises(kvgpu.KvgError) as e:
            ctx.rescan_mdev(recs, other)
        assert e.value.rc == -1
    assert ctx.rescan_mdev(recs, types + [b"NVIDIA NEW-1Q\n"]).had_baseline


def test_twenty_tick_churn_matches_the_oracle(ctx, text, ids):
    base = O.gen_pci(0, 200_000, ids, 16)
    mbase = O.gen_mdev(0, 20_000)
    types = O.gen_type_names(256)
    prev = prev_m = None
    for t in range(20):
        recs, mrecs = churn_pci(base, t), churn_mdev(mbase, t, 256)
        cur, cur_m = oracle_pci(recs, text), oracle_mdev(mrecs, types, text)
        r, rm = ctx.rescan_pci(recs), ctx.rescan_mdev(mrecs, types)
        if prev is not None:
            check_pci(r, prev, cur)
            check_mdev(rm, prev_m, cur_m)
        prev, prev_m = cur, cur_m


def test_rediscover_on_a_mutated_tree(tmp_path, text):
    root = str(tmp_path)
    ent = util.c1_tree_entries()
    base = util.make_pci_tree(os.path.join(root, "p"), ent)
    parents = {"0000:04:00.0": "0\n", "0000:84:00.0": "1\n"}
    mdevs = {"3f4c2b1a-0000-4000-8000-%012x" % k: dict(type="GRID P40-%dQ\n" % (1 + k % 2),
                                                        parent="0000:04:00.0" if k < 3 else "0000:84:00.0")
             for k in range(6)}
    vdir, pdir = util.make_mdev_tree(os.path.join(root, "m"), parents, mdevs)
    ids_path = os.path.join(root, "pci.ids")
    with open(ids_path, "wb") as f:
        f.write(text)
    ds = kvgpu.DiscoveryScan(ids_path, base, vdir)
    try:
        first = ds.rediscover()
        assert sorted((e.kind, e.key) for e in first) == sorted(
            [("start", k) for k in ds.maps.deviceMap] + [("start", k) for k in ds.maps.vGpuMap])
        before = kvgpu.canonical_dump(ds.maps)
        maps_obj = ds.maps
        # bind a new 10de function to vfio-pci, unbind one, change a numa node
        real = os.path.join(root, "p", "real")
        ent2 = {"0000:88:00.0": dict(vendor="10de", device="2330", driver="vfio-pci", iommu_group="60",
                                     numa_node="1\n")}
        util.make_pci_tree(os.path.join(root, "p"), ent2)
        os.remove(os.path.join(real, "0000:05:00.0", "driver"))
        os.symlink(os.path.join(root, "p", "targets", "drivers", "nvidia"), os.path.join(real, "0000:05:00.0", "driver"))
        with open(os.path.join(real, "0000:06:00.0", "numa_node"), "w") as f:
            f.write("1\n")
        # create and remove mdev links
        os.remove(os.path.join(vdir, "3f4c2b1a-0000-4000-8000-000000000001"))
        util.make_mdev_tree(os.path.join(root, "m"), {}, {"3f4c2b1a-0000-4000-8000-0000000000aa": dict(
            type="GRID P40-8Q\n", parent="0000:84:00.0")})
        old = parse_dump(before)
        events = ds.rediscover()
        assert ds.maps is maps_obj                    # updated in place
        fresh = kvgpu.DiscoveryScan(ids_path, base, vdir)
        try:
            fresh.create_iommu_device_map()
            fresh.create_vgpu_id_map()
            assert kvgpu.canonical_dump(ds.maps) == kvgpu.canonical_dump(fresh.maps)
        finally:
            fresh.close()
        new = parse_dump(kvgpu.canonical_dump(ds.maps))
        want = []
        for tag, vgpu in (("D", False), ("V", True)):
            a, r, c = dict_diff(old[tag], new[tag])
            want += [("start", k, vgpu) for k in a] + [("stop", k, vgpu) for k in r] + [("update", k, vgpu) for k in c]
        assert sorted((e.kind, e.key, e.vgpu) for e in events) == sorted(want)
        assert ("start", "2330", False) in want and ("update", "1b38", False) in want
        assert ("start", "GRID_P40-8Q", True) in want
        specs = {(s.vgpu, s.key): s for s in ds.create_device_plugins()}
        for e in events:
            if e.kind != "stop":
                assert e.spec == specs[(e.vgpu, e.key)]
    finally:
        ds.close()
