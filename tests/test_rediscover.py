"""CPU, real gRPC: serve.RediscoveryFeed applies the PluginEvents of a rediscovery to running plugins against a
mock kubelet (added key -> a new registration, removed key -> its socket goes, changed key -> ListAndWatch re-sends
the whole new list, Allocate reads the swapped maps, replace_all), `--rediscover-period 0` keeps the one-shot
start-up, and without a device the rescan entry points compute nothing."""
import ctypes as C
import os
import shutil
import tempfile
import types

import numpy as np
import pytest

import conftest
import kvgpu
from kvgpu import __main__ as kmain
from kvgpu import serve


def maps_a():
    m = kvgpu.Maps()
    m.deviceMap["1b38"] = [kvgpu.NvidiaGpuDevice("0000:04:00.0", 0), kvgpu.NvidiaGpuDevice("0000:05:00.0", 0)]
    m.deviceNames["1b38"] = "GP102GL_TESLA_P40"
    m.iommuMap = {"40": [kvgpu.NvidiaGpuDevice("0000:04:00.0", 0)], "41": [kvgpu.NvidiaGpuDevice("0000:05:00.0", 0)]}
    m.bdfToIommuMap = {"0000:04:00.0": "40", "0000:05:00.0": "41"}
    return m


def maps_b():
    """0000:05:00.0 moved to numa 1 and group 45, a new device id appeared, 0000:04:00.0 left"""
    m = kvgpu.Maps()
    m.deviceMap["1b38"] = [kvgpu.NvidiaGpuDevice("0000:05:00.0", 1)]
    m.deviceNames["1b38"] = "GP102GL_TESLA_P40"
    m.deviceMap["2330"] = [kvgpu.NvidiaGpuDevice("0000:88:00.0", 1)]
    m.deviceNames["2330"] = "GH100_H100_SXM5_80GB"
    m.iommuMap = {"45": [kvgpu.NvidiaGpuDevice("0000:05:00.0", 1)], "60": [kvgpu.NvidiaGpuDevice("0000:88:00.0", 1)]}
    m.bdfToIommuMap = {"0000:05:00.0": "45", "0000:88:00.0": "60"}
    return m


def test_maps_still_pickle_and_compare_equal():
    """the swap lock is not part of the maps: sharded scans send Maps between processes"""
    import copy
    import pickle
    m = maps_b()
    back = pickle.loads(pickle.dumps(m))
    assert back == m and back.lock is not m.lock
    assert copy.deepcopy(m) == m
    with back.lock:
        pass


class FakeScan:
    """DiscoveryScan's rediscover() contract without a GPU: swap in the next scripted maps, return its events."""

    def __init__(self, first, script):
        self.maps = first
        self.script = list(script)

    def rediscover(self):
        nxt, events = self.script.pop(0)
        self.maps.swap(nxt)
        specs = {(s.vgpu, s.key): s for s in kvgpu.plugin_specs_from_maps(self.maps)}
        return [kvgpu.PluginEvent(kind, key, vgpu, specs.get((vgpu, key))) for kind, key, vgpu in events]


class Links:
    """the revalidator's view of sysfs: every advertised address is an NVIDIA function in its group"""

    def __init__(self, maps):
        self.maps = maps

    def read_link(self, base, addr, link):
        g = self.maps.bdfToIommuMap.get(addr)
        return (g, False) if g is not None else ("", True)

    def read_id(self, base, addr, prop):
        return ("10de", False)


def fake_scan_pci(recs):
    import numpy as np
    keep = recs["vendor"] == 0x10de
    surv = np.zeros(int(keep.sum()), dtype=kvgpu.PCI_SURV)
    surv["addr"], surv["iommu_group"] = recs["addr"][keep], recs["iommu_group"][keep]
    return types.SimpleNamespace(survivors=surv)


@pytest.fixture
def sockdir():
    d = tempfile.mkdtemp(prefix="kvg", dir="/tmp")   # unix socket paths are limited to 107 bytes
    yield d
    shutil.rmtree(d, ignore_errors=True)


def test_feed_starts_stops_and_updates_plugins(sockdir):
    kubelet = serve.MockKubelet(sockdir).start()
    ds = FakeScan(maps_a(), [(maps_b(), [("start", "2330", False), ("update", "1b38", False)]),
                             (maps_b(), [("stop", "2330", False)])])
    links = Links(ds.maps)
    reval = serve.BatchRevalidator(fake_scan_pci, sockdir, links.read_link, links.read_id)
    specs = kvgpu.plugin_specs_from_maps(ds.maps)
    plugins = serve.plugins_from_specs(specs, ds.maps, reval, socket_dir=sockdir, base_path=sockdir,
                                       root_path=sockdir, discover_egm=lambda: [])
    live = {(s.vgpu, s.key): p for s, p in zip(specs, plugins)}
    feed = serve.RediscoveryFeed(ds, live, 3600.0, revalidate=reval, watch=False, socket_dir=sockdir,
                                 base_path=sockdir, root_path=sockdir, discover_egm=lambda: [])
    try:
        for p in plugins:
            p.start()
        regs = kubelet.wait_for(1)
        c = kubelet.connect(regs[0])
        stream = c.list_and_watch()
        assert [(d.ID, d.topology.nodes[0].ID) for d in next(stream).devices] == [("0000:04:00.0", 0),
                                                                                    ("0000:05:00.0", 0)]
        r = c.allocate(["0000:05:00.0"]).container_responses
        assert [d.host_path for d in r[0].devices] == ["/dev/vfio/vfio", "/dev/vfio/41"]

        feed.tick()
        # the added key registers a new resource
        regs = kubelet.wait_for(2)
        assert regs[1].resource_name == "nvidia.com/GH100_H100_SXM5_80GB"
        assert os.path.exists(os.path.join(sockdir, "kubevirt-GH100_H100_SXM5_80GB.sock"))
        # the changed key's stream receives the whole new list
        assert [(d.ID, d.topology.nodes[0].ID) for d in next(stream).devices] == [("0000:05:00.0", 1)]
        # Allocate sees the new IOMMU group after the swap
        r = c.allocate(["0000:05:00.0"]).container_responses
        assert [d.host_path for d in r[0].devices] == ["/dev/vfio/vfio", "/dev/vfio/45"]
        stream.cancel()
        c.close()

        feed.tick()
        # the removed key's plugin stops: its socket disappears
        assert not os.path.exists(os.path.join(sockdir, "kubevirt-GH100_H100_SXM5_80GB.sock"))
        assert set(live) == {(False, "1b38")}
    finally:
        feed.stop()
        for p in list(live.values()) + plugins:
            p.stop()
        kubelet.stop()


def test_replace_all_restarts_every_plugin(sockdir):
    kubelet = serve.MockKubelet(sockdir).start()
    ds = FakeScan(maps_a(), [(maps_b(), [("replace_all", None, False)])])
    live = {}
    feed = serve.RediscoveryFeed(ds, live, 3600.0, watch=False, socket_dir=sockdir, base_path=sockdir,
                                 root_path=sockdir, discover_egm=lambda: [])
    try:
        feed.tick()
        regs = kubelet.wait_for(2)
        assert sorted(r.resource_name for r in regs) == ["nvidia.com/GH100_H100_SXM5_80GB",
                                                         "nvidia.com/GP102GL_TESLA_P40"]
        assert set(live) == {(False, "1b38"), (False, "2330")}
    finally:
        feed.stop()
        for p in live.values():
            p.stop()
        kubelet.stop()


def test_index_mode_snapshots_lead_to_replace_all(monkeypatch, tmp_path):
    """DiscoveryScan.rediscover with a snapshot that has no stable identities: full scans, no delta path"""
    from kvgpu import plugin as P
    calls = []

    class Ctx:
        def pciids_load(self, text):
            pass

        def rescan_reset(self):
            calls.append("reset")

        def rescan_pci(self, recs):
            raise AssertionError("index-mode snapshots must not reach the delta path")

        rescan_mdev = rescan_pci

        def scan_pci(self, recs):
            calls.append("scan_pci")
            return types.SimpleNamespace(survivors=np.zeros(0, kvgpu.PCI_SURV), dev_keys=[], grp_keys=[])

        def scan_mdev(self, recs, raw):
            calls.append("scan_mdev")
            return types.SimpleNamespace(survivors=np.zeros(0, kvgpu.MDEV_SURV), type_keys=[],
                                         par_keys=[])

        def name_lookup(self, key):
            return ""

    ds = P.DiscoveryScan.__new__(P.DiscoveryScan)
    ds.pciIdsFilePath, ds.basePath, ds.vGpuBasePath = str(tmp_path / "ids"), str(tmp_path), str(tmp_path)
    ds.ctx, ds.maps, ds._loaded_path = Ctx(), kvgpu.Maps(), None
    ds._raw_types, ds._type_index = [], {}
    snap = P.PciSnapshot(np.zeros(0, kvgpu.PCI_REC), [], False, None)   # index mode
    monkeypatch.setattr(P, "snapshot_pci_tree", lambda base: snap)
    monkeypatch.setattr(P, "snapshot_mdev_tree", lambda v, p: P.MdevSnapshot(
        np.zeros(0, kvgpu.MDEV_REC), [], [], None, True))
    events = ds.rediscover()
    assert [e.kind for e in events] == ["replace_all"]
    assert calls == ["reset", "scan_pci", "scan_mdev"]


@pytest.mark.parametrize("period,feeds", [("0", 0), ("5", 1)])
def test_rediscover_period_zero_starts_no_feed(monkeypatch, period, feeds):
    made, scans = [], []

    class DS:
        def __init__(self, *a):
            self.maps, self.ctx = maps_a(), types.SimpleNamespace(scan_pci=None)

        def create_iommu_device_map(self):
            scans.append("full")

        def create_vgpu_id_map(self):
            pass

        def rediscover(self):
            scans.append("rediscover")
            return []

        def create_device_plugins(self):
            return []

        def close(self):
            pass

    class Feed:
        def __init__(self, *a, **kw):
            made.append(a)
            self.plugins = {}

        def start(self):
            pass

        def stop(self):
            pass

    class SetEvent:
        def wait(self, *a):
            return True

        def set(self):
            pass

    monkeypatch.setattr(kvgpu, "DiscoveryScan", DS)
    monkeypatch.setattr(serve, "RediscoveryFeed", Feed)
    monkeypatch.setattr(kmain, "threading", types.SimpleNamespace(Event=SetEvent))
    assert kmain.main(["--rediscover-period", period, "--socket-dir", "/nonexistent"]) == 0
    assert len(made) == feeds
    assert scans == (["full"] if feeds == 0 else ["rediscover"])


@pytest.mark.skipif(conftest.HAS_GPU, reason="checks the no-GPU failure mode")
def test_rescan_entry_points_without_a_device():
    lib = kvgpu.load()
    with pytest.raises(kvgpu.KvgError) as e:
        kvgpu.Context(0)
    assert e.value.rc == -2                       # KVG_ECUDA: no context, so no rescan, and no CPU fallback
    h = C.c_void_p()
    assert lib.kvg_ctx_create(0, C.byref(h)) == -2 and not h.value
    pr, mr = C.POINTER(kvgpu._lib.PciRescanC)(), C.POINTER(kvgpu._lib.MdevRescanC)()
    assert lib.kvg_rescan_pci(None, None, 0, C.byref(pr)) == -1
    assert lib.kvg_rescan_mdev(None, None, 0, None, C.byref(mr)) == -1
    assert lib.kvg_rescan_reset(None) == -1
