"""Host-side mirror of the reference's plugin interface for the scan path.

Same names, argument meaning and error behaviour as pkg/device_plugin/device_plugin.go, but the
filter / join / bucketing run in libkvgpu.so on the GPU:

    snapshot_pci_tree / snapshot_mdev_tree   the five sysfs readers (:294-357) turned into a flat
                                             record array (syscalls stay on the CPU, nothing is
                                             pre-filtered: read failures travel as flag bits)
    DiscoveryScan.create_iommu_device_map    createIommuDeviceMap  (:187-247)
    DiscoveryScan.create_vgpu_id_map         createVgpuIDMap       (:255-291)
    DiscoveryScan.get_device_name            getDeviceName         (:371-422)
    DiscoveryScan.rediscover                 a fresh snapshot diffed against the previous one on the GPU
                                             (Context.rescan_pci / rescan_mdev) -> plugin start / stop / update
    DiscoveryScan.create_device_plugins      the payload half of createDevicePlugins (:99-157):
                                             per key the pluginapi.Device list, resource name,
                                             socket path and env key the Go servers would use
    canonical_dump                           SURVEY.md 8c parity artefact

This module never imports the oracle and has no CPU implementation of the filter/join: without
libkvgpu.so and a CUDA device DiscoveryScan cannot be constructed.
"""
from __future__ import annotations

import os
import threading
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from .context import Context, MdevResult, PciResult

HEXD = "0123456789abcdef"
DEVICE_NAMESPACE = "nvidia.com"                       # generic_device_plugin.go:51
DEVICE_PLUGIN_PATH = "/var/lib/kubelet/device-plugins/"  # pluginapi.DevicePluginPath
GPU_PREFIX = "PCI_RESOURCE_NVIDIA_COM"                # generic_device_plugin.go:57
VGPU_PREFIX = "MDEV_PCI_RESOURCE_NVIDIA_COM"          # generic_device_plugin.go:58
HEALTHY, UNHEALTHY = "Healthy", "Unhealthy"           # pluginapi constants


class ReferencePanic(RuntimeError):
    """The Go reference would panic on this sysfs content (e.g. data[2:] on a 1-byte file)."""


def format_bdf(p: int) -> str:
    return "%04x:%02x:%02x.%x" % (p >> 16, (p >> 8) & 0xFF, (p >> 3) & 0x1F, p & 7)


def parse_bdf(s: str):
    """'dddd:bb:dd.f' -> packed value, or None if `s` is not exactly that canonical form."""
    if len(s) != 12 or s[4] != ":" or s[7] != ":" or s[10] != ".":
        return None
    hx = s[0:4] + s[5:7] + s[8:10] + s[11]
    if any(c not in HEXD for c in hx):
        return None
    dom, bus, dev, fn = int(s[0:4], 16), int(s[5:7], 16), int(s[8:10], 16), int(s[11], 16)
    if dev > 31 or fn > 7:
        return None
    return (dom << 16) | (bus << 8) | (dev << 3) | fn


def format_uuid(u) -> str:
    h = bytes(u).hex()
    return "%s-%s-%s-%s-%s" % (h[0:8], h[8:12], h[12:16], h[16:20], h[20:32])


# ------------------------------------------------------------------------------------------------
# filepath.Walk + the five readers -> flat snapshot
# ------------------------------------------------------------------------------------------------
def _walk(root: str):
    """filepath.Walk order and Lstat semantics: yields (name, is_dir, err) for every visited
    entry; real directories are descended, symlinks are not followed."""
    try:
        st = os.lstat(root)
    except OSError:
        yield os.path.basename(root), False, True
        return
    import stat as _stat

    def rec(path, name, st):
        if not _stat.S_ISDIR(st.st_mode):
            yield name, False, False
            return
        try:
            names = sorted(os.listdir(path), key=lambda s: s.encode())
            err = False
        except OSError:
            names, err = [], True
        yield name, True, err
        if err:
            return
        for n in names:
            child = os.path.join(path, n)
            try:
                cst = os.lstat(child)
            except OSError:
                yield n, False, True
                return
            yield from rec(child, n, cst)

    yield from rec(root, os.path.basename(root), st)


def _read_file(path):
    try:
        with open(path, "rb") as f:
            return f.read()
    except OSError:
        return None


def _read_id(base, addr, prop):
    """readIDFromFileFunc :294-302 -> (string, err)"""
    data = _read_file(os.path.join(base, addr, prop))
    if data is None:
        return "", True
    if len(data) < 2:
        raise ReferencePanic("slice bounds out of range reading %s/%s" % (addr, prop))
    return data[2:].strip(b"\n").decode("latin-1"), False


def _read_link(base, addr, link):
    """readLinkFunc :323-331 -> (basename, err)"""
    try:
        target = os.readlink(os.path.join(base, addr, link))
    except OSError:
        return "", True
    return target.rsplit("/", 1)[-1], False


# unicode.IsSpace (Go): NOT the same set as Python's str.strip() default
_GO_SPACE = "\t\n\v\f\r \u0085\u00a0\u1680\u2028\u2029\u202f\u205f\u3000" + "".join(
    chr(c) for c in range(0x2000, 0x200B))


def _read_numa(base, addr):
    """readNUMANodeFunc :304-320 -> (raw value, err).  The clamp (<0 -> 0) is left to the GPU."""
    data = _read_file(os.path.join(base, addr, "numa_node"))
    if data is None:
        return 0, True
    try:
        s = data.decode("utf-8")
    except UnicodeDecodeError:
        s = data.decode("latin-1")
    s = s.strip(_GO_SPACE)  # strings.TrimSpace
    body = s[1:] if s[:1] in "+-" else s
    if not body or any(c not in "0123456789" for c in body):
        return 0, True
    v = int(s)
    if v < -(1 << 63) or v > (1 << 63) - 1:
        return 0, True
    return v, False


@dataclass
class PciSnapshot:
    recs: np.ndarray
    names: list            # Walk-order entry names (record i <-> names[i])
    packed_addr: bool      # True: recs.addr is the packed BDF; False: the Walk index
    group_names: list | None   # None: iommu_group is the number itself; else interned strings
    device_names: list | None = None   # None: recs.device is the id itself ("%04x"); else interned `device` strings


def snapshot_pci_tree(base_path: str) -> PciSnapshot:
    """Walk `base_path` like createIommuDeviceMap and record what each reader returned."""
    rows, names = [], []
    for name, is_dir, err in _walk(base_path):
        if err:      # :193-196 the walk aborts; entries seen so far stay
            break
        if is_dir:   # :197-200
            continue
        flags, vendor, device, group, driver, numa = 0, 0xFFFF, 0, "", L.DRV_NONE, 0
        v, e = _read_id(base_path, name, "vendor")
        if e:
            flags |= L.PF_VENDOR_ERR
        elif len(v) == 4 and all(c in HEXD for c in v):
            vendor = int(v, 16)
        if not e and v == "10de":
            # same short-circuit order as :212-238 — a later file is only touched when the
            # reference would touch it (so a panic can only happen where the reference panics)
            d, e = _read_link(base_path, name, "driver")
            if e:
                flags |= L.PF_DRIVER_ERR
            else:
                driver = {"vfio-pci": L.DRV_VFIO_PCI,
                          "nvgrace_gpu_vfio_pci": L.DRV_NVGRACE}.get(d, L.DRV_OTHER)
            if not e and driver in (L.DRV_VFIO_PCI, L.DRV_NVGRACE):
                group, e = _read_link(base_path, name, "iommu_group")
                if e:
                    flags |= L.PF_IOMMU_ERR
                else:
                    numa, e = _read_numa(base_path, name)
                    if e:
                        flags |= L.PF_NUMA_ERR
                    dv, e = _read_id(base_path, name, "device")
                    if e:
                        flags |= L.PF_DEVICE_ERR
                    else:
                        device = dv   # the reference keeps WHATEVER the file holds as the map key (:240, :294-302)
        rows.append((name, vendor, device, group, driver, flags, numa))
        names.append(name)
    packed = [parse_bdf(n) for n in names]
    packed_ok = all(p is not None for p in packed) and all(
        packed[i] < packed[i + 1] for i in range(len(packed) - 1))

    def canon_dec(s):
        return s.isdigit() and s.isascii() and (s == "0" or s[0] != "0") and int(s) < (1 << 32)

    groups_numeric = all(canon_dec(r[3]) for r in rows if r[3] != "")
    group_names, intern = (None, None) if groups_numeric else ([], {})
    # `device`: "%04x" strings travel as the number; anything else switches the column to index mode (interned
    # strings, like the groups): the GPU groups by the interned id, the host keeps the strings and asks
    # getDeviceName with the exact bytes
    devs = [r[2] for r in rows if isinstance(r[2], str)]
    devices_numeric = all(len(d) == 4 and all(c in HEXD for c in d) for d in devs)
    device_names, dintern = (None, None) if devices_numeric else ([], {})
    recs = np.zeros(len(rows), dtype=L.PCI_REC)
    for i, (name, vendor, device, group, driver, flags, numa) in enumerate(rows):
        if isinstance(device, str):
            if devices_numeric:
                device = int(device, 16)
            else:
                k = dintern.setdefault(device, len(dintern))
                if k == len(device_names):
                    device_names.append(device)
                if k > 0xFFFF:
                    raise L.KvgError(L.KVG_ERANGE, "more than 65536 distinct non-canonical device strings")
                device = k
        if group == "":
            g = 0
        elif groups_numeric:
            g = int(group)
        else:
            g = intern.setdefault(group, len(intern))
            if g == len(group_names):
                group_names.append(group)
        if not -32768 <= numa <= 32767:
            raise L.KvgError(L.KVG_ERANGE, "numa_node %d of %s does not fit int16" % (numa, name))
        recs[i] = (packed[i] if packed_ok else i, vendor, device, g, driver, flags, numa)
    return PciSnapshot(recs, names, packed_ok, group_names, device_names)


def _read_vgpu_raw(base, addr, prop):
    data = _read_file(os.path.join(base, addr, prop))
    return (None, True) if data is None else (data, False)


def _read_gpu_id_for_vgpu(base, addr):
    """readGpuIDForVgpuFunc :347-357"""
    try:
        target = os.readlink(os.path.join(base, addr))
    except OSError:
        return "", True
    parts = target.split("/")
    if len(parts) < 2:
        raise ReferencePanic("index out of range splitting link target %r" % target)
    return parts[-2].strip("\n"), False


@dataclass
class MdevSnapshot:
    recs: np.ndarray
    names: list
    raw_types: list            # raw mdev_type/name contents (bytes), dictionary order
    parent_names: list | None  # None: parent is a packed BDF; else interned strings
    uuid_ok: bool


def snapshot_mdev_tree(vgpu_base: str, pci_base: str) -> MdevSnapshot:
    rows, names = [], []
    type_ids, raw_types = {}, []
    for name, is_dir, err in _walk(vgpu_base):
        if err:
            break
        if is_dir:
            continue
        flags, tidx, parent, numa = 0, 0, "", 0
        raw, e = _read_vgpu_raw(vgpu_base, name, "mdev_type/name")
        if e:
            flags |= L.MF_TYPE_ERR
        else:
            tidx = type_ids.setdefault(raw, len(type_ids))
            if tidx == len(raw_types):
                raw_types.append(raw)
        if not e:  # :275 is only reached when the type read succeeded
            parent, e2 = _read_gpu_id_for_vgpu(vgpu_base, name)
            if e2:
                flags |= L.MF_PARENT_ERR
            else:
                numa, e3 = _read_numa(pci_base, parent)
                if e3:
                    flags |= L.MF_NUMA_ERR
        rows.append((name, parent, tidx, flags, numa))
        names.append(name)
    ppacked = [parse_bdf(r[1]) for r in rows if r[1] != ""]
    parents_packed = all(p is not None for p in ppacked)
    parent_names, intern = (None, None) if parents_packed else ([], {})

    def uuid_bytes(s):
        h = s.replace("-", "")
        if len(s) == 36 and len(h) == 32 and all(c in HEXD for c in h) and format_uuid(
                bytes.fromhex(h)) == s:
            return bytes.fromhex(h)
        return None

    ub = [uuid_bytes(n) for n in names]
    uuid_ok = all(u is not None for u in ub) and all(ub[i] < ub[i + 1] for i in range(len(ub) - 1))
    recs = np.zeros(len(rows), dtype=L.MDEV_REC)
    for i, (name, parent, tidx, flags, numa) in enumerate(rows):
        if parent == "":
            p = 0
        elif parents_packed:
            p = parse_bdf(parent)
        else:
            p = intern.setdefault(parent, len(intern))
            if p == len(parent_names):
                parent_names.append(parent)
        if uuid_ok:
            recs[i]["uuid"] = np.frombuffer(ub[i], dtype=np.uint8)
        else:
            recs[i]["uuid"][:4] = np.frombuffer(int(i).to_bytes(4, "big"), dtype=np.uint8)
        recs[i]["parent"], recs[i]["type_idx"], recs[i]["flags"] = p, tidx, flags
        recs[i]["parent_numa"] = numa
    return MdevSnapshot(recs, names, raw_types, parent_names, uuid_ok)


# ------------------------------------------------------------------------------------------------
# the five maps rebuilt from flat GPU results
# ------------------------------------------------------------------------------------------------
@dataclass
class NvidiaGpuDevice:      # device_plugin.go:50-53
    addr: str
    numaNode: int


@dataclass
class Maps:
    iommuMap: dict = field(default_factory=dict)       # :56
    deviceMap: dict = field(default_factory=dict)      # :59
    bdfToIommuMap: dict = field(default_factory=dict)  # :62
    vGpuMap: dict = field(default_factory=dict)        # :65
    gpuVgpuMap: dict = field(default_factory=dict)     # :68
    deviceNames: dict = field(default_factory=dict)    # key -> getDeviceName(key) ("" = miss)
    # held while the maps are swapped for a rediscovered set and while Allocate reads them
    lock: threading.Lock = field(default_factory=threading.Lock, compare=False, repr=False)

    def __getstate__(self):  # the maps travel between processes (sharded scans); the lock stays behind
        state = dict(self.__dict__)
        del state["lock"]
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)
        self.lock = threading.Lock()

    def swap(self, other: "Maps"):
        """Take over `other`'s maps in one step with respect to readers holding `lock`."""
        with self.lock:
            self.iommuMap, self.deviceMap, self.bdfToIommuMap = other.iommuMap, other.deviceMap, other.bdfToIommuMap
            self.vGpuMap, self.gpuVgpuMap, self.deviceNames = other.vGpuMap, other.gpuVgpuMap, other.deviceNames


def pci_maps_from_result(res: PciResult, snap: PciSnapshot | None = None, maps: Maps | None = None,
                         name_of=None) -> Maps:
    """name_of(key) -> getDeviceName(key): needed (and only used) when the snapshot carries the `device`
    strings in index mode — the GPU's per-survivor join is keyed by the numeric id and does not apply."""
    m = maps or Maps()
    m.iommuMap, m.deviceMap, m.bdfToIommuMap = {}, {}, {}  # :188-190
    s = res.survivors
    if snap is None or snap.packed_addr:
        addr = [format_bdf(int(a)) for a in s["addr"]]
    else:
        addr = [snap.names[int(a)] for a in s["addr"]]
    if snap is None or snap.group_names is None:
        gname = lambda g: str(int(g))
    else:
        gname = lambda g: snap.group_names[int(g)]
    numa = s["numa"]
    dev_index = snap is not None and snap.device_names is not None
    if dev_index and name_of is None:
        raise ValueError("snapshot carries device strings in index mode: pass name_of (Context.name_lookup)")
    for k in range(len(res.dev_keys)):
        key = snap.device_names[int(res.dev_keys[k])] if dev_index else "%04x" % int(res.dev_keys[k])
        idx = res.dev_perm[res.dev_off[k]:res.dev_off[k + 1]]
        m.deviceMap[key] = [NvidiaGpuDevice(addr[i], int(numa[i])) for i in idx]
        m.deviceNames[key] = name_of(key) if dev_index else res.name_at(int(res.dev_name_slot[k]))
    for k in range(len(res.grp_keys)):
        idx = res.grp_perm[res.grp_off[k]:res.grp_off[k + 1]]
        m.iommuMap[gname(res.grp_keys[k])] = [NvidiaGpuDevice(addr[i], int(numa[i])) for i in idx]
    for i in range(len(s)):
        m.bdfToIommuMap[addr[i]] = gname(s["iommu_group"][i])
    return m


def mdev_maps_from_result(res: MdevResult, snap: MdevSnapshot | None = None, maps: Maps | None = None) -> Maps:
    m = maps or Maps()
    m.vGpuMap, m.gpuVgpuMap = {}, {}  # :256-257
    s = res.survivors
    if snap is None or snap.uuid_ok:
        uid = [format_uuid(u) for u in s["uuid"]]
    else:
        uid = [snap.names[int(i)] for i in s["src"]]
    if snap is None or snap.parent_names is None:
        pname = lambda p: format_bdf(int(p))
    else:
        pname = lambda p: snap.parent_names[int(p)]
    for k in range(len(res.type_keys)):
        t = int(res.type_keys[k])
        label = res.labels[t].decode("latin-1")
        idx = res.type_perm[res.type_off[k]:res.type_off[k + 1]]
        m.vGpuMap[label] = [NvidiaGpuDevice(uid[i], int(s["numa"][i])) for i in idx]
        m.deviceNames[label] = res.type_names[t]
    for k in range(len(res.par_keys)):
        idx = res.par_perm[res.par_off[k]:res.par_off[k + 1]]
        m.gpuVgpuMap[pname(res.par_keys[k])] = [uid[i] for i in idx]
    return m


def canonical_dump(m: Maps) -> bytes:
    """Byte-identical to oracle kvo_dump for the same maps (SURVEY.md 8c)."""
    out = []
    bkey = lambda s: s.encode("latin-1")

    def dev_section(tag, mp):
        for key in sorted(mp, key=bkey):
            name = m.deviceNames.get(key, "")
            out.append("%s %s %s nvidia.com/%s %d\n" % (tag, key, name or "-", name or key,
                                                        len(mp[key])))
            out.extend("  %s %d\n" % (d.addr, d.numaNode) for d in mp[key])

    dev_section("D", m.deviceMap)
    for key in sorted(m.iommuMap, key=bkey):
        out.append("I %s %d\n" % (key, len(m.iommuMap[key])))
        out.extend("  %s %d\n" % (d.addr, d.numaNode) for d in m.iommuMap[key])
    for key in sorted(m.bdfToIommuMap, key=bkey):
        out.append("B %s %s\n" % (key, m.bdfToIommuMap[key]))
    dev_section("V", m.vGpuMap)
    for key in sorted(m.gpuVgpuMap, key=bkey):
        out.append("G %s %d\n" % (key, len(m.gpuVgpuMap[key])))
        out.extend("  %s\n" % u for u in m.gpuVgpuMap[key])
    return "".join(out).encode("latin-1")


# ------------------------------------------------------------------------------------------------
# the controller half the Go host keeps (payload only — the gRPC servers stay in Go)
# ------------------------------------------------------------------------------------------------
@dataclass
class PluginSpec:
    """What NewGenericDevicePlugin / NewGenericVGpuDevicePlugin + Register would be given."""
    key: str
    device_name: str          # getDeviceName(key) or the key itself (:125-128, :153-155)
    resource_name: str        # "nvidia.com/<name>"   generic_device_plugin.go:299
    socket_path: str          # generic_device_plugin.go:87 / generic_vgpu_device_plugin.go:69
    env_key: str              # generic_device_plugin.go:420 / generic_vgpu_device_plugin.go:223
    devs: list                # [{ID, Health, Topology:{Nodes:[{ID}]}}]  (:111-123, :141-150)
    vgpu: bool = False


@dataclass
class PluginEvent:
    """What a rediscovery asks of the plugin servers: "start" a plugin for a new deviceMap / vGpuMap key,
    "stop" the plugin of a removed key, "update" the device list of a changed key, or "replace_all" (stop
    every plugin, start one per key of the new maps: what a restart of the plugin does)."""
    kind: str
    key: str | None = None
    vgpu: bool = False
    spec: PluginSpec | None = None


class DiscoveryScan:
    """InitiateDevicePlugin's scan half (device_plugin.go:89-96) on the GPU."""

    def __init__(self, pci_ids_path: str = "/usr/pci.ids", base_path: str = "/sys/bus/pci/devices",
                 vgpu_base_path: str = "/sys/bus/mdev/devices", device: int = 0):
        self.pciIdsFilePath, self.basePath, self.vGpuBasePath = pci_ids_path, base_path, vgpu_base_path
        self.ctx = Context(device)
        self.maps = Maps()
        self._loaded_path = None
        # rediscover(): the raw mdev type dictionary only ever grows, so canonical type ids stay stable
        self._raw_types, self._type_index = [], {}

    def close(self):
        self.ctx.close()

    def _ensure_table(self):
        if self._loaded_path == self.pciIdsFilePath:
            return
        # (kvg_pciids_load drops the rescan baselines: the next rediscover() starts from "everything added")
        data = _read_file(self.pciIdsFilePath)
        # unreadable file -> getDeviceName returns "" for every key (:373-377): an empty table
        self.ctx.pciids_load(data if data is not None else b"")
        self._loaded_path = self.pciIdsFilePath

    def get_device_name(self, device_id: str) -> str:
        self._ensure_table()
        return self.ctx.name_lookup(device_id)

    def create_iommu_device_map(self) -> Maps:
        self._ensure_table()
        try:
            snap = snapshot_pci_tree(self.basePath)
        except ReferencePanic:
            raise
        res = self.ctx.scan_pci(snap.recs)
        return pci_maps_from_result(res, snap, self.maps, name_of=self.ctx.name_lookup)

    def create_vgpu_id_map(self) -> Maps:
        self._ensure_table()
        snap = snapshot_mdev_tree(self.vGpuBasePath, self.basePath)
        res = self.ctx.scan_mdev(snap.recs, snap.raw_types)
        return mdev_maps_from_result(res, snap, self.maps)

    def create_device_plugins(self) -> list:
        return plugin_specs_from_maps(self.maps)

    def rediscover(self) -> list:
        """Snapshot both trees again and bring self.maps up to date (in place, one swap).  Returns the
        PluginEvents that take the plugin servers from the previous maps to the new ones.  Snapshots in
        numeric mode go through the GPU diff; a snapshot in index mode has no stable identities and
        yields [PluginEvent("replace_all")]."""
        self._ensure_table()
        psnap = snapshot_pci_tree(self.basePath)
        msnap = snapshot_mdev_tree(self.vGpuBasePath, self.basePath)
        remap = []
        for raw in msnap.raw_types:
            if raw not in self._type_index:
                self._type_index[raw] = len(self._raw_types)
                self._raw_types.append(raw)
            remap.append(self._type_index[raw])
        remap = np.array(remap, dtype=np.uint16)
        recs = msnap.recs.copy()
        if len(remap):
            ok = (recs["flags"] & L.MF_TYPE_ERR) == 0
            recs["type_idx"][ok] = remap[recs["type_idx"][ok]]
        numeric = (psnap.packed_addr and psnap.group_names is None and psnap.device_names is None
                   and msnap.uuid_ok and msnap.parent_names is None)
        fresh = Maps()
        if not numeric:
            self.ctx.rescan_reset()
            pci_maps_from_result(self.ctx.scan_pci(psnap.recs), psnap, fresh, name_of=self.ctx.name_lookup)
            mdev_maps_from_result(self.ctx.scan_mdev(recs, self._raw_types), msnap, fresh)
            self.maps.swap(fresh)
            return [PluginEvent("replace_all")]
        pr = self.ctx.rescan_pci(psnap.recs)
        mr = self.ctx.rescan_mdev(recs, self._raw_types)
        pci_maps_from_result(pr.scan, psnap, fresh, name_of=self.ctx.name_lookup)
        mdev_maps_from_result(mr.scan, msnap, fresh)
        self.maps.swap(fresh)
        specs = {(s.vgpu, s.key): s for s in plugin_specs_from_maps(fresh)}
        events = []
        for vgpu, delta, key_of in ((False, pr.dev, lambda k: "%04x" % k),
                                    (True, mr.type, lambda k: mr.scan.labels[k].decode("latin-1"))):
            events += [PluginEvent("stop", key_of(int(k)), vgpu) for k in delta.removed]
            events += [PluginEvent("start", key_of(int(k)), vgpu, specs[(vgpu, key_of(int(k)))]) for k in delta.added]
            events += [PluginEvent("update", key_of(int(k)), vgpu, specs[(vgpu, key_of(int(k)))])
                       for k in delta.changed]
        return events


def plugin_specs_from_maps(maps: Maps) -> list:
    """createDevicePlugins' payload half (device_plugin.go:99-157): one PluginSpec per deviceMap key,
    then one per vGpuMap key; name falls back to the key when getDeviceName returned ""."""
    specs = []
    for key, devs in maps.deviceMap.items():
        name = maps.deviceNames.get(key, "") or key
        specs.append(PluginSpec(
            key, name, "%s/%s" % (DEVICE_NAMESPACE, name),
            "%skubevirt-%s.sock" % (DEVICE_PLUGIN_PATH, name),
            "%s_%s" % (GPU_PREFIX, name.upper()),
            [{"ID": d.addr, "Health": HEALTHY, "Topology": {"Nodes": [{"ID": d.numaNode}]}}
             for d in devs]))
    for key, devs in maps.vGpuMap.items():
        name = maps.deviceNames.get(key, "") or key
        specs.append(PluginSpec(
            key, name, "%s/%s" % (DEVICE_NAMESPACE, name),
            "%skubevirt-%s.sock" % (DEVICE_PLUGIN_PATH, name),
            "%s_%s" % (VGPU_PREFIX, name.upper()),
            [{"ID": d.addr, "Health": HEALTHY, "Topology": {"Nodes": [{"ID": d.numaNode}]}}
             for d in devs], vgpu=True))
    return specs
