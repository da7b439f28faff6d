"""The consumer side of the scan: the kubelet-facing DevicePlugin servers fed by the GPU results.

SURVEY.md 8(f): (1) host glue + a mock kubelet to replay Register -> ListAndWatch -> Allocate,
(2) Allocate-time re-validation as ONE batched re-scan, (3) a health feed driven by the K6 delta
kernel, (4) GetPreferredAllocation NUMA packing and EGM path selection (host logic, pinned by the
reference's own tests).  Function by function this mirrors

    pkg/device_plugin/generic_device_plugin.go       (passthrough plugin)
    pkg/device_plugin/generic_vgpu_device_plugin.go  (vGPU plugin)

with the same names, argument meaning and error strings, so tests/test_serve.py reads like the
reference's generic_device_plugin_test.go.  In a deployment these servers stay in Go
(INTEGRATION.md); this Python mirror exists so that "drops in behind Register / ListAndWatch /
Allocate" is testable end to end in an image without a Go toolchain.

Nothing here computes on the CPU what the scan computes on the GPU: the maps come from
plugin.DiscoveryScan (libkvgpu.so); the re-validation's classification goes through
Context.scan_pci (K3); the health feed through Context.health_rescan (K6).
"""
from __future__ import annotations

import os
import queue
import sys
import threading
import time
from concurrent import futures
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L
from . import dpapi
from .plugin import (DEVICE_NAMESPACE, GPU_PREFIX, VGPU_PREFIX, Maps, PluginSpec, ReferencePanic, _read_id,
                     _read_link, _read_vgpu_raw, plugin_specs_from_maps)

VFIO_DEVICE_PATH = "/dev/vfio"      # generic_device_plugin.go:54
IOMMU_DEVICE_PATH = "/dev/iommu"    # :55
EGM_CLASS_PATH = "/sys/class/egm"   # :56
DEVICE_DIR = "/dev"
NVIDIA_VENDOR_ID = "10de"           # device_plugin.go:46
CONNECTION_TIMEOUT = 5.0            # generic_device_plugin.go:53


class AllocateError(Exception):
    """An error return of Allocate / GetPreferredAllocation (the text is the reference's)."""


# ------------------------------------------------------------------------------------------------
# host logic, pinned by the reference's tests (tests/golden/plugin_vectors.json)
# ------------------------------------------------------------------------------------------------
def preferred_allocation(devs, available, must_include, allocation_size) -> list:
    """GetPreferredAllocation for ONE container request (generic_device_plugin.go:470-608).

    devs: iterable of (device id, numa node or None).  Must-include devices first (request order),
    then try to complete from a single NUMA node — nodes of the must-include devices first, then
    nodes in order of first appearance in `available` — else fall back to kubelet order."""
    device_to_numa = {d: n for d, n in devs if n is not None}

    def numa_of(dev_id):
        return device_to_numa.get(dev_id, -1)

    numa_to_devices, node_order = {}, []
    for dev_id in available:
        node = numa_of(dev_id)
        if node not in numa_to_devices:
            numa_to_devices[node] = []
            node_order.append(node)
        numa_to_devices[node].append(dev_id)

    preferred, chosen, selected_per_node = [], set(), {}

    def add(dev_id):
        if dev_id in chosen:
            return
        chosen.add(dev_id)
        node = numa_of(dev_id)
        selected_per_node[node] = selected_per_node.get(node, 0) + 1
        preferred.append(dev_id)

    selected_node_order = []
    for dev_id in must_include:
        if dev_id in chosen:
            continue
        add(dev_id)
        node = numa_of(dev_id)
        if node not in selected_node_order:
            selected_node_order.append(node)
    if len(preferred) > allocation_size:
        raise AllocateError("number of MustIncludeDeviceIDs (%d) exceeds allocation size (%d)"
                            % (len(preferred), allocation_size))
    if len(preferred) < allocation_size:
        target = None
        candidates = selected_node_order + [n for n in node_order if n not in selected_node_order]
        for node in candidates:
            free = sum(1 for d in numa_to_devices.get(node, []) if d not in chosen)
            if selected_per_node.get(node, 0) + free >= allocation_size:
                target = node
                break
        # the reference encodes "no node" as -1, which is also the id of devices without topology:
        # such a pseudo-node is never used as a target (:552-575)
        if target is not None and target != -1:
            for dev_id in numa_to_devices.get(target, []):
                if len(preferred) >= allocation_size:
                    break
                add(dev_id)
    if len(preferred) < allocation_size:
        for dev_id in available:
            if len(preferred) >= allocation_size:
                break
            add(dev_id)
    return preferred


@dataclass
class EGMDeviceInfo:      # generic_device_plugin.go:62-65
    dev_path: str
    gpu_bdfs: list


def discover_egm_devices(root_path: str = "/") -> list:
    """discoverEGMDevicesFunc :120-157 (a missing class directory is not an error)."""
    class_dir = os.path.join(root_path, EGM_CLASS_PATH.lstrip("/"))
    try:
        entries = sorted(os.listdir(class_dir))
    except FileNotFoundError:
        return []
    out = []
    for name in entries:
        if not name.startswith("egm"):
            continue
        try:
            with open(os.path.join(class_dir, name, "gpu_devices"), "rb") as f:
                raw = f.read().decode("utf-8", "replace")
        except OSError:
            continue
        bdfs = raw.split()
        if not bdfs:
            continue
        dev_path = os.path.join(DEVICE_DIR, name)
        if not os.path.exists(os.path.join(root_path, dev_path.lstrip("/"))):
            continue
        out.append(EGMDeviceInfo(dev_path, bdfs))
    out.sort(key=lambda e: e.dev_path)
    return out


def egm_paths_for_allocated_gpus(allocated_bdfs, egm_devices) -> list:
    """egmPathsForAllocatedGPUs :159-184: an EGM node is injected only when ALL its GPUs are allocated."""
    allocated = {b.strip().lower() for b in allocated_bdfs}
    return sorted(e.dev_path for e in (egm_devices or [])
                  if all(g.strip().lower() in allocated for g in e.gpu_bdfs))


def supports_iommufd(root_path: str = "/") -> bool:
    """supportsIOMMUFD :692-701"""
    try:
        os.stat(os.path.join(root_path, IOMMU_DEVICE_PATH.lstrip("/")))
        return True
    except FileNotFoundError:
        return False
    except OSError as e:
        raise AllocateError("could not determine iommufd support: %s" % e)


def read_vfio_dev(base_path: str, addr: str) -> str:
    """readVFIODev :702-716: the first vfio* directory under <addr>/vfio-dev."""
    d = os.path.join(base_path, addr, "vfio-dev")
    for name in sorted(os.listdir(d)):          # os.ReadDir sorts by filename
        if os.path.isdir(os.path.join(d, name)) and name.startswith("vfio"):
            return name
    raise OSError("no iommufd device found")


# ------------------------------------------------------------------------------------------------
# Allocate-time re-validation as one batched re-scan (SURVEY.md 8(f) rank 2)
# ------------------------------------------------------------------------------------------------
class BatchRevalidator:
    """Re-check every device of every requested IOMMU group in ONE pass of the classification
    kernel instead of one readLink + one readIDFromFile round per device
    (generic_device_plugin.go:387-399).

    The sysfs reads use the reference's own readers, in the reference's order; what they returned
    becomes ordinary scan records (index mode: addr = position in the batch, iommu_group = interned
    group string).  The record's driver is pinned to vfio-pci and its device id to a constant,
    because Allocate re-checks ONLY the group link and the vendor — with that, K3's predicate
    (vendor == 10de, no vendor / iommu read error) is exactly the reference's acceptance test and
    the survivor's group id says whether the link still points at the expected group."""

    def __init__(self, scan_pci, base_path: str = "/sys/bus/pci/devices",
                 read_link=_read_link, read_id=_read_id):
        self.scan_pci, self.base_path = scan_pci, base_path
        self.read_link, self.read_id = read_link, read_id

    def __call__(self, pairs):
        """pairs: [(addr, expected iommu group)] in the order the reference would visit them.
        Returns the index of the first device the reference would reject, or None.  A reader panic
        (short vendor file) is re-raised only if the reference would have reached that read."""
        n = len(pairs)
        if n == 0:
            return None
        recs = np.zeros(n, dtype=L.PCI_REC)
        intern, panics = {}, {}
        for i, (addr, expect) in enumerate(pairs):
            want = intern.setdefault(expect, len(intern))
            flags, vendor, group = 0, 0xFFFF, want
            got, err = self.read_link(self.base_path, addr, "iommu_group")
            if err:
                flags |= L.PF_IOMMU_ERR
            else:
                group = intern.setdefault(got, len(intern))
            try:
                v, err = self.read_id(self.base_path, addr, "vendor")
            except ReferencePanic as e:
                panics[i] = e
                v, err = "", True
            if err:
                flags |= L.PF_VENDOR_ERR
            elif v == NVIDIA_VENDOR_ID:
                vendor = 0x10de
            recs[i] = (i, vendor, 0, group, L.DRV_VFIO_PCI, flags, 0)
        res = self.scan_pci(recs)
        ok_group = {int(s["addr"]): int(s["iommu_group"]) for s in res.survivors}
        for i, (addr, expect) in enumerate(pairs):
            link_ok = not (int(recs[i]["flags"]) & L.PF_IOMMU_ERR) and int(recs[i]["iommu_group"]) == intern[expect]
            if link_ok and i in panics:   # the reference reads the vendor only after the link check passed
                raise panics[i]
            if ok_group.get(i) != intern[expect]:
                return i
        return None


# ------------------------------------------------------------------------------------------------
# the plugins
# ------------------------------------------------------------------------------------------------
def devices_from_spec(spec: PluginSpec) -> list:
    """PluginSpec.devs -> []*pluginapi.Device (device_plugin.go:111-123, :141-150)."""
    return [dpapi.Device(ID=d["ID"], health=d["Health"],
                         topology=dpapi.TopologyInfo(nodes=[dpapi.NUMANode(ID=n["ID"]) for n in d["Topology"]["Nodes"]]))
            for d in spec.devs]


class _PluginBase:
    """Start / Stop / Register / ListAndWatch shared by both plugins
    (generic_device_plugin.go:216-349, generic_vgpu_device_plugin.go:75-205)."""
    vgpu = False

    def __init__(self, device_name: str, devs: list, socket_dir: str = dpapi.DEVICE_PLUGIN_PATH,
                 kubelet_socket: str | None = None):
        self.device_name = device_name
        self.devs = list(devs)
        self.socket_path = os.path.join(socket_dir, "kubevirt-%s.sock" % device_name)
        self.kubelet_socket = kubelet_socket or os.path.join(socket_dir, "kubelet.sock")
        self.server = None
        self._events = queue.Queue()     # ("healthy" | "unhealthy", device id): the two Go channels
        self._stop = threading.Event()
        self._term = threading.Event()
        self._lock = threading.Lock()

    # -- the two channels of the reference (dpi.healthy / dpi.unhealthy)
    def healthy(self, dev_id: str):
        self._events.put(("healthy", dev_id))

    def unhealthy(self, dev_id: str):
        self._events.put(("unhealthy", dev_id))

    def set_devices(self, devs: list):
        """A rediscovery changed what this plugin advertises: ListAndWatch re-sends the whole new list."""
        with self._lock:
            self.devs = list(devs)
        self._events.put(("devices", None))

    def resource_name(self) -> str:
        return "%s/%s" % (DEVICE_NAMESPACE, self.device_name)

    # -- gRPC methods
    def GetDevicePluginOptions(self, request, context):
        # passthrough: preferred allocation available (:451-457); vGPU: not (:252-257)
        return dpapi.DevicePluginOptions(pre_start_required=False,
                                         get_preferred_allocation_available=not self.vgpu)

    def PreStartContainer(self, request, context):
        return dpapi.PreStartContainerResponse()

    def ListAndWatch(self, request, context):
        """:312-349 — send the list once, then the whole list again after every health flip."""
        yield dpapi.ListAndWatchResponse(devices=self.devs)
        while not (self._stop.is_set() or self._term.is_set()):
            if context is not None and not context.is_active():
                return
            try:
                kind, dev_id = self._events.get(timeout=0.02)
            except queue.Empty:
                continue
            with self._lock:
                if kind != "devices":        # "devices": set_devices replaced the whole list
                    for dev in self.devs:
                        if dev.ID == dev_id:
                            dev.health = dpapi.HEALTHY if kind == "healthy" else dpapi.UNHEALTHY
                devs = self.devs
            yield dpapi.ListAndWatchResponse(devices=devs)

    # -- lifecycle
    def _handlers(self):
        import grpc
        table = {}
        for mname, (req, resp, stream) in dpapi.SERVICES["DevicePlugin"].items():
            fn = self._wrap(getattr(self, mname))
            make = grpc.unary_stream_rpc_method_handler if stream else grpc.unary_unary_rpc_method_handler
            table[mname] = make(fn, request_deserializer=dpapi.MESSAGES[req].FromString,
                                response_serializer=dpapi.MESSAGES[resp].SerializeToString)
        return grpc.method_handlers_generic_handler(dpapi.service_name("DevicePlugin"), table)

    @staticmethod
    def _wrap(fn):
        import grpc
        import inspect
        if inspect.isgeneratorfunction(fn):
            return fn

        def call(request, context):
            try:
                return fn(request, context)
            except AllocateError as e:    # a Go `return nil, err` -> status UNKNOWN with the text
                context.abort(grpc.StatusCode.UNKNOWN, str(e))
        return call

    def start(self):
        """Start :216-257: serve on the plugin socket, then Register with the kubelet."""
        import grpc
        if self.server is not None:
            raise RuntimeError("gRPC server already started")
        self._stop.clear()
        self._term.clear()
        self.cleanup()
        self.server = grpc.server(futures.ThreadPoolExecutor(max_workers=8))
        self.server.add_generic_rpc_handlers((self._handlers(),))
        self.server.add_insecure_port("unix://" + self.socket_path)
        self.server.start()
        self.register()

    def stop(self):
        """Stop :260-273"""
        if self.server is None:
            return
        self._term.set()
        self.server.stop(0.2).wait(2.0)
        self.server = None
        self.cleanup()

    def restart(self):
        """restart :276-287 (kubelet restarted: the plugin socket was removed under us)."""
        if self.server is None:
            raise RuntimeError("grpc server instance not found for %s" % self.device_name)
        self.stop()
        self.start()

    def cleanup(self):
        try:
            os.remove(self.socket_path)
        except FileNotFoundError:
            pass

    def register(self):
        """Register :289-309"""
        import grpc
        with grpc.insecure_channel("unix://" + self.kubelet_socket) as ch:
            grpc.channel_ready_future(ch).result(timeout=CONNECTION_TIMEOUT)
            call = ch.unary_unary(dpapi.method_path("Registration", "Register"),
                                  request_serializer=dpapi.RegisterRequest.SerializeToString,
                                  response_deserializer=dpapi.Empty.FromString)
            call(dpapi.RegisterRequest(version=dpapi.VERSION, endpoint=os.path.basename(self.socket_path),
                                       resource_name=self.resource_name()), timeout=CONNECTION_TIMEOUT)


class GenericDevicePlugin(_PluginBase):
    """The passthrough plugin (generic_device_plugin.go).  `maps` supplies what returnIommuMap /
    returnBdfToIommuMap supply in the reference; `revalidate` is the Allocate-time re-check
    (default: BatchRevalidator over the given scan function)."""

    def __init__(self, device_name, device_path, devs, maps: Maps, *, revalidate=None,
                 base_path="/sys/bus/pci/devices", root_path="/", discover_egm=None, **kw):
        super().__init__(device_name, devs, **kw)
        self.device_path, self.maps = device_path, maps
        self.base_path, self.root_path = base_path, root_path
        self.revalidate = revalidate
        self.discover_egm = discover_egm or (lambda: discover_egm_devices(self.root_path))

    def GetPreferredAllocation(self, request, context):
        resp = dpapi.PreferredAllocationResponse()
        devs = [(d.ID, d.topology.nodes[0].ID if len(d.topology.nodes) else None) for d in self.devs]
        for req in request.container_requests:
            ids = preferred_allocation(devs, list(req.available_deviceIDs), list(req.must_include_deviceIDs),
                                       int(req.allocation_size))
            resp.container_responses.append(dpapi.ContainerPreferredAllocationResponse(deviceIDs=ids))
        return resp

    def Allocate(self, request, context):
        """:352-447.  The sequence of checks, device specs and env values is the reference's; the
        per-device re-validation of a request is handed to `self.revalidate` as one batch."""
        if self.revalidate is None:
            raise AllocateError("no re-validation function configured (the scan context is required)")
        responses = dpapi.AllocateResponse()
        env_list = {}                       # declared OUTSIDE the request loop in the reference (:361)
        iommufd = supports_iommufd(self.root_path)
        try:
            egm_devices = self.discover_egm()
        except Exception:                   # :366-370 a discovery failure only disables EGM mounts
            egm_devices = None
        for req in request.container_requests:
            specs, seen = [], set()

            def append_spec(host_path):
                if host_path not in seen:   # appendDeviceSpec :108-118
                    seen.add(host_path)
                    specs.append(dpapi.DeviceSpec(host_path=host_path, container_path=host_path, permissions="mrw"))

            with self.maps.lock:           # a rediscovery swaps both maps together (Maps.swap)
                iommu_map, bdf_to_iommu = self.maps.iommuMap, self.maps.bdfToIommuMap
            # plan: which devices would be visited, in order, and where a lookup error would stop
            plan, lookup_error_at = [], None
            for k, bdf in enumerate(req.devices_ids):
                group = bdf_to_iommu.get(bdf)
                members = iommu_map.get(group, []) if group is not None else []
                if group is None or not members:
                    lookup_error_at = (k, bdf)
                    break
                plan.append((bdf, group, members))
            pairs = [(d.addr, group) for _, group, members in plan for d in members]
            bad = self.revalidate(pairs)    # ONE batch for the whole container request
            pos = 0
            for bdf, group, members in plan:   # replay in the reference's order: the FIRST error wins
                addrs, found = [], False
                for dev in members:
                    if bad is not None and pos == bad:
                        raise AllocateError("invalid allocation request: unknown device: %s" % dev.addr)
                    pos += 1
                    addrs.append(dev.addr)
                    found = found or dev.addr == bdf
                    if iommufd:
                        try:
                            vfiodev = read_vfio_dev(self.base_path, dev.addr)
                        except OSError as e:
                            raise AllocateError("could not determine iommufd device for device %s: %s"
                                                % (dev.addr, e))
                        append_spec(os.path.join(VFIO_DEVICE_PATH, "devices", vfiodev))
                if not found:
                    raise AllocateError("invalid allocation request: unknown device: %s" % bdf)
                append_spec(os.path.join(VFIO_DEVICE_PATH, "vfio"))
                append_spec(os.path.join(VFIO_DEVICE_PATH, group))
                if iommufd:
                    append_spec(IOMMU_DEVICE_PATH)
                env_list.setdefault("%s_%s" % (GPU_PREFIX, self.device_name.upper()), []).extend(addrs)
            if lookup_error_at is not None:
                raise AllocateError("invalid allocation request: unknown device: %s" % lookup_error_at[1])
            for path in egm_paths_for_allocated_gpus(list(req.devices_ids), egm_devices):
                append_spec(path)
            responses.container_responses.append(dpapi.ContainerAllocateResponse(
                envs={k: ",".join(v) for k, v in env_list.items()}, devices=specs))   # buildEnv :100-106
        return responses


class GenericVGpuDevicePlugin(_PluginBase):
    """The vGPU plugin (generic_vgpu_device_plugin.go)."""
    vgpu = True

    def __init__(self, device_name, device_path, devs, *, vgpu_base_path="/sys/bus/mdev/devices",
                 read_vgpu_id=None, **kw):
        super().__init__(device_name, devs, **kw)
        self.device_path, self.vgpu_base_path = device_path, vgpu_base_path
        self.read_vgpu_id = read_vgpu_id or _read_vgpu_label

    def GetPreferredAllocation(self, request, context):
        # "has not been implemented" in the reference: returns (nil, nil) (:262-271) -> empty message
        return dpapi.PreferredAllocationResponse()

    def Allocate(self, request, context):
        """:208-245 — ids whose type label no longer equals the plugin's name are skipped, not errors."""
        responses = dpapi.AllocateResponse()
        for req in request.container_requests:
            env_list = {}
            for dev_id in req.devices_ids:
                label, err = self.read_vgpu_id(self.vgpu_base_path, dev_id, "mdev_type/name")
                if err or label != self.device_name:
                    continue
                env_list.setdefault("%s_%s" % (VGPU_PREFIX, self.device_name.upper()), []).append(dev_id)
            spec = dpapi.DeviceSpec(host_path=VFIO_DEVICE_PATH, container_path=VFIO_DEVICE_PATH, permissions="mrw")
            responses.container_responses.append(dpapi.ContainerAllocateResponse(
                envs={k: ",".join(v) for k, v in env_list.items()}, devices=[spec]))
        return responses


def _read_vgpu_label(base, addr, prop):
    """readVgpuIDFromFileFunc :334-344 for ONE id at Allocate time: trim '\\n', \\s+ -> '_'."""
    import re
    raw, err = _read_vgpu_raw(base, addr, prop)
    if err:
        return "", True
    return re.sub(rb"[\t\n\f\r ]+", b"_", raw.strip(b"\n")).decode("latin-1"), False


def plugins_from_specs(specs, maps: Maps, revalidate, **kw) -> list:
    """createDevicePlugins' server half (device_plugin.go:99-157): one plugin object per spec."""
    out = []
    for spec in specs:
        devs = devices_from_spec(spec)
        if spec.vgpu:
            out.append(GenericVGpuDevicePlugin(spec.device_name, "vgpu", devs,
                                               **{k: v for k, v in kw.items() if k in ("socket_dir", "kubelet_socket",
                                                                                          "vgpu_base_path")}))
        else:
            out.append(GenericDevicePlugin(spec.device_name, VFIO_DEVICE_PATH, devs, maps, revalidate=revalidate,
                                           **{k: v for k, v in kw.items() if k != "vgpu_base_path"}))
    return out


# ------------------------------------------------------------------------------------------------
# health feed driven by the K6 delta kernel (SURVEY.md 8(f) rank 3)
# ------------------------------------------------------------------------------------------------
class HealthRescanFeed:
    """Periodic re-snapshot -> Context.health_rescan (K6) -> healthy / unhealthy events.

    `snapshot()` returns (records, ids): the PCI snapshot in a FIXED device order and the device id
    of every record.  Each transition the kernel reports ((index << 1) | alive) is routed to the
    plugin that advertises that id.  The first tick only establishes the alive set."""

    def __init__(self, health_rescan, snapshot, plugins, period_s: float = 0.001):
        self.health_rescan, self.snapshot, self.period_s = health_rescan, snapshot, period_s
        self.owner = {d.ID: p for p in plugins for d in p.devs}
        self._primed = False
        self._stop = threading.Event()
        self._thread = None

    def tick(self) -> int:
        recs, ids = self.snapshot()
        delta = self.health_rescan(recs)
        sent = 0
        if self._primed:
            for word in delta.changed:
                idx, alive = int(word) >> 1, int(word) & 1
                plugin = self.owner.get(ids[idx])
                if plugin is not None:
                    (plugin.healthy if alive else plugin.unhealthy)(ids[idx])
                    sent += 1
        self._primed = True
        return sent

    def start(self):
        def loop():
            while not self._stop.is_set():
                self.tick()
                time.sleep(self.period_s)
        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(2.0)


# ------------------------------------------------------------------------------------------------
# runtime rediscovery: GPU-diffed rescans start, stop and update plugins
# ------------------------------------------------------------------------------------------------
class RediscoveryFeed:
    """Every `period_s`: ds.rediscover() (DiscoveryScan) and apply its PluginEvents to `plugins`, a dict
    (vgpu, key) -> plugin shared with the caller.  start: build, start (register with the kubelet) and watch
    a plugin; stop: stop it; update: replace its device list, which ListAndWatch re-sends whole;
    replace_all: stop everything and start one plugin per key of the new maps.  `plugin_kw` are the
    keyword arguments of plugins_from_specs (socket_dir, base_path, ...); `revalidate` goes to passthrough
    plugins."""

    def __init__(self, ds, plugins: dict, period_s: float, revalidate=None, watch: bool = True, **plugin_kw):
        self.ds, self.plugins, self.period_s = ds, plugins, period_s
        self.revalidate, self.watch, self.plugin_kw = revalidate, watch, plugin_kw
        self.watchers = {}
        self._stop = threading.Event()
        self._thread = None

    def _start(self, spec):
        plugin = plugins_from_specs([spec], self.ds.maps, self.revalidate, **self.plugin_kw)[0]
        plugin.start()
        self.plugins[(spec.vgpu, spec.key)] = plugin
        if self.watch:
            w = DeviceNodeWatcher(plugin)
            w.start()
            self.watchers[(spec.vgpu, spec.key)] = w

    def _stop_one(self, k):
        w = self.watchers.pop(k, None)
        if w is not None:
            w.stop()
        p = self.plugins.pop(k, None)
        if p is not None:
            p.stop()

    def tick(self) -> list:
        events = self.ds.rediscover()
        for ev in events:
            k = (ev.vgpu, ev.key)
            try:
                if ev.kind == "replace_all":
                    for old in list(self.plugins):
                        self._stop_one(old)
                    for spec in plugin_specs_from_maps(self.ds.maps):
                        self._start(spec)
                elif ev.kind == "stop":
                    self._stop_one(k)
                elif ev.kind == "update" or (ev.kind == "start" and k in self.plugins):
                    self.plugins[k].set_devices(devices_from_spec(ev.spec))
                    if k in self.watchers:   # the watcher maps device nodes through the previous bdfToIommuMap
                        self.watchers.pop(k).stop()
                        w = DeviceNodeWatcher(self.plugins[k])
                        w.start()
                        self.watchers[k] = w
                else:
                    self._start(ev.spec)
            except Exception as e:        # noqa: BLE001  a failed start is logged, the rest go on (:131-137)
                print("kvgpu: rediscovery: %s %s: %s" % (ev.kind, ev.key, e), file=sys.stderr)
        return events

    def start(self):
        def loop():
            while not self._stop.wait(self.period_s):
                try:
                    self.tick()
                except Exception as e:    # noqa: BLE001  a failed tick keeps the current plugins
                    print("kvgpu: rediscovery failed: %s" % e, file=sys.stderr)
        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(5.0)
        for w in self.watchers.values():
            w.stop()
        self.watchers.clear()


# ------------------------------------------------------------------------------------------------
# NVML XID events -> vGPU health (generic_vgpu_device_plugin.go:330-339 and watchXIDsFunc :387-433)
# ------------------------------------------------------------------------------------------------
XID_APPLICATION_ERRORS = (31, 43, 45)   # :413-417 "Application errors: the GPU should still be healthy"


class XidEventRouter:
    """The decision logic between an NVML XidCriticalError event and the `unhealthy` channel of a vGPU plugin,
    without NVML itself (the binding stays in the Go host; out of scope here):

      on_event(xid, uuid)    XIDs 31 / 43 / 45 are ignored (:415); an event without a device UUID marks EVERY GPU
                             (:419-424); otherwise the GPU with that UUID (:427-431)
      on_unsupported(uuid)   registration failed with "Not Supported": that GPU is marked at once (:392-397)
      a marked GPU           -> every vGPU of returnGpuVgpuMap()[gpu.PCI.BusID] goes to plugin.unhealthy (:333-338)

    `gpus`: list of (uuid, bus_id) in NVML enumeration order; `gpu_vgpu_map`: the scan's gpuVgpuMap
    (parent BDF -> [mdev uuid]); `plugins`: the vGPU plugins (an id is routed to the plugin that advertises it;
    the reference sends it down ITS OWN channel whether or not the id is its own — ListAndWatch then finds no
    such device and changes nothing, :186-199)."""

    def __init__(self, gpus, gpu_vgpu_map, plugins):
        self.gpus, self.gpu_vgpu_map = list(gpus), gpu_vgpu_map
        self.owner = {d.ID: p for p in plugins for d in p.devs}

    def _mark(self, bus_id) -> int:
        sent = 0
        for vgpu in self.gpu_vgpu_map.get(bus_id, []):
            plugin = self.owner.get(vgpu)
            if plugin is not None:
                plugin.unhealthy(vgpu)
                sent += 1
        return sent

    def on_unsupported(self, uuid) -> int:
        return sum(self._mark(bus) for u, bus in self.gpus if u == uuid)

    def on_event(self, xid: int, uuid=None) -> int:
        if xid in XID_APPLICATION_ERRORS:
            return 0
        if not uuid:
            return sum(self._mark(bus) for _, bus in self.gpus)
        return sum(self._mark(bus) for u, bus in self.gpus if u == uuid)


# ------------------------------------------------------------------------------------------------
# a mock kubelet: Registration server + DevicePlugin client (SURVEY.md 8(f) rank 1)
# ------------------------------------------------------------------------------------------------
@dataclass
class Registration:
    version: str
    endpoint: str
    resource_name: str
    options: object = None


class PluginClient:
    """What the kubelet's device manager does with a registered endpoint."""

    def __init__(self, socket_path: str):
        import grpc
        self.channel = grpc.insecure_channel("unix://" + socket_path)
        grpc.channel_ready_future(self.channel).result(timeout=CONNECTION_TIMEOUT)
        self._calls = {}
        for mname, (req, resp, stream) in dpapi.SERVICES["DevicePlugin"].items():
            make = self.channel.unary_stream if stream else self.channel.unary_unary
            self._calls[mname] = make(dpapi.method_path("DevicePlugin", mname),
                                      request_serializer=dpapi.MESSAGES[req].SerializeToString,
                                      response_deserializer=dpapi.MESSAGES[resp].FromString)

    def options(self):
        return self._calls["GetDevicePluginOptions"](dpapi.Empty(), timeout=CONNECTION_TIMEOUT)

    def list_and_watch(self):
        return self._calls["ListAndWatch"](dpapi.Empty())

    def allocate(self, *container_device_ids):
        req = dpapi.AllocateRequest(container_requests=[dpapi.ContainerAllocateRequest(devices_ids=list(ids))
                                                        for ids in container_device_ids])
        return self._calls["Allocate"](req, timeout=CONNECTION_TIMEOUT)

    def preferred_allocation(self, available, must_include, size):
        req = dpapi.PreferredAllocationRequest(container_requests=[dpapi.ContainerPreferredAllocationRequest(
            available_deviceIDs=list(available), must_include_deviceIDs=list(must_include), allocation_size=size)])
        return self._calls["GetPreferredAllocation"](req, timeout=CONNECTION_TIMEOUT)

    def close(self):
        self.channel.close()


@dataclass
class MockKubelet:
    """Serves v1beta1.Registration on <socket_dir>/kubelet.sock and remembers who registered."""
    socket_dir: str
    registrations: list = field(default_factory=list)

    def __post_init__(self):
        self.socket_path = os.path.join(self.socket_dir, "kubelet.sock")
        self._cv = threading.Condition()
        self.server = None

    def _register(self, request, context):
        with self._cv:
            self.registrations.append(Registration(request.version, request.endpoint, request.resource_name,
                                                   request.options))
            self._cv.notify_all()
        return dpapi.Empty()

    def start(self):
        import grpc
        try:
            os.remove(self.socket_path)
        except FileNotFoundError:
            pass
        self.server = grpc.server(futures.ThreadPoolExecutor(max_workers=4))
        handler = grpc.unary_unary_rpc_method_handler(
            self._register, request_deserializer=dpapi.RegisterRequest.FromString,
            response_serializer=dpapi.Empty.SerializeToString)
        self.server.add_generic_rpc_handlers((grpc.method_handlers_generic_handler(
            dpapi.service_name("Registration"), {"Register": handler}),))
        self.server.add_insecure_port("unix://" + self.socket_path)
        self.server.start()
        return self

    def wait_for(self, n: int, timeout: float = CONNECTION_TIMEOUT) -> list:
        with self._cv:
            self._cv.wait_for(lambda: len(self.registrations) >= n, timeout)
            return list(self.registrations)

    def connect(self, registration: Registration) -> PluginClient:
        return PluginClient(os.path.join(self.socket_dir, registration.endpoint))

    def stop(self):
        if self.server is not None:
            self.server.stop(0.2).wait(2.0)
            self.server = None
        try:
            os.remove(self.socket_path)
        except FileNotFoundError:
            pass


# ------------------------------------------------------------------------------------------------
# healthCheck(): the reference's own health source (generic_device_plugin.go:611-690) — inotify on the
# device nodes and on the plugin socket.  (HealthRescanFeed above is the GPU-side alternative.)
# ------------------------------------------------------------------------------------------------
class DeviceNodeWatcher:
    """Watches <device_path>/<iommu group> for every advertised device and the plugin's own socket:

      node created            -> healthy(id)   for every device of that group   (:659-662)
      node removed / renamed  -> unhealthy(id)                                   (:663-668)
      plugin socket removed   -> kubelet restarted: restart() = Stop + Start + Register (:669-679).  The
                                 reference's Start() spawns a fresh healthCheck goroutine and the old one
                                 returns; here the SAME watcher keeps running (its inotify watches are on the
                                 parent directories and survive), so every later restart is handled too.

    For a vGPU plugin the watched nodes are <vgpu_base_path>/<uuid> (generic_vgpu_device_plugin.go:319-351).

    fsnotify watches the PARENT directories; so does this (inotify through libc, no extra package)."""
    IN_CREATE, IN_DELETE, IN_MOVED_FROM, IN_DELETE_SELF, IN_MOVE_SELF = 0x100, 0x200, 0x40, 0x400, 0x800

    def __init__(self, plugin: GenericDevicePlugin, bdf_to_iommu=None):
        import ctypes
        self.plugin = plugin
        self._libc = ctypes.CDLL("libc.so.6", use_errno=True)
        self._fd = self._libc.inotify_init1(0o4000)          # IN_NONBLOCK
        if self._fd < 0:
            raise OSError(ctypes.get_errno(), "inotify_init1")
        self.path_devices = {}                               # node path -> [device ids]
        if getattr(plugin, "vgpu", False):
            for dev in plugin.devs:                          # one node per mediated device
                self.path_devices.setdefault(os.path.join(plugin.vgpu_base_path, dev.ID), []).append(dev.ID)
        else:
            bdf_to_iommu = bdf_to_iommu if bdf_to_iommu is not None else plugin.maps.bdfToIommuMap
            for dev in plugin.devs:
                group = bdf_to_iommu.get(dev.ID)
                if group is None:                            # :634-637 logged and skipped
                    continue
                self.path_devices.setdefault(os.path.join(plugin.device_path, group), []).append(dev.ID)
        self._wd_dir = {}
        dirs = {os.path.dirname(p) for p in self.path_devices} | {os.path.dirname(plugin.socket_path)}
        mask = self.IN_CREATE | self.IN_DELETE | self.IN_MOVED_FROM
        for d in sorted(dirs):
            wd = self._libc.inotify_add_watch(self._fd, d.encode(), mask)
            if wd < 0:
                err = ctypes.get_errno()
                os.close(self._fd)
                raise OSError(err, "inotify_add_watch(%s)" % d)
            self._wd_dir[wd] = d
        self._stop = threading.Event()
        self._thread = None
        self.restarted = threading.Event()
        self.restarts = 0

    def poll_once(self) -> int:
        """Drain pending inotify events; returns how many health / restart actions were taken."""
        import struct
        try:
            buf = os.read(self._fd, 65536)
        except BlockingIOError:
            return 0
        acted, off = 0, 0
        while off + 16 <= len(buf):
            wd, mask, _cookie, ln = struct.unpack_from("iIII", buf, off)
            name = buf[off + 16:off + 16 + ln].split(b"\0", 1)[0].decode()
            off += 16 + ln
            path = os.path.join(self._wd_dir.get(wd, ""), name)
            ids = self.path_devices.get(path)
            if ids is not None:
                if mask & self.IN_CREATE:
                    for i in ids:
                        self.plugin.healthy(i)
                    acted += len(ids)
                elif mask & (self.IN_DELETE | self.IN_MOVED_FROM):
                    for i in ids:
                        self.plugin.unhealthy(i)
                    acted += len(ids)
            elif path == self.plugin.socket_path and mask & self.IN_DELETE:
                self.plugin.restart()
                self.restarts += 1
                self.restarted.set()
                acted += 1
        return acted

    def start(self, period_s: float = 0.01):
        def loop():
            while not self._stop.is_set():
                self.poll_once()
                time.sleep(period_s)
        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(2.0)
        try:
            os.close(self._fd)
        except OSError:
            pass
