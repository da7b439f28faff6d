"""Context: thin object wrapper over the C-ABI (one CUDA stream, single-threaded)."""
from __future__ import annotations

import ctypes as C
import threading
from dataclasses import dataclass

import numpy as np

from . import _lib as L


@dataclass
class PciResult:
    """Flat output of kvg_scan_pci (see include/kvgpu.h kvg_pci_result)."""
    n_records: int
    survivors: np.ndarray       # PCI_SURV, Walk order
    dev_keys: np.ndarray        # u16 ascending
    dev_off: np.ndarray
    dev_perm: np.ndarray
    dev_name_slot: np.ndarray
    grp_keys: np.ndarray        # u32 ascending
    grp_off: np.ndarray
    grp_perm: np.ndarray
    name_pool: bytes

    def name_at(self, slot: int) -> str:
        if slot == L.KVG_NO_NAME:
            return ""
        n = self.name_pool[slot] | (self.name_pool[slot + 1] << 8)
        return self.name_pool[slot + 2:slot + 2 + n].decode("latin-1")


@dataclass
class MdevResult:
    n_records: int
    survivors: np.ndarray       # MDEV_SURV
    type_keys: np.ndarray
    type_off: np.ndarray
    type_perm: np.ndarray
    labels: list                # sanitised label per raw dictionary entry (bytes)
    type_canon: np.ndarray
    type_names: list            # getDeviceName(label) per raw entry (str, "" = miss)
    par_keys: np.ndarray
    par_off: np.ndarray
    par_perm: np.ndarray


@dataclass
class PciShardResult:
    """One rank's part of a sharded PCI scan (include/kvgpu.h kvg_pci_shard_result): its own shard's
    survivors, and ALL members of the device ids / iommu groups it owns (key % nranks == rank)."""
    n_records: int
    local: np.ndarray           # PCI_SURV, this shard's survivors, Walk order
    dev: PciResult              # deviceMap part: survivors = the owned members (grp_* arrays empty)
    grp: PciResult              # iommuMap part:  survivors = the owned members (dev_* arrays empty)


@dataclass
class MdevShardResult:
    n_records: int
    local: np.ndarray           # MDEV_SURV
    by_type: MdevResult         # vGpuMap part (par_* empty)
    by_parent: MdevResult       # gpuVgpuMap part (type_* empty)


@dataclass
class HealthDelta:
    n_records: int
    n_alive: int
    changed: np.ndarray         # (index << 1) | now_alive


@dataclass
class KeyDelta:
    """Key changes of one group-by map between two rescans (include/kvgpu.h kvg_key_delta); ascending."""
    added: np.ndarray           # u32 keys absent before, present now
    removed: np.ndarray         # u32 keys present before, absent now
    changed: np.ndarray         # u32 keys present in both whose member list differs


@dataclass
class PciRescan:
    """kvg_rescan_pci: the full scan plus its diff against the previous rescan."""
    scan: PciResult
    had_baseline: bool
    added: np.ndarray           # indices into scan.survivors
    removed: np.ndarray         # PCI_SURV, previous survivors
    moved: np.ndarray           # indices into scan.survivors
    dev: KeyDelta               # deviceMap
    grp: KeyDelta               # iommuMap


@dataclass
class MdevRescan:
    scan: MdevResult
    had_baseline: bool
    added: np.ndarray
    removed: np.ndarray         # MDEV_SURV
    moved: np.ndarray
    type: KeyDelta              # vGpuMap (canonical type ids)
    parent: KeyDelta            # gpuVgpuMap (parent handles)


def _key_delta(k) -> KeyDelta:
    return KeyDelta(L._arr(k.added, k.n_added, np.uint32), L._arr(k.removed, k.n_removed, np.uint32),
                    L._arr(k.changed, k.n_changed, np.uint32))


class _LockedLib:
    """A kvg_ctx is single-threaded (include/kvgpu.h).  gRPC handler threads, the health feed and the
    Allocate re-validation all share one Context (kvgpu/serve.py), so every C call on it is serialised."""

    def __init__(self, lib, lock):
        self._lib, self._lock = lib, lock

    def __getattr__(self, name):
        fn = getattr(self._lib, name)

        def call(*a):
            with self._lock:
                return fn(*a)
        return call


class Context:
    def __init__(self, device: int = 0):
        self._lock = threading.RLock()
        self._lib = _LockedLib(L.load(), self._lock)
        h = C.c_void_p()
        rc = self._lib.kvg_ctx_create(device, C.byref(h))
        if rc != 0:
            raise L.KvgError(rc, (self._lib.kvg_last_error(None) or b"").decode())
        self._h = h
        self.device = device

    # -- plumbing ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.kvg_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise L.KvgError(rc, (self._lib.kvg_last_error(self._h) or b"").decode())

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return int(self._lib.kvg_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._lib.kvg_launch_count(self._h))

    # -- pci.ids ----------------------------------------------------------------------------
    def pciids_load(self, text: bytes):
        buf = C.create_string_buffer(text, len(text)) if text else None
        self._ck(self._lib.kvg_pciids_load(self._h, C.cast(buf, C.c_void_p) if buf else None,
                                           len(text)))

    def name_lookup(self, key) -> str:
        """getDeviceName(key) — device_plugin.go:371-422."""
        if isinstance(key, str):
            key = key.encode("latin-1")
        cap = 1 << 17
        out = C.create_string_buffer(cap)
        n = C.c_size_t()
        self._ck(self._lib.kvg_name_lookup(self._h, key, len(key), out, cap, C.byref(n)))
        return out.raw[:n.value].decode("latin-1")

    def name_table(self, first: int = 0, count: int = 65536) -> list:
        off = np.zeros(count + 1, dtype=np.uint32)
        cap = 1 << 22
        out = np.zeros(cap, dtype=np.uint8)
        self._ck(self._lib.kvg_name_table(self._h, first, count, off.ctypes.data, out.ctypes.data,
                                          cap))
        raw = out.tobytes()
        return [raw[off[i]:off[i + 1]].decode("latin-1") for i in range(count)]

    def pciids_info(self) -> dict:
        v = [C.c_uint32() for _ in range(4)]
        self._ck(self._lib.kvg_pciids_info(self._h, *[C.byref(x) for x in v]))
        return dict(zip(("vendor_off", "section_end", "n_entries", "n_lines"),
                        [x.value for x in v]))

    # -- scans ------------------------------------------------------------------------------
    def _take_pci(self, res, free: bool = True) -> PciResult:
        r = res.contents
        S, KD, G = int(r.n_survivors), int(r.n_dev_keys), int(r.n_groups)
        dev_off = L._arr(r.dev_off, KD + 1, np.uint32)
        grp_off = L._arr(r.grp_off, G + 1, np.uint32)
        # a sharded scan orders only the keys this rank owns: perms are as long as off[-1]
        out = PciResult(
            n_records=int(r.n_records),
            survivors=L._arr(r.survivors, S, L.PCI_SURV),
            dev_keys=L._arr(r.dev_keys, KD, np.uint16),
            dev_off=dev_off,
            dev_perm=L._arr(r.dev_perm, int(dev_off[-1]), np.uint32),
            dev_name_slot=L._arr(r.dev_name_slot, KD, np.uint32),
            grp_keys=L._arr(r.grp_keys, G, np.uint32),
            grp_off=grp_off,
            grp_perm=L._arr(r.grp_perm, int(grp_off[-1]), np.uint32),
            name_pool=C.string_at(r.name_pool, r.name_pool_len) if r.name_pool_len else b"")
        if free:
            self._lib.kvg_result_free(res)
        return out

    def scan_pci(self, recs: np.ndarray) -> PciResult:
        """createIommuDeviceMap on a flat snapshot — device_plugin.go:187-247."""
        recs = np.ascontiguousarray(recs, dtype=L.PCI_REC)
        res = C.POINTER(L.PciResultC)()
        self._ck(self._lib.kvg_scan_pci(self._h, recs.ctypes.data, len(recs), C.byref(res)))
        return self._take_pci(res)

    @staticmethod
    def _type_dict(raw_types):
        off = np.zeros(len(raw_types) + 1, dtype=np.uint32)
        for i, t in enumerate(raw_types):
            off[i + 1] = off[i] + len(t)
        blob = np.frombuffer(b"".join(raw_types) + b"\0", dtype=np.uint8).copy()
        td = L.TypeDict(len(raw_types), off.ctypes.data_as(C.POINTER(C.c_uint32)),
                        blob.ctypes.data_as(C.POINTER(C.c_uint8)))
        return td, (off, blob)

    def _take_mdev(self, res, free: bool = True) -> MdevResult:
        r = res.contents
        S, KT, P, nt = int(r.n_survivors), int(r.n_type_keys), int(r.n_parents), int(r.n_types)
        loff = L._arr(r.label_off, nt + 1, np.uint32)
        noff = L._arr(r.type_name_off, nt + 1, np.uint32)
        lbytes = C.string_at(r.label_bytes, int(loff[-1])) if nt and loff[-1] else b""
        nbytes = C.string_at(r.type_name_bytes, int(noff[-1])) if nt and noff[-1] else b""
        out = MdevResult(
            n_records=int(r.n_records),
            survivors=L._arr(r.survivors, S, L.MDEV_SURV),
            type_keys=L._arr(r.type_keys, KT, np.uint16),
            type_off=L._arr(r.type_off, KT + 1, np.uint32),
            type_perm=L._arr(r.type_perm, S, np.uint32),
            labels=[lbytes[loff[i]:loff[i + 1]] for i in range(nt)],
            type_canon=L._arr(r.type_canon, nt, np.uint16),
            type_names=[nbytes[noff[i]:noff[i + 1]].decode("latin-1") for i in range(nt)],
            par_keys=L._arr(r.par_keys, P, np.uint32),
            par_off=L._arr(r.par_off, P + 1, np.uint32),
            par_perm=L._arr(r.par_perm, S, np.uint32))
        if free:
            self._lib.kvg_result_free(res)
        return out

    def scan_mdev(self, recs: np.ndarray, raw_types: list) -> MdevResult:
        """createVgpuIDMap on a flat snapshot — device_plugin.go:255-291."""
        recs = np.ascontiguousarray(recs, dtype=L.MDEV_REC)
        td, keep = self._type_dict(raw_types)
        res = C.POINTER(L.MdevResultC)()
        self._ck(self._lib.kvg_scan_mdev(self._h, recs.ctypes.data, len(recs), C.byref(td),
                                         C.byref(res)))
        del keep
        return self._take_mdev(res)

    def health_rescan(self, recs: np.ndarray) -> HealthDelta:
        recs = np.ascontiguousarray(recs, dtype=L.PCI_REC)
        res = C.POINTER(L.HealthDeltaC)()
        self._ck(self._lib.kvg_health_rescan(self._h, recs.ctypes.data, len(recs), C.byref(res)))
        r = res.contents
        out = HealthDelta(int(r.n_records), int(r.n_alive),
                          L._arr(r.changed, int(r.n_changed), np.uint32))
        self._lib.kvg_result_free(res)
        return out

    def health_reset(self):
        self._ck(self._lib.kvg_health_reset(self._h))

    def rescan_pci(self, recs: np.ndarray) -> PciRescan:
        """A full scan of `recs` (numeric mode, Walk order) diffed against the previous rescan."""
        recs = np.ascontiguousarray(recs, dtype=L.PCI_REC)
        res = C.POINTER(L.PciRescanC)()
        self._ck(self._lib.kvg_rescan_pci(self._h, recs.ctypes.data, len(recs), C.byref(res)))
        r = res.contents
        out = PciRescan(self._take_pci(C.pointer(r.scan), free=False), bool(r.had_baseline),
                        L._arr(r.added, r.n_added, np.uint32), L._arr(r.removed, r.n_removed, L.PCI_SURV),
                        L._arr(r.moved, r.n_moved, np.uint32), _key_delta(r.dev), _key_delta(r.grp))
        self._lib.kvg_result_free(res)
        return out

    def rescan_mdev(self, recs: np.ndarray, raw_types: list) -> MdevRescan:
        """The same for mdevs; `raw_types` must extend the previous rescan's dictionary (append only)."""
        recs = np.ascontiguousarray(recs, dtype=L.MDEV_REC)
        td, keep = self._type_dict(raw_types)
        res = C.POINTER(L.MdevRescanC)()
        self._ck(self._lib.kvg_rescan_mdev(self._h, recs.ctypes.data, len(recs), C.byref(td), C.byref(res)))
        del keep
        r = res.contents
        out = MdevRescan(self._take_mdev(C.pointer(r.scan), free=False), bool(r.had_baseline),
                         L._arr(r.added, r.n_added, np.uint32), L._arr(r.removed, r.n_removed, L.MDEV_SURV),
                         L._arr(r.moved, r.n_moved, np.uint32), _key_delta(r.type), _key_delta(r.parent))
        self._lib.kvg_result_free(res)
        return out

    def rescan_reset(self):
        self._ck(self._lib.kvg_rescan_reset(self._h))

    # -- device-resident entry points (raw device pointers, e.g. torch tensor.data_ptr()) ----
    def text_pad(self, n: int) -> int:
        return int(self._lib.kvg_text_pad(n))

    def dev_pciids_parse(self, d_text: int, length: int, stride: int, n_files: int = 1):
        self._ck(self._lib.kvg_dev_pciids_parse(self._h, d_text, length, stride, n_files))

    def dev_scan_pci(self, d_recs: int, n: int):
        self._ck(self._lib.kvg_dev_scan_pci(self._h, d_recs, n))

    def dev_scan_pci_fetch(self) -> PciResult:
        res = C.POINTER(L.PciResultC)()
        self._ck(self._lib.kvg_dev_scan_pci_fetch(self._h, C.byref(res)))
        return self._take_pci(res)

    def dev_scan_pci_count(self):
        s, k, g = C.c_uint64(), C.c_uint32(), C.c_uint32()
        self._ck(self._lib.kvg_dev_scan_pci_count(self._h, C.byref(s), C.byref(k), C.byref(g)))
        return s.value, k.value, g.value

    def dev_gen_pci(self, d_recs: int, first: int, n: int, nv_ids: np.ndarray, group_bits: int = 0):
        ids = np.ascontiguousarray(nv_ids, dtype=np.uint16)
        self._ck(self._lib.kvg_dev_gen_pci(self._h, d_recs, first, n, ids.ctypes.data, len(ids),
                                           group_bits))

    def dev_gen_mdev(self, d_recs: int, first: int, n: int):
        self._ck(self._lib.kvg_dev_gen_mdev(self._h, d_recs, first, n))

    def dev_scan_mdev(self, d_recs: int, n: int, raw_types: list):
        td, keep = self._type_dict(raw_types)
        self._ck(self._lib.kvg_dev_scan_mdev(self._h, d_recs, n, C.byref(td)))
        del keep

    def dev_scan_mdev_fetch(self) -> MdevResult:
        res = C.POINTER(L.MdevResultC)()
        self._ck(self._lib.kvg_dev_scan_mdev_fetch(self._h, C.byref(res)))
        return self._take_mdev(res)

    def dev_flush_l2(self):
        self._ck(self._lib.kvg_dev_flush_l2(self._h))

    def set_kernel_timing(self, on: bool):
        self._ck(self._lib.kvg_set_kernel_timing(self._h, 1 if on else 0))

    def kernel_times(self, max_n: int = 4096):
        ms = (C.c_float * max_n)()
        names = C.create_string_buffer(64 * max_n)
        n = self._lib.kvg_kernel_times(self._h, ms, names, len(names), max_n)
        if n < 0:
            self._ck(n)
        parts = names.raw.split(b"\0")
        return [(parts[i].decode(), float(ms[i])) for i in range(n)]

    # -- multi-GPU --------------------------------------------------------------------------
    def comm_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        rc = self._lib.kvg_comm_unique_id(buf)
        if rc != 0:
            raise L.KvgError(rc, (self._lib.kvg_last_error(None) or b"").decode())
        return buf.raw

    def comm_init(self, rank: int, nranks: int, uid: bytes):
        buf = C.create_string_buffer(uid, 128)
        self._ck(self._lib.kvg_comm_init(self._h, rank, nranks, buf))

    def comm_p2p_export(self, rank: int, nranks: int, cap_local: int) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self._lib.kvg_comm_p2p_export(self._h, rank, nranks, cap_local, buf))
        return buf.raw

    def comm_p2p_import(self, all_handles: bytes):
        buf = C.create_string_buffer(all_handles, len(all_handles))
        self._ck(self._lib.kvg_comm_p2p_import(self._h, buf))

    def comm_p2p_enable(self, on: bool):
        self._ck(self._lib.kvg_comm_p2p_enable(self._h, 1 if on else 0))

    def comm_destroy(self):
        self._ck(self._lib.kvg_comm_destroy(self._h))

    def dev_scan_pci_sharded(self, d_recs: int, n_local: int):
        self._ck(self._lib.kvg_dev_scan_pci_sharded(self._h, d_recs, n_local))

    def dev_scan_pci_shard_fetch(self) -> PciShardResult:
        res = C.POINTER(L.PciShardResultC)()
        self._ck(self._lib.kvg_dev_scan_pci_shard_fetch(self._h, C.byref(res)))
        r = res.contents
        KD, G = int(r.n_dev_keys), int(r.n_groups)
        pool = C.string_at(r.name_pool, r.name_pool_len) if r.name_pool_len else b""
        e32, e16 = np.zeros(0, np.uint32), np.zeros(0, np.uint16)
        z32 = np.zeros(1, np.uint32)
        dev = PciResult(int(r.n_records), L._arr(r.dev_members, int(r.n_dev_members), L.PCI_SURV),
                        L._arr(r.dev_keys, KD, np.uint16), L._arr(r.dev_off, KD + 1, np.uint32),
                        L._arr(r.dev_perm, int(r.n_dev_members), np.uint32), L._arr(r.dev_name_slot, KD, np.uint32),
                        e32, z32, e32, pool)
        grp = PciResult(int(r.n_records), L._arr(r.grp_members, int(r.n_grp_members), L.PCI_SURV),
                        e16, z32, e32, e32, L._arr(r.grp_keys, G, np.uint32), L._arr(r.grp_off, G + 1, np.uint32),
                        L._arr(r.grp_perm, int(r.n_grp_members), np.uint32), pool)
        out = PciShardResult(int(r.n_records), L._arr(r.local, int(r.n_local), L.PCI_SURV), dev, grp)
        self._lib.kvg_result_free(res)
        return out

    def dev_scan_mdev_sharded(self, d_recs: int, n_local: int, raw_types: list):
        td, keep = self._type_dict(raw_types)
        self._ck(self._lib.kvg_dev_scan_mdev_sharded(self._h, d_recs, n_local, C.byref(td)))
        del keep

    def dev_scan_mdev_shard_fetch(self) -> MdevShardResult:
        res = C.POINTER(L.MdevShardResultC)()
        self._ck(self._lib.kvg_dev_scan_mdev_shard_fetch(self._h, C.byref(res)))
        r = res.contents
        KT, NP, nt = int(r.n_type_keys), int(r.n_parents), int(r.n_types)
        loff = L._arr(r.label_off, nt + 1, np.uint32)
        noff = L._arr(r.type_name_off, nt + 1, np.uint32)
        lbytes = C.string_at(r.label_bytes, int(loff[-1])) if nt and loff[-1] else b""
        nbytes = C.string_at(r.type_name_bytes, int(noff[-1])) if nt and noff[-1] else b""
        labels = [lbytes[loff[i]:loff[i + 1]] for i in range(nt)]
        names = [nbytes[noff[i]:noff[i + 1]].decode("latin-1") for i in range(nt)]
        canon = L._arr(r.type_canon, nt, np.uint16)
        e32, e16, z32 = np.zeros(0, np.uint32), np.zeros(0, np.uint16), np.zeros(1, np.uint32)
        by_type = MdevResult(int(r.n_records), L._arr(r.type_members, int(r.n_type_members), L.MDEV_SURV),
                             L._arr(r.type_keys, KT, np.uint16), L._arr(r.type_off, KT + 1, np.uint32),
                             L._arr(r.type_perm, int(r.n_type_members), np.uint32), labels, canon, names, e32, z32, e32)
        by_parent = MdevResult(int(r.n_records), L._arr(r.par_members, int(r.n_par_members), L.MDEV_SURV),
                               e16, z32, e32, labels, canon, names, L._arr(r.par_keys, NP, np.uint32),
                               L._arr(r.par_off, NP + 1, np.uint32), L._arr(r.par_perm, int(r.n_par_members), np.uint32))
        out = MdevShardResult(int(r.n_records), L._arr(r.local, int(r.n_local), L.MDEV_SURV), by_type, by_parent)
        self._lib.kvg_result_free(res)
        return out
