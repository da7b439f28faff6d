"""ctypes binding of libkvgpu.so — exactly the symbols include/kvgpu.h declares.

There is no CPU fallback: if the library is missing or no CUDA device is usable, every compute
entry point raises KvgError.
"""
from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np

_PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG, "libkvgpu.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "kvgpu.h")

KVG_OK, KVG_EINVAL, KVG_ECUDA, KVG_ENOMEM, KVG_ENCCL, KVG_ESTATE, KVG_ERANGE = 0, -1, -2, -3, -4, -5, -6
KVG_NO_NAME = 0xFFFFFFFF
ERR_NAMES = {0: "KVG_OK", -1: "KVG_EINVAL", -2: "KVG_ECUDA", -3: "KVG_ENOMEM", -4: "KVG_ENCCL",
             -5: "KVG_ESTATE", -6: "KVG_ERANGE"}

DRV_NONE, DRV_VFIO_PCI, DRV_NVGRACE, DRV_OTHER = 0, 1, 2, 3
PF_VENDOR_ERR, PF_DRIVER_ERR, PF_IOMMU_ERR, PF_DEVICE_ERR, PF_NUMA_ERR = 1, 2, 4, 8, 16
MF_TYPE_ERR, MF_PARENT_ERR, MF_NUMA_ERR = 1, 2, 4

PCI_REC = np.dtype([("addr", "<u4"), ("vendor", "<u2"), ("device", "<u2"), ("iommu_group", "<u4"),
                    ("driver", "u1"), ("flags", "u1"), ("numa", "<i2")])
PCI_SURV = np.dtype([("addr", "<u4"), ("iommu_group", "<u4"), ("device", "<u2"), ("numa", "<u2"),
                     ("name_slot", "<u4")])
MDEV_REC = np.dtype([("uuid", "u1", (16,)), ("parent", "<u4"), ("type_idx", "<u2"), ("flags", "u1"),
                     ("pad0", "u1"), ("parent_numa", "<i2"), ("pad1", "u1", (6,))])
MDEV_SURV = np.dtype([("uuid", "u1", (16,)), ("parent", "<u4"), ("type_key", "<u2"),
                      ("numa", "<u2"), ("src", "<u4"), ("pad", "<u4")])
assert PCI_REC.itemsize == 16 and PCI_SURV.itemsize == 16
assert MDEV_REC.itemsize == 32 and MDEV_SURV.itemsize == 32


class KvgError(RuntimeError):
    def __init__(self, rc, msg):
        super().__init__("%s: %s" % (ERR_NAMES.get(rc, rc), msg))
        self.rc = rc


class TypeDict(C.Structure):
    _fields_ = [("n_types", C.c_uint32), ("off", C.POINTER(C.c_uint32)),
                ("bytes", C.POINTER(C.c_uint8))]


class PciResultC(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_survivors", C.c_uint64),
                ("survivors", C.c_void_p),
                ("n_dev_keys", C.c_uint32), ("dev_keys", C.c_void_p), ("dev_off", C.c_void_p),
                ("dev_perm", C.c_void_p), ("dev_name_slot", C.c_void_p),
                ("n_groups", C.c_uint32), ("grp_keys", C.c_void_p), ("grp_off", C.c_void_p),
                ("grp_perm", C.c_void_p),
                ("name_pool", C.c_void_p), ("name_pool_len", C.c_size_t)]


class MdevResultC(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_survivors", C.c_uint64),
                ("survivors", C.c_void_p),
                ("n_type_keys", C.c_uint32), ("type_keys", C.c_void_p), ("type_off", C.c_void_p),
                ("type_perm", C.c_void_p),
                ("n_types", C.c_uint32), ("label_off", C.c_void_p), ("label_bytes", C.c_void_p),
                ("type_canon", C.c_void_p), ("type_name_off", C.c_void_p),
                ("type_name_bytes", C.c_void_p),
                ("n_parents", C.c_uint32), ("par_keys", C.c_void_p), ("par_off", C.c_void_p),
                ("par_perm", C.c_void_p)]


class PciShardResultC(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_local", C.c_uint64), ("local", C.c_void_p),
                ("n_dev_members", C.c_uint64), ("dev_members", C.c_void_p),
                ("n_dev_keys", C.c_uint32), ("dev_keys", C.c_void_p), ("dev_off", C.c_void_p),
                ("dev_perm", C.c_void_p), ("dev_name_slot", C.c_void_p),
                ("n_grp_members", C.c_uint64), ("grp_members", C.c_void_p),
                ("n_groups", C.c_uint32), ("grp_keys", C.c_void_p), ("grp_off", C.c_void_p),
                ("grp_perm", C.c_void_p),
                ("name_pool", C.c_void_p), ("name_pool_len", C.c_size_t)]


class MdevShardResultC(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_local", C.c_uint64), ("local", C.c_void_p),
                ("n_type_members", C.c_uint64), ("type_members", C.c_void_p),
                ("n_type_keys", C.c_uint32), ("type_keys", C.c_void_p), ("type_off", C.c_void_p),
                ("type_perm", C.c_void_p),
                ("n_par_members", C.c_uint64), ("par_members", C.c_void_p),
                ("n_parents", C.c_uint32), ("par_keys", C.c_void_p), ("par_off", C.c_void_p),
                ("par_perm", C.c_void_p),
                ("n_types", C.c_uint32), ("label_off", C.c_void_p), ("label_bytes", C.c_void_p),
                ("type_canon", C.c_void_p), ("type_name_off", C.c_void_p),
                ("type_name_bytes", C.c_void_p)]


class HealthDeltaC(C.Structure):
    _fields_ = [("n_records", C.c_uint32), ("n_alive", C.c_uint32), ("n_changed", C.c_uint32),
                ("changed", C.c_void_p)]


class KeyDeltaC(C.Structure):
    _fields_ = [("n_added", C.c_uint32), ("added", C.c_void_p), ("n_removed", C.c_uint32),
                ("removed", C.c_void_p), ("n_changed", C.c_uint32), ("changed", C.c_void_p)]


class PciRescanC(C.Structure):
    _fields_ = [("scan", PciResultC), ("had_baseline", C.c_uint32),
                ("n_added", C.c_uint64), ("added", C.c_void_p), ("n_removed", C.c_uint64),
                ("removed", C.c_void_p), ("n_moved", C.c_uint64), ("moved", C.c_void_p),
                ("dev", KeyDeltaC), ("grp", KeyDeltaC)]


class MdevRescanC(C.Structure):
    _fields_ = [("scan", MdevResultC), ("had_baseline", C.c_uint32),
                ("n_added", C.c_uint64), ("added", C.c_void_p), ("n_removed", C.c_uint64),
                ("removed", C.c_void_p), ("n_moved", C.c_uint64), ("moved", C.c_void_p),
                ("type", KeyDeltaC), ("parent", KeyDeltaC)]


def declared_symbols() -> list[str]:
    """Every function name include/kvgpu.h declares (used by the export test)."""
    src = open(HEADER_PATH).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(kvg_[a-z0-9_]+)\s*\(", src)))


_lib = None


def load() -> C.CDLL:
    """dlopen libkvgpu.so (built in-tree by __graft_entry__.build / csrc/Makefile)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise KvgError(KVG_ECUDA, "libkvgpu.so is not built (%s); run `python -c 'import "
                       "__graft_entry__ as g; g.build()'` — there is no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, sz, u32, u64 = C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64
    P = C.POINTER
    sig = {
        "kvg_abi_version": (C.c_int, []),
        "kvg_ctx_create": (C.c_int, [C.c_int, P(vp)]),
        "kvg_ctx_destroy": (None, [vp]),
        "kvg_last_error": (C.c_char_p, [vp]),
        "kvg_result_free": (None, [vp]),
        "kvg_launch_count": (u64, [vp]),
        "kvg_stream": (vp, [vp]),
        "kvg_pciids_load": (C.c_int, [vp, vp, sz]),
        "kvg_name_lookup": (C.c_int, [vp, C.c_char_p, sz, C.c_char_p, sz, P(sz)]),
        "kvg_name_table": (C.c_int, [vp, u32, u32, vp, vp, sz]),
        "kvg_pciids_info": (C.c_int, [vp, P(u32), P(u32), P(u32), P(u32)]),
        "kvg_scan_pci": (C.c_int, [vp, vp, sz, P(P(PciResultC))]),
        "kvg_scan_mdev": (C.c_int, [vp, vp, sz, P(TypeDict), P(P(MdevResultC))]),
        "kvg_health_rescan": (C.c_int, [vp, vp, sz, P(P(HealthDeltaC))]),
        "kvg_health_reset": (C.c_int, [vp]),
        "kvg_rescan_pci": (C.c_int, [vp, vp, sz, P(P(PciRescanC))]),
        "kvg_rescan_mdev": (C.c_int, [vp, vp, sz, P(TypeDict), P(P(MdevRescanC))]),
        "kvg_rescan_reset": (C.c_int, [vp]),
        "kvg_text_pad": (sz, [sz]),
        "kvg_dev_pciids_parse": (C.c_int, [vp, vp, sz, sz, u32]),
        "kvg_dev_scan_pci": (C.c_int, [vp, vp, sz]),
        "kvg_dev_scan_pci_fetch": (C.c_int, [vp, P(P(PciResultC))]),
        "kvg_dev_scan_pci_count": (C.c_int, [vp, P(u64), P(u32), P(u32)]),
        "kvg_dev_gen_pci": (C.c_int, [vp, vp, u64, sz, vp, u32, u32]),
        "kvg_dev_gen_mdev": (C.c_int, [vp, vp, u64, sz]),
        "kvg_dev_scan_mdev": (C.c_int, [vp, vp, sz, P(TypeDict)]),
        "kvg_dev_scan_mdev_fetch": (C.c_int, [vp, P(P(MdevResultC))]),
        "kvg_dev_flush_l2": (C.c_int, [vp]),
        "kvg_kernel_times": (C.c_int, [vp, P(C.c_float), C.c_char_p, sz, C.c_int]),
        "kvg_set_kernel_timing": (C.c_int, [vp, C.c_int]),
        "kvg_comm_unique_id": (C.c_int, [vp]),
        "kvg_comm_init": (C.c_int, [vp, C.c_int, C.c_int, vp]),
        "kvg_comm_destroy": (C.c_int, [vp]),
        "kvg_comm_p2p_export": (C.c_int, [vp, C.c_int, C.c_int, sz, vp]),
        "kvg_comm_p2p_import": (C.c_int, [vp, vp]),
        "kvg_comm_p2p_enable": (C.c_int, [vp, C.c_int]),
        "kvg_debug_radix_plan": (C.c_int, [C.c_uint32, C.c_uint32, C.c_uint32, vp, vp, vp]),
        "kvg_dev_scan_pci_sharded": (C.c_int, [vp, vp, sz]),
        "kvg_dev_scan_pci_shard_fetch": (C.c_int, [vp, P(P(PciShardResultC))]),
        "kvg_dev_scan_mdev_sharded": (C.c_int, [vp, vp, sz, P(TypeDict)]),
        "kvg_dev_scan_mdev_shard_fetch": (C.c_int, [vp, P(P(MdevShardResultC))]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def _arr(ptr, n, dtype):
    """copy n items of dtype out of a library-owned buffer"""
    if not n:
        return np.zeros(0, dtype=dtype)
    nbytes = int(n) * np.dtype(dtype).itemsize
    return np.frombuffer(C.string_at(ptr, nbytes), dtype=dtype).copy()
