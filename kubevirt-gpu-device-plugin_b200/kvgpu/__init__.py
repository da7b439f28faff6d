"""kvgpu — B200-native discovery-and-classification scan for the KubeVirt GPU device plugin.

The compute lives in libkvgpu.so (hand-written sm_100a CUDA, C-ABI in include/kvgpu.h); this
package is the host-side mirror of the reference's plugin interface for that path.
"""
from ._lib import (KVG_NO_NAME, MDEV_REC, MDEV_SURV, PCI_REC, PCI_SURV, KvgError, declared_symbols,
                   load)
from .context import (Context, HealthDelta, KeyDelta, MdevRescan, MdevResult, MdevShardResult, PciRescan, PciResult,
                      PciShardResult)
from .plugin import (DiscoveryScan, Maps, MdevSnapshot, NvidiaGpuDevice, PciSnapshot, PluginEvent, PluginSpec,
                     ReferencePanic, canonical_dump, format_bdf, format_uuid,
                     mdev_maps_from_result, parse_bdf, pci_maps_from_result, plugin_specs_from_maps,
                     snapshot_mdev_tree,
                     snapshot_pci_tree)
from .parallel import (ShardedScan, allgatherv_torch, concat_in_rank_order, mdev_maps_from_shard, merge_parts,
                       pci_maps_from_shard, shard_range)

__all__ = [n for n in dir() if not n.startswith("_")]
