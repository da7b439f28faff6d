// kvg_api.cu — the C-ABI of libkvgpu.so (include/kvgpu.h): context, HBM layout, launch sequencing
// and result marshalling around the kernels in kvg_parse.cuh / kvg_scan.cuh.
//
// HBM layout owned by a context (all cudaMalloc'd once and grown geometrically, never per call):
//   text      pci.ids image(s), padded with '\n' to a tile multiple + 16 (TMA halo)
//   dev_off   per image 65,536 x u32: line offset of the first "\t<id>" line under a 10de header
//   nv_index  65,536 x u32: device id -> name pool slot (what the scans join against)
//   pool      sanitised names of the NVIDIA section, slot = line offset - section offset
//   recs      record staging (host entry points only)
//   surv      compacted survivors, Walk order
//   sort      2 x (keys,vals) ping-pong per ordering (device-id ordering, iommu-group ordering)
//   seg       distinct keys + offsets per ordering
// No CPU fallback exists anywhere below: every compute entry point fails with KVG_ECUDA when the
// CUDA runtime is unusable.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <string>
#include <vector>

#include "../../include/kvgpu.h"
#include "kvg_common.cuh"
#include "kvg_parse.cuh"
#include "kvg_parse_k1.cuh"
#include "kvg_scan.cuh"
#include "kvg_order.cuh"
#include "kvg_shard.cuh"
#include "kvg_rescan.cuh"

using namespace kvg;

#include "api/kvg_api_ctx.inc"
#include "api/kvg_api_core.inc"
#include "api/kvg_api_pciids.inc"
#include "api/kvg_api_scan.inc"
#include "api/kvg_api_health.inc"
#include "api/kvg_api_mdev.inc"
#include "api/kvg_api_util.inc"
#include "api/kvg_api_shard.inc"
#include "api/kvg_api_rescan.inc"
