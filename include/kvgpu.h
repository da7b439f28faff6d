/*
 * kvgpu.h — C-ABI of libkvgpu.so: the B200 (sm_100a) discovery-and-classification scan
 * that replaces the CPU scan of NVIDIA/kubevirt-gpu-device-plugin.
 *
 * The reference has NO FFI on this path today (it is pure Go).  The seam a maintainer binds is
 * the reference's own injection points; each entry point below cites the reference function it
 * replaces (paths relative to the reference repo root):
 *
 *   kvg_pciids_load   + kvg_name_lookup   <- getDeviceName / locateVendor
 *                                            pkg/device_plugin/device_plugin.go:371-438
 *   kvg_scan_pci                          <- createIommuDeviceMap   device_plugin.go:187-247
 *                                            (+ isSupportedVfioDriver :249-252, name join :124-128)
 *   kvg_scan_mdev                         <- createVgpuIDMap        device_plugin.go:255-291
 *                                            (+ readVgpuIDFromFileFunc label rule :334-344, join :152-155)
 *   kvg_health_rescan                     <- health flips fed to ListAndWatch
 *                                            generic_device_plugin.go:325-342, :611-690
 *   kvg_rescan_pci, kvg_rescan_mdev       <- (no reference equivalent: the reference scans once at start-up,
 *                                            device_plugin.go:89-96)
 *   kvg_comm_*, kvg_scan_pci_sharded      <- (no reference equivalent; BASELINE.json config 4)
 *
 * Plain C: pointers + sizes only, no C++ types, no exceptions cross this boundary.
 * Return value: 0 = KVG_OK, negative = error; text via kvg_last_error().
 * There is NO CPU fallback: without a usable CUDA device every compute call returns KVG_ECUDA.
 *
 * Threading: a kvg_ctx owns one CUDA stream and is single-threaded (caller serialises);
 * distinct contexts are independent.  The library never calls back into the caller and never
 * retains caller pointers after a call returns (cgo pointer rule): host inputs are copied into
 * pinned staging memory inside the call.  Result objects are library-owned, flat, pointer+length
 * arrays in host memory, valid until kvg_result_free().
 */
#ifndef KVGPU_H
#define KVGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KVG_ABI_VERSION 1

/* ---- error codes --------------------------------------------------------------------------- */
enum {
  KVG_OK = 0,
  KVG_EINVAL = -1, /* bad argument */
  KVG_ECUDA = -2,  /* CUDA runtime / no device / kernel failure */
  KVG_ENOMEM = -3, /* host or device allocation failed */
  KVG_ENCCL = -4,  /* NCCL not loadable or a collective failed */
  KVG_ESTATE = -5, /* call order (e.g. scan before kvg_pciids_load) */
  KVG_ERANGE = -6  /* output buffer too small / value does not fit the wire format */
};

/* ---- wire format ---------------------------------------------------------------------------- */

/* driver dictionary codes produced by the snapshotter (device_plugin.go:75-78, :212-220) */
enum {
  KVG_DRV_NONE = 0,   /* no driver link (readLink error; also sets KVG_PF_DRIVER_ERR) */
  KVG_DRV_VFIO_PCI = 1, /* "vfio-pci" */
  KVG_DRV_NVGRACE = 2,  /* "nvgrace_gpu_vfio_pci" */
  KVG_DRV_OTHER = 3     /* anything else; codes >= 3 are all "unsupported" */
};

/* kvg_pci_rec.flags: which sysfs read FAILED for this entry (device_plugin.go:202-238) */
enum {
  KVG_PF_VENDOR_ERR = 1u << 0, /* readIDFromFile(vendor) error   -> drop (:203-206) */
  KVG_PF_DRIVER_ERR = 1u << 1, /* readLink(driver) error         -> drop (:213-216) */
  KVG_PF_IOMMU_ERR = 1u << 2,  /* readLink(iommu_group) error    -> drop (:222-225) */
  KVG_PF_DEVICE_ERR = 1u << 3, /* readIDFromFile(device) error   -> drop (:235-238) */
  KVG_PF_NUMA_ERR = 1u << 4    /* readNUMANode error             -> numa 0, KEPT (:227-230) */
};

/* One PCI function as snapshotted from /sys/bus/pci/devices/<addr>/, 16 bytes = one uint4.
 * Records are stored in filepath.Walk order (ascending byte-wise entry name). */
typedef struct kvg_pci_rec {
  uint32_t addr;        /* address handle: packed BDF domain<<16|bus<<8|dev<<3|fn, or the Walk
                           index when the snapshot is in index mode (names kept by the host) */
  uint16_t vendor;      /* sysfs "vendor" as a number (0x10de = NVIDIA); strings that are not
                           "0x%04x" can never equal "10de" and are stored as 0xffff            */
  uint16_t device;      /* sysfs "device" as a number -> key "%04x"                            */
  uint32_t iommu_group; /* basename of the iommu_group link as a number (or interned id)       */
  uint8_t driver;       /* KVG_DRV_*                                                            */
  uint8_t flags;        /* KVG_PF_*                                                             */
  int16_t numa;         /* raw numa_node value (may be -1); ignored when KVG_PF_NUMA_ERR        */
} kvg_pci_rec;

/* One surviving (advertised) PCI function, 16 bytes.  Order = Walk order (stable compaction). */
typedef struct kvg_pci_surv {
  uint32_t addr;
  uint32_t iommu_group;
  uint16_t device;
  uint16_t numa;      /* clamped: negative or unreadable -> 0 (device_plugin.go:316-318, :227-230) */
  uint32_t name_slot; /* offset into the context's name pool, or KVG_NO_NAME (getDeviceName == "") */
} kvg_pci_surv;

#define KVG_NO_NAME 0xffffffffu

/* kvg_mdev_rec.flags (device_plugin.go:269-284) */
enum {
  KVG_MF_TYPE_ERR = 1u << 0,   /* readVgpuIDFromFile error -> drop (:270-273) */
  KVG_MF_PARENT_ERR = 1u << 1, /* readGpuIDForVgpu error   -> drop (:276-279) */
  KVG_MF_NUMA_ERR = 1u << 2    /* parent numa unreadable   -> 0, KEPT (:281-284) */
};

/* One mediated device from /sys/bus/mdev/devices/<uuid>, 32 bytes, Walk order. */
typedef struct kvg_mdev_rec {
  uint8_t uuid[16];    /* big-endian UUID bytes (index mode: bytes 0..3 = BE Walk index) */
  uint32_t parent;     /* parent GPU address handle (packed BDF or interned id)          */
  uint16_t type_idx;   /* index into the raw type-name dictionary                        */
  uint8_t flags;       /* KVG_MF_*                                                        */
  uint8_t pad0;
  int16_t parent_numa; /* raw numa_node of the parent (may be -1)                        */
  uint8_t pad1[6];
} kvg_mdev_rec;

/* One surviving mdev, 32 bytes, Walk order. */
typedef struct kvg_mdev_surv {
  uint8_t uuid[16];
  uint32_t parent;
  uint16_t type_key; /* canonical type id = smallest raw index with the same sanitised label */
  uint16_t numa;
  uint32_t src;      /* index of the source record */
  uint32_t pad;
} kvg_mdev_surv;

/* Raw mdev_type/name file contents, unsanitised (the GPU applies device_plugin.go:341-342). */
typedef struct kvg_type_dict {
  uint32_t n_types;
  const uint32_t *off; /* n_types+1 offsets into bytes */
  const uint8_t *bytes;
} kvg_type_dict;

/* ---- results (library-owned host memory; free with kvg_result_free) ----------------------- */

typedef struct kvg_pci_result {
  uint64_t n_records;
  uint64_t n_survivors;
  const kvg_pci_surv *survivors; /* [n_survivors] Walk order == bdfToIommuMap insertion order */
  /* deviceMap (device_plugin.go:240): keys ascending; members of key k are
     survivors[dev_perm[dev_off[k] .. dev_off[k+1])], in Walk order */
  uint32_t n_dev_keys;
  const uint16_t *dev_keys;
  const uint32_t *dev_off;  /* [n_dev_keys+1] */
  const uint32_t *dev_perm; /* [n_survivors] */
  const uint32_t *dev_name_slot; /* [n_dev_keys] name pool offset or KVG_NO_NAME */
  /* iommuMap (device_plugin.go:241-242): same encoding, keys ascending numerically */
  uint32_t n_groups;
  const uint32_t *grp_keys;
  const uint32_t *grp_off;  /* [n_groups+1] */
  const uint32_t *grp_perm; /* [n_survivors] */
  /* sanitised names produced by the GPU; entry at slot s: uint16 length, then the bytes */
  const uint8_t *name_pool;
  size_t name_pool_len;
} kvg_pci_result;

typedef struct kvg_mdev_result {
  uint64_t n_records;
  uint64_t n_survivors;
  const kvg_mdev_surv *survivors;
  /* vGpuMap (device_plugin.go:288): keyed by canonical type id */
  uint32_t n_type_keys;
  const uint16_t *type_keys;
  const uint32_t *type_off;
  const uint32_t *type_perm;
  /* sanitised label of every raw dictionary entry (GPU output), and the resource-name join
     (getDeviceName(label), device_plugin.go:152): slot or KVG_NO_NAME */
  uint32_t n_types;
  const uint32_t *label_off; /* [n_types+1] into label_bytes */
  const uint8_t *label_bytes;
  const uint16_t *type_canon; /* [n_types] canonical id of each raw entry */
  const uint32_t *type_name_off; /* [n_types+1] into type_name_bytes: sanitised pci.ids name or empty */
  const uint8_t *type_name_bytes;
  /* gpuVgpuMap (device_plugin.go:287): keyed by parent handle ascending */
  uint32_t n_parents;
  const uint32_t *par_keys;
  const uint32_t *par_off;
  const uint32_t *par_perm;
} kvg_mdev_result;

/* ---- results of the SHARDED scans (one process per GPU; BASELINE.json config 4) ---------------------
 * Rank r scans records [r*N/P, (r+1)*N/P).  Its survivors stay local (concatenating the ranks' `local`
 * lists in rank order is the global Walk-order list, i.e. bdfToIommuMap / the mdev list).  The two group-by
 * maps are partitioned BY KEY: rank r holds exactly the keys with key % nranks == r, with ALL their members
 * (from every shard, Walk order).  Key sets of different ranks are disjoint; their union is the global map. */
typedef struct kvg_pci_shard_result {
  uint64_t n_records;             /* records of this rank's shard */
  uint64_t n_local;
  const kvg_pci_surv *local;      /* [n_local] this shard's survivors, Walk order */
  /* deviceMap part: members of the device ids this rank owns; key k = dev_members[dev_perm[dev_off[k]..)] */
  uint64_t n_dev_members;
  const kvg_pci_surv *dev_members;
  uint32_t n_dev_keys;
  const uint16_t *dev_keys;
  const uint32_t *dev_off;
  const uint32_t *dev_perm;
  const uint32_t *dev_name_slot;
  /* iommuMap part */
  uint64_t n_grp_members;
  const kvg_pci_surv *grp_members;
  uint32_t n_groups;
  const uint32_t *grp_keys;
  const uint32_t *grp_off;
  const uint32_t *grp_perm;
  const uint8_t *name_pool;
  size_t name_pool_len;
} kvg_pci_shard_result;

typedef struct kvg_mdev_shard_result {
  uint64_t n_records;
  uint64_t n_local;
  const kvg_mdev_surv *local;     /* [n_local] this shard's surviving mdevs, Walk order */
  /* vGpuMap part: canonical type ids owned by this rank */
  uint64_t n_type_members;
  const kvg_mdev_surv *type_members;
  uint32_t n_type_keys;
  const uint16_t *type_keys;
  const uint32_t *type_off;
  const uint32_t *type_perm;
  /* gpuVgpuMap part: parent handles owned by this rank */
  uint64_t n_par_members;
  const kvg_mdev_surv *par_members;
  uint32_t n_parents;
  const uint32_t *par_keys;
  const uint32_t *par_off;
  const uint32_t *par_perm;
  /* the type dictionary as in kvg_mdev_result (every rank loads the same dictionary) */
  uint32_t n_types;
  const uint32_t *label_off;
  const uint8_t *label_bytes;
  const uint16_t *type_canon;
  const uint32_t *type_name_off;
  const uint8_t *type_name_bytes;
} kvg_mdev_shard_result;

/* Health transitions of one re-scan relative to the previous one (record order). */
typedef struct kvg_health_delta {
  uint32_t n_records;
  uint32_t n_alive;   /* records passing the classification predicate now */
  uint32_t n_changed;
  const uint32_t *changed; /* [n_changed] (record index << 1) | now_alive, ascending index */
} kvg_health_delta;

/* ---- rescans (runtime rediscovery) -----------------------------------------------------------
 * A rescan is a full scan of a fresh snapshot, diffed ON THE DEVICE against the previous successful rescan of
 * the same kind on the same context (its baseline).
 *
 * Identity: a survivor is identified by `addr` (PCI) or by its 16 uuid bytes compared as a big-endian string
 * (mdev).  The survivors of a snapshot must be strictly ascending in that identity, which is Walk order in
 * numeric mode; the device checks it, and a violation returns KVG_EINVAL and keeps the baseline.  Snapshots in
 * index mode (addresses / uuids that are Walk indices, interned groups, devices or parents) have no stable
 * identity; the library cannot detect them and they must not be passed here.
 *
 * moved: identity in both lists, a map-relevant field differs (PCI: iommu_group, device, numa; mdev: type_key,
 * parent, numa; name_slot and src never count).
 * changed key: present before and after, and its member list AS THAT MAP STORES IT differs.  deviceMap,
 * iommuMap and vGpuMap store (addr|uuid, numa) in Walk order; gpuVgpuMap stores uuids only.  So a group-only
 * move changes two iommuMap keys and no deviceMap key; a numa-only mdev move changes its vGpuMap key and no
 * gpuVgpuMap key.
 * Type ids: the `types` of kvg_rescan_mdev must start with the previous rescan's dictionary byte for byte (new
 * raw names may only be appended), else KVG_EINVAL: canonical type ids are only stable under that rule.
 * Resets: kvg_pciids_load and kvg_rescan_reset drop both baselines; the next rescan then reports every
 * survivor and key as added.  Baselines are independent of kvg_scan_*, kvg_dev_* and the health state.
 * The result is one library-owned block, freed with kvg_result_free. */
typedef struct kvg_key_delta { /* one group-by map; every list ascending */
  uint32_t n_added;   const uint32_t *added;   /* keys absent before, present now             */
  uint32_t n_removed; const uint32_t *removed; /* keys present before, absent now             */
  uint32_t n_changed; const uint32_t *changed; /* present before and now, member list differs */
} kvg_key_delta;

typedef struct kvg_pci_rescan {
  kvg_pci_result scan;             /* identical to kvg_scan_pci on the same records */
  uint32_t had_baseline;           /* 0: first rescan since a reset -> everything is "added" */
  uint64_t n_added;   const uint32_t *added;       /* indices into scan.survivors, ascending */
  uint64_t n_removed; const kvg_pci_surv *removed; /* previous survivors, ascending addr      */
  uint64_t n_moved;   const uint32_t *moved;       /* indices into scan.survivors: same addr,
                                                      iommu_group / device / numa changed    */
  kvg_key_delta dev;               /* deviceMap, keys = device ids */
  kvg_key_delta grp;               /* iommuMap,  keys = group ids  */
} kvg_pci_rescan;

typedef struct kvg_mdev_rescan {
  kvg_mdev_result scan;            /* identical to kvg_scan_mdev */
  uint32_t had_baseline;
  uint64_t n_added;   const uint32_t *added;
  uint64_t n_removed; const kvg_mdev_surv *removed;
  uint64_t n_moved;   const uint32_t *moved;       /* same uuid, type_key / parent / numa changed */
  kvg_key_delta type;              /* vGpuMap,    keys = canonical type ids */
  kvg_key_delta parent;            /* gpuVgpuMap, keys = parent handles     */
} kvg_mdev_rescan;

/* ---- context -------------------------------------------------------------------------------- */
typedef struct kvg_ctx kvg_ctx;

int kvg_abi_version(void);
int kvg_ctx_create(int cuda_device, kvg_ctx **out);
void kvg_ctx_destroy(kvg_ctx *ctx);
const char *kvg_last_error(kvg_ctx *ctx); /* ctx may be NULL: last create error */
void kvg_result_free(void *result);
/* kernels launched by this context since creation (bench.py "gpu_launches") */
uint64_t kvg_launch_count(kvg_ctx *ctx);
/* the context's cudaStream_t, for CUDA-event timing on the launching stream */
void *kvg_stream(kvg_ctx *ctx);

/* ---- pci.ids name table (getDeviceName, device_plugin.go:371-438) --------------------------- */

/* Parse `text` on the GPU: line split, vendor context, (vendor,device)->line hash, NVIDIA
 * section bounds, sanitised names.  Idempotent: a second call replaces the table.
 * Pageable `text` (Go, Python bytes): copied and published before the call returns.
 * Page-locked `text` (cudaHostAlloc / cudaHostRegister): the call only ENQUEUES copy + parse, so
 * that the next call's host-to-device traffic overlaps it; the buffer must stay valid, and a
 * table-capacity error is reported, by the first later call on `ctx` that consumes the table
 * (kvg_name_lookup / kvg_name_table / kvg_pciids_info / any scan). */
int kvg_pciids_load(kvg_ctx *ctx, const uint8_t *text, size_t len);

/* Exact getDeviceName(key) for ANY key bytes: "" (outlen 0) when not found.  4-lower-hex keys go
 * through the table; every other key through the prefix-match kernel (device_plugin.go:388-400). */
int kvg_name_lookup(kvg_ctx *ctx, const char *key, size_t keylen, char *out, size_t cap,
                    size_t *outlen);

/* Bulk form used by tests and the Go shim: names of device ids [first, first+count) through the
 * table path; out_off has count+1 entries into out_bytes (cap bytes). */
int kvg_name_table(kvg_ctx *ctx, uint32_t first, uint32_t count, uint32_t *out_off,
                   uint8_t *out_bytes, size_t cap);

/* table facts after load: byte offsets of the first "10de" line and of the section end,
 * number of (vendor,device) entries inserted, number of text lines */
int kvg_pciids_info(kvg_ctx *ctx, uint32_t *vendor_off, uint32_t *section_end, uint32_t *n_entries,
                    uint32_t *n_lines);

/* ---- scans, host buffers in / host results out (the reference-facing calls) ---------------- */
int kvg_scan_pci(kvg_ctx *ctx, const kvg_pci_rec *recs, size_t n, kvg_pci_result **res);
/* (128 Ki <= n <= 16 Mi records: the snapshot is copied, classified and its survivors returned
 *  chunk by chunk on separate copy streams; results are identical.  KVG_PIPELINE=0 disables.) */
int kvg_scan_mdev(kvg_ctx *ctx, const kvg_mdev_rec *recs, size_t n, const kvg_type_dict *types,
                  kvg_mdev_result **res);
/* Classify `recs`, diff against the alive-set of the previous call on this context (first call:
 * against "nothing alive").  n must stay constant between calls; kvg_health_reset() re-arms. */
int kvg_health_rescan(kvg_ctx *ctx, const kvg_pci_rec *recs, size_t n, kvg_health_delta **delta);
int kvg_health_reset(kvg_ctx *ctx);
/* Scan `recs` exactly as kvg_scan_pci / kvg_scan_mdev do and diff the result against the baseline (see
 * "rescans" above); on success the new scan becomes the baseline. */
int kvg_rescan_pci(kvg_ctx *ctx, const kvg_pci_rec *recs, size_t n, kvg_pci_rescan **res);
int kvg_rescan_mdev(kvg_ctx *ctx, const kvg_mdev_rec *recs, size_t n, const kvg_type_dict *types,
                    kvg_mdev_rescan **res);
int kvg_rescan_reset(kvg_ctx *ctx); /* drops both baselines */

/* ---- device-resident entry points (inputs already in HBM; used by bench.py "value") -------- */

/* Layout contract for device text: 16-byte aligned `d_text`, 16 readable bytes BEFORE it and
 * kvg_text_pad(len) readable bytes from it, all padding bytes '\n'.  n_files images of `len`
 * bytes each, image f at d_text + f*stride (stride % 16 == 0, stride >= kvg_text_pad(len)+16).
 * Image 0 becomes the context's table; images >= 1 are parsed into scratch tables (batch
 * throughput measurement: every byte is split, every line start classified).
 * The first call on an image publishes its table (synchronous).  A later call on the SAME single image
 * re-parses it asynchronously on the context's side stream: it starts when everything enqueued before it
 * has finished, kvg_dev_scan_pci / kvg_dev_scan_pci_sharded enqueued after it classify and sort beside
 * it and join the names in their last kernel, every other consumer of the table waits for it first.
 * d_text must stay valid until the next call on the context that synchronises (any fetch / count). */
size_t kvg_text_pad(size_t len);
int kvg_dev_pciids_parse(kvg_ctx *ctx, const void *d_text, size_t len, size_t stride,
                         uint32_t n_files);
/* enqueue classify + stable compaction + both bucketings on the context stream; no host sync */
int kvg_dev_scan_pci(kvg_ctx *ctx, const void *d_recs, size_t n);
/* synchronise, copy the result of the last kvg_dev_scan_pci to the host */
int kvg_dev_scan_pci_fetch(kvg_ctx *ctx, kvg_pci_result **res);
/* survivor count of the last enqueued scan (synchronises the stream) */
int kvg_dev_scan_pci_count(kvg_ctx *ctx, uint64_t *n_survivors, uint32_t *n_dev_keys,
                           uint32_t *n_groups);
/* synthetic snapshot generators (counter-based splitmix64; oracle/kvg_oracle.c has the CPU twin) */
int kvg_dev_gen_pci(kvg_ctx *ctx, void *d_recs, uint64_t first, size_t n, const uint16_t *nv_ids,
                    uint32_t n_nv_ids, uint32_t group_bits);
int kvg_dev_gen_mdev(kvg_ctx *ctx, void *d_recs, uint64_t first, size_t n);
int kvg_dev_scan_mdev(kvg_ctx *ctx, const void *d_recs, size_t n, const kvg_type_dict *types);
int kvg_dev_scan_mdev_fetch(kvg_ctx *ctx, kvg_mdev_result **res);
/* Diagnostics: the pass structure (count, shift and width of each pass) the radix kernels derive on
 * the device for an ordering whose largest key is `max_key` (key_bits_max 16 or 32; max_bits 11, or 8 for
 * inputs >= 8 Mi records): pass 0 always takes the low max_bits bits, the remaining key bits are split
 * evenly over the fewest further passes.  Pure host arithmetic: usable without a GPU. */
int kvg_debug_radix_plan(uint32_t max_key, uint32_t key_bits_max, uint32_t max_bits, uint32_t *npass,
                         uint32_t *shifts4, uint32_t *bits4);

/* write `bytes` of zeros through a scratch buffer larger than L2 (timing hygiene, untimed) */
int kvg_dev_flush_l2(kvg_ctx *ctx);
/* per-kernel device time of the last kvg_dev_scan_pci / kvg_dev_pciids_parse, CUDA events on the
 * context stream; names is a NUL-separated list; returns count */
int kvg_kernel_times(kvg_ctx *ctx, float *ms, char *names, size_t names_cap, int max_n);
int kvg_set_kernel_timing(kvg_ctx *ctx, int enabled);

/* ---- multi-GPU (BASELINE.json config 4): one process per GPU, records range-sharded --------- */
#define KVG_UNIQUE_ID_BYTES 128
int kvg_comm_unique_id(void *out128);
int kvg_comm_init(kvg_ctx *ctx, int rank, int nranks, const void *unique_id128);
int kvg_comm_destroy(kvg_ctx *ctx);
/* Peer-memory exchange (CUDA IPC over NVLink, one process per GPU of ONE node): export allocates this
 * rank's receive window for shards of up to cap_local PCI records (cap_local / 2 mdev records) and returns
 * a 64-byte handle; import opens all ranks' handles (nranks x 64 bytes, rank order).  Afterwards the sharded
 * scans exchange by storing into the owners' windows and need neither NCCL nor a host synchronisation.
 * If either call fails the NCCL path (kvg_comm_init) remains usable. */
int kvg_comm_p2p_export(kvg_ctx *ctx, int rank, int nranks, size_t cap_local, void *handle_out64);
int kvg_comm_p2p_import(kvg_ctx *ctx, const void *all_handles);
/* collective decision: enable only when import succeeded on every rank */
int kvg_comm_p2p_enable(kvg_ctx *ctx, int on);
/* Classify the local shard (device memory), send every survivor to the owner of its key (once per
 * group-by map: key % nranks), order the owned members.  Peer windows: the multisplit stores straight into
 * the owners' windows over NVLink, nothing returns to the host.  NCCL mode: one allgatherv of the survivor
 * lists (two host synchronisations for the counts), then the same kernels keep what this rank owns.
 * Collective: every rank of the communicator must call it, in the same order. */
int kvg_dev_scan_pci_sharded(kvg_ctx *ctx, const void *d_recs, size_t n_local);
int kvg_dev_scan_pci_shard_fetch(kvg_ctx *ctx, kvg_pci_shard_result **res);
/* the same for mdev records (createVgpuIDMap): type / parent orderings of the owned members */
int kvg_dev_scan_mdev_sharded(kvg_ctx *ctx, const void *d_recs, size_t n_local, const kvg_type_dict *types);
int kvg_dev_scan_mdev_shard_fetch(kvg_ctx *ctx, kvg_mdev_shard_result **res);

#ifdef __cplusplus
}
#endif
#endif /* KVGPU_H */
