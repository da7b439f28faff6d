//go:build cgo

// Package device_plugin — cgo shim that routes the reference's discovery scan through libkvgpu.so.
//
// SOURCE ONLY: this image has no Go toolchain, so this file has never been compiled here (round-1 review
// findings — cgo pointer rule for the type dictionary, locking, range checks — are addressed in source).  It is
// the binding a maintainer of NVIDIA/kubevirt-gpu-device-plugin drops into pkg/device_plugin/
// next to device_plugin.go (see INTEGRATION.md).  It contains marshalling only — every decision
// (filter, join, bucketing, name sanitising) is made by the CUDA library behind include/kvgpu.h.
//
// It replaces the BODIES of three functions and keeps their signatures and side effects:
//
//	createIommuDeviceMap()            device_plugin.go:187  -> createIommuDeviceMapGPU()
//	createVgpuIDMap()                 device_plugin.go:255  -> createVgpuIDMapGPU()
//	getDeviceName(deviceID string)    device_plugin.go:371  -> getDeviceNameGPU(deviceID)
//
// The five sysfs readers stay the reference's own package variables (readIDFromFile, readLink,
// readNUMANode, readVgpuIDFromFile is replaced by a raw read, readGpuIDForVgpu :80-85), so the
// existing Ginkgo fakes keep working unchanged.
package device_plugin

/*
#cgo CFLAGS: -I${SRCDIR}/../../include
#cgo LDFLAGS: -L${SRCDIR}/.. -lkvgpu -Wl,-rpath,${SRCDIR}/..
#include <stdlib.h>
#include "kvgpu.h"
*/
import "C"

import (
	"fmt"
	"log"
	"os"
	"path/filepath"
	"sort"
	"strconv"
	"strings"
	"sync"
	"unsafe"
)

var kvgCtx *C.kvg_ctx
var kvgLoadedPath string

// A kvg_ctx is single-threaded (include/kvgpu.h).  The scans run on the main goroutine before any server
// starts, but getDeviceNameGPU and revalidateBatchGPU are reached from gRPC handler goroutines (grpc-go runs
// one goroutine per stream) and from healthCheck goroutines: every entry into the library takes kvgMu.
var kvgMu sync.Mutex

// kvgEnsure creates the context once and (re)loads the pci.ids table when the path changed.
// A CUDA failure is reported like the reference reports a failed walk: log + empty maps.
func kvgEnsure() error {
	if kvgCtx == nil {
		if rc := C.kvg_ctx_create(0, &kvgCtx); rc != C.KVG_OK {
			return fmt.Errorf("kvg_ctx_create: %d %s", int(rc), C.GoString(C.kvg_last_error(nil)))
		}
	}
	if kvgLoadedPath != pciIdsFilePath {
		data, err := os.ReadFile(pciIdsFilePath)
		if err != nil {
			log.Printf("Error opening pci ids file %s", pciIdsFilePath) // :375
			data = nil                                                  // empty table: every name is ""
		}
		var p *C.uint8_t
		if len(data) > 0 {
			p = (*C.uint8_t)(unsafe.Pointer(&data[0]))
		}
		if rc := C.kvg_pciids_load(kvgCtx, p, C.size_t(len(data))); rc != C.KVG_OK {
			return fmt.Errorf("kvg_pciids_load: %s", C.GoString(C.kvg_last_error(kvgCtx)))
		}
		kvgLoadedPath = pciIdsFilePath
	}
	return nil
}

func getDeviceNameGPU(deviceID string) string {
	kvgMu.Lock()
	defer kvgMu.Unlock()
	return getDeviceNameLocked(deviceID)
}

func getDeviceNameLocked(deviceID string) string {
	if err := kvgEnsure(); err != nil {
		log.Printf("Error: %v", err)
		return ""
	}
	out := make([]byte, 1<<17)
	var n C.size_t
	key := C.CString(deviceID)
	defer C.free(unsafe.Pointer(key))
	rc := C.kvg_name_lookup(kvgCtx, key, C.size_t(len(deviceID)), (*C.char)(unsafe.Pointer(&out[0])),
		C.size_t(len(out)), &n)
	if rc != C.KVG_OK {
		return ""
	}
	return string(out[:n])
}

func parseHex4(s string) (uint16, bool) {
	if len(s) != 4 {
		return 0, false
	}
	v, err := strconv.ParseUint(s, 16, 16)
	if err != nil || strings.ToLower(s) != s {
		return 0, false
	}
	return uint16(v), true
}

// createIommuDeviceMapGPU: same walk, same readers, same short-circuit order as :192-246, but the
// entries are only RECORDED (read failures become flag bits); the GPU filters, joins and buckets.
func createIommuDeviceMapGPU() {
	kvgMu.Lock()
	defer kvgMu.Unlock()
	iommuMap = make(map[string][]NvidiaGpuDevice)
	deviceMap = make(map[string][]NvidiaGpuDevice)
	bdfToIommuMap = make(map[string]string)
	var names []string
	var recs []C.kvg_pci_rec
	groupIDs := map[string]uint32{}
	var groupNames []string
	// `device` strings travel in index mode: the reference keeps WHATEVER the file holds as the map key
	// (:240, :294-302), so the record carries an interned id and the string stays here
	deviceIDs := map[string]uint16{}
	var deviceNames []string
	rangeErr := ""
	filepath.Walk(basePath, func(path string, info os.FileInfo, err error) error {
		if err != nil {
			log.Printf("Error accessing file path %q: %v\n", path, err)
			return err
		}
		if info.IsDir() {
			return nil
		}
		var r C.kvg_pci_rec
		r.addr = C.uint32_t(len(names)) // index mode: names[] maps the handle back
		r.vendor = 0xffff
		vendorID, err := readIDFromFile(basePath, info.Name(), "vendor")
		if err != nil {
			r.flags |= C.KVG_PF_VENDOR_ERR
		} else if v, ok := parseHex4(vendorID); ok {
			r.vendor = C.uint16_t(v)
		}
		if err == nil && vendorID == nvidiaVendorID {
			driver, err := readLink(basePath, info.Name(), "driver")
			switch {
			case err != nil:
				r.flags |= C.KVG_PF_DRIVER_ERR
			case driver == "vfio-pci":
				r.driver = C.KVG_DRV_VFIO_PCI
			case driver == "nvgrace_gpu_vfio_pci":
				r.driver = C.KVG_DRV_NVGRACE
			default:
				r.driver = C.KVG_DRV_OTHER
			}
			if err == nil && isSupportedVfioDriver(driver) {
				iommuGroup, err := readLink(basePath, info.Name(), "iommu_group")
				if err != nil {
					r.flags |= C.KVG_PF_IOMMU_ERR
				} else {
					id, ok := groupIDs[iommuGroup]
					if !ok {
						id = uint32(len(groupNames))
						groupIDs[iommuGroup] = id
						groupNames = append(groupNames, iommuGroup)
					}
					r.iommu_group = C.uint32_t(id)
					numaNode, err := readNUMANode(basePath, info.Name())
					if err != nil {
						r.flags |= C.KVG_PF_NUMA_ERR
					} else if numaNode < -32768 || numaNode > 32767 {
						// the 16-byte record carries an int16: refuse loudly (kvgpu/plugin.py: KVG_ERANGE)
						rangeErr = fmt.Sprintf("numa_node %d of %s does not fit the wire format", numaNode, info.Name())
					}
					r.numa = C.int16_t(numaNode)
					deviceID, err := readIDFromFile(basePath, info.Name(), "device")
					if err != nil {
						r.flags |= C.KVG_PF_DEVICE_ERR
					} else {
						id, ok := deviceIDs[deviceID]
						if !ok {
							if len(deviceNames) > 0xffff {
								rangeErr = "more than 65536 distinct device strings"
							}
							id = uint16(len(deviceNames))
							deviceIDs[deviceID] = id
							deviceNames = append(deviceNames, deviceID)
						}
						r.device = C.uint16_t(id)
					}
				}
			}
		}
		names = append(names, info.Name())
		recs = append(recs, r)
		return nil
	})
	if rangeErr != "" {
		log.Printf("Error: %s", rangeErr) // maps stay empty, like a failed walk (:193-196)
		return
	}
	if err := kvgEnsure(); err != nil {
		log.Printf("Error: %v", err) // maps stay empty, like a failed walk (:193-196)
		return
	}
	var res *C.kvg_pci_result
	var p *C.kvg_pci_rec
	if len(recs) > 0 {
		p = &recs[0]
	}
	if rc := C.kvg_scan_pci(kvgCtx, p, C.size_t(len(recs)), &res); rc != C.KVG_OK {
		log.Printf("Error: kvg_scan_pci: %s", C.GoString(C.kvg_last_error(kvgCtx)))
		return
	}
	defer C.kvg_result_free(unsafe.Pointer(res))
	S := int(res.n_survivors)
	surv := unsafe.Slice(res.survivors, S)
	dev := func(i uint32) NvidiaGpuDevice {
		return NvidiaGpuDevice{addr: names[surv[i].addr], numaNode: int64(surv[i].numa)}
	}
	devKeys := unsafe.Slice(res.dev_keys, int(res.n_dev_keys))
	devOff := unsafe.Slice(res.dev_off, int(res.n_dev_keys)+1)
	devPerm := unsafe.Slice(res.dev_perm, S)
	for k := range devKeys {
		key := deviceNames[devKeys[k]] // index mode; getDeviceName(key) is asked later with these exact bytes
		for _, i := range devPerm[devOff[k]:devOff[k+1]] {
			deviceMap[key] = append(deviceMap[key], dev(uint32(i)))
		}
	}
	grpKeys := unsafe.Slice(res.grp_keys, int(res.n_groups))
	grpOff := unsafe.Slice(res.grp_off, int(res.n_groups)+1)
	grpPerm := unsafe.Slice(res.grp_perm, S)
	for k := range grpKeys {
		g := groupNames[grpKeys[k]]
		for _, i := range grpPerm[grpOff[k]:grpOff[k+1]] {
			iommuMap[g] = append(iommuMap[g], dev(uint32(i)))
		}
	}
	for i := 0; i < S; i++ {
		bdfToIommuMap[names[surv[i].addr]] = groupNames[surv[i].iommu_group]
	}
}

// createVgpuIDMapGPU: :259-290 with the label rule (:341-342) and both group-bys on the GPU.
func createVgpuIDMapGPU() {
	kvgMu.Lock()
	defer kvgMu.Unlock()
	vGpuMap = make(map[string][]NvidiaGpuDevice)
	gpuVgpuMap = make(map[string][]string)
	var names, parentNames []string
	var recs []C.kvg_mdev_rec
	typeIDs := map[string]uint16{}
	var rawTypes [][]byte
	parentIDs := map[string]uint32{}
	filepath.Walk(vGpuBasePath, func(path string, info os.FileInfo, err error) error {
		if err != nil {
			return err
		}
		if info.IsDir() {
			return nil
		}
		var r C.kvg_mdev_rec
		idx := uint32(len(names))
		r.uuid[0], r.uuid[1], r.uuid[2], r.uuid[3] = C.uint8_t(idx>>24), C.uint8_t(idx>>16), C.uint8_t(idx>>8), C.uint8_t(idx)
		raw, err := os.ReadFile(filepath.Join(vGpuBasePath, info.Name(), "mdev_type/name")) // raw: the GPU sanitises
		if err != nil {
			r.flags |= C.KVG_MF_TYPE_ERR
		} else {
			id, ok := typeIDs[string(raw)]
			if !ok {
				id = uint16(len(rawTypes))
				typeIDs[string(raw)] = id
				rawTypes = append(rawTypes, raw)
			}
			r.type_idx = C.uint16_t(id)
			gpuID, err := readGpuIDForVgpu(vGpuBasePath, info.Name())
			if err != nil {
				r.flags |= C.KVG_MF_PARENT_ERR
			} else {
				id, ok := parentIDs[gpuID]
				if !ok {
					id = uint32(len(parentNames))
					parentIDs[gpuID] = id
					parentNames = append(parentNames, gpuID)
				}
				r.parent = C.uint32_t(id)
				numaNode, err := readNUMANode(basePath, gpuID)
				if err != nil {
					r.flags |= C.KVG_MF_NUMA_ERR
				}
				r.parent_numa = C.int16_t(numaNode)
			}
		}
		names = append(names, info.Name())
		recs = append(recs, r)
		return nil
	})
	if err := kvgEnsure(); err != nil {
		log.Printf("Error: %v", err)
		return
	}
	// The dictionary struct holds two pointers: they must not be Go pointers (cgo rule: a Go pointer passed to
	// C may not point at memory that itself holds Go pointers), so both arrays live in C memory for the call.
	total := 0
	for _, t := range rawTypes {
		total += len(t)
	}
	cOff := (*C.uint32_t)(C.malloc(C.size_t(4 * (len(rawTypes) + 1))))
	cBlob := (*C.uint8_t)(C.malloc(C.size_t(total + 1)))
	defer C.free(unsafe.Pointer(cOff))
	defer C.free(unsafe.Pointer(cBlob))
	off := unsafe.Slice(cOff, len(rawTypes)+1)
	blob := unsafe.Slice((*byte)(unsafe.Pointer(cBlob)), total+1)
	off[0] = 0
	pos := 0
	for i, t := range rawTypes {
		pos += copy(blob[pos:], t)
		off[i+1] = C.uint32_t(pos)
	}
	blob[total] = 0
	dict := C.kvg_type_dict{n_types: C.uint32_t(len(rawTypes)), off: cOff, bytes: cBlob}
	var res *C.kvg_mdev_result
	var p *C.kvg_mdev_rec
	if len(recs) > 0 {
		p = &recs[0]
	}
	if rc := C.kvg_scan_mdev(kvgCtx, p, C.size_t(len(recs)), &dict, &res); rc != C.KVG_OK {
		log.Printf("Error: kvg_scan_mdev: %s", C.GoString(C.kvg_last_error(kvgCtx)))
		return
	}
	defer C.kvg_result_free(unsafe.Pointer(res))
	S := int(res.n_survivors)
	surv := unsafe.Slice(res.survivors, S)
	labelOff := unsafe.Slice(res.label_off, int(res.n_types)+1)
	labels := unsafe.Slice((*byte)(unsafe.Pointer(res.label_bytes)), int(labelOff[res.n_types]))
	tKeys := unsafe.Slice(res.type_keys, int(res.n_type_keys))
	tOff := unsafe.Slice(res.type_off, int(res.n_type_keys)+1)
	tPerm := unsafe.Slice(res.type_perm, S)
	for k := range tKeys {
		t := tKeys[k]
		label := string(labels[labelOff[t]:labelOff[t+1]])
		for _, i := range tPerm[tOff[k]:tOff[k+1]] {
			vGpuMap[label] = append(vGpuMap[label], NvidiaGpuDevice{addr: names[surv[i].src], numaNode: int64(surv[i].numa)})
		}
	}
	pKeys := unsafe.Slice(res.par_keys, int(res.n_parents))
	pOff := unsafe.Slice(res.par_off, int(res.n_parents)+1)
	pPerm := unsafe.Slice(res.par_perm, S)
	for k := range pKeys {
		g := parentNames[pKeys[k]]
		for _, i := range pPerm[pOff[k]:pOff[k+1]] {
			gpuVgpuMap[g] = append(gpuVgpuMap[g], names[surv[i].src])
		}
	}
	_ = sort.Strings // (kept: callers that want deterministic logs sort the keys)
}

// revalidateBatchGPU is the Allocate-time re-check of generic_device_plugin.go:387-399 for ALL devices
// of a container request in one pass of the classification kernel (Python twin:
// kvgpu/serve.py BatchRevalidator, pinned by tests/test_serve.py).  devs[i] is re-read with the
// reference's own readers, in the reference's order; want[i] is the IOMMU group the maps hold for it.
// It returns the index of the first device the reference would reject, or -1.
//
// The record's driver is pinned to vfio-pci and its device id to 0 because Allocate re-checks only the
// group link and the vendor; K3's predicate is then exactly "vendor is 10de and both reads worked" and
// the survivor's interned group id says whether the link still points at the expected group.
//
// Call site (generic_device_plugin.go:376-416): collect (dev.addr, iommuId) for every dev of every
// requested BDF, call this once, and return the "unknown device" error for devs[first] if first >= 0.
func revalidateBatchGPU(devs []string, want []string) (first int, err error) {
	if len(devs) == 0 {
		return -1, nil
	}
	kvgMu.Lock()
	defer kvgMu.Unlock()
	if err := kvgEnsure(); err != nil {
		return 0, err
	}
	intern := map[string]uint32{}
	id := func(s string) uint32 {
		if v, ok := intern[s]; ok {
			return v
		}
		v := uint32(len(intern))
		intern[s] = v
		return v
	}
	recs := make([]C.kvg_pci_rec, len(devs))
	for i, addr := range devs {
		r := &recs[i]
		r.addr = C.uint32_t(i)
		r.vendor = 0xffff
		r.driver = C.KVG_DRV_VFIO_PCI
		r.iommu_group = C.uint32_t(id(want[i]))
		group, err := readLink(basePath, addr, "iommu_group")
		if err != nil {
			r.flags |= C.KVG_PF_IOMMU_ERR
		} else {
			r.iommu_group = C.uint32_t(id(group))
		}
		vendorID, err := readIDFromFile(basePath, addr, "vendor")
		if err != nil {
			r.flags |= C.KVG_PF_VENDOR_ERR
		} else if vendorID == nvidiaVendorID {
			r.vendor = 0x10de
		}
	}
	var res *C.kvg_pci_result
	if rc := C.kvg_scan_pci(kvgCtx, &recs[0], C.size_t(len(recs)), &res); rc != C.KVG_OK {
		return 0, fmt.Errorf("kvg_scan_pci: %s", C.GoString(C.kvg_last_error(kvgCtx)))
	}
	defer C.kvg_result_free(unsafe.Pointer(res))
	ok := make(map[uint32]uint32, int(res.n_survivors))
	for _, s := range unsafe.Slice(res.survivors, int(res.n_survivors)) {
		ok[uint32(s.addr)] = uint32(s.iommu_group)
	}
	for i := range devs {
		if g, alive := ok[uint32(i)]; !alive || g != intern[want[i]] {
			return i, nil
		}
	}
	return -1, nil
}

// pluginDelta is what one rediscovery asks of the plugin servers (createDevicePlugins :131-137, :158-165).
type pluginDelta struct {
	Start, Stop, Resend []string // deviceMap keys ("%04x"); vGPU keys are returned by type id below
	StartVgpu, StopVgpu, ResendVgpu []uint16
}

// rescanGPU: runtime rediscovery (SOURCE ONLY, unverified like the rest of this file).  The caller builds
// snapshots in NUMERIC mode (addr = packed BDF, mdev uuid bytes, numeric groups and device ids, Walk order) and a
// raw type dictionary that only grows at its end; the GPU diffs them against the previous rescan
// (kvg_rescan_pci / kvg_rescan_mdev) and the key deltas become plugin actions: an added key starts a plugin, a
// removed key stops it, a changed key re-sends its ListAndWatch list.  Changed iommuMap / gpuVgpuMap keys need no
// plugin action: returnIommuMap / returnGpuVgpuMap read the rebuilt maps.  A snapshot that cannot be numeric
// (interned names) must not come here: restart the plugins instead.  firstScan reports a missing baseline.
func rescanGPU(pci []C.kvg_pci_rec, mdev []C.kvg_mdev_rec, dictOff []uint32, dictBytes []byte) (d pluginDelta, firstScan bool, err error) {
	kvgMu.Lock()
	defer kvgMu.Unlock()
	if err := kvgEnsure(); err != nil {
		return d, false, err
	}
	var pr *C.kvg_pci_rescan
	var pp *C.kvg_pci_rec
	if len(pci) > 0 {
		pp = &pci[0]
	}
	if rc := C.kvg_rescan_pci(kvgCtx, pp, C.size_t(len(pci)), &pr); rc != C.KVG_OK {
		return d, false, fmt.Errorf("kvg_rescan_pci: %s", C.GoString(C.kvg_last_error(kvgCtx)))
	}
	defer C.kvg_result_free(unsafe.Pointer(pr))
	keys := func(k C.kvg_key_delta) (a, r, c []uint32) {
		a = append(a, unsafe.Slice((*uint32)(unsafe.Pointer(k.added)), int(k.n_added))...)
		r = append(r, unsafe.Slice((*uint32)(unsafe.Pointer(k.removed)), int(k.n_removed))...)
		c = append(c, unsafe.Slice((*uint32)(unsafe.Pointer(k.changed)), int(k.n_changed))...)
		return
	}
	a, r, c := keys(pr.dev)
	hex := func(v []uint32) (out []string) {
		for _, k := range v {
			out = append(out, fmt.Sprintf("%04x", k))
		}
		return
	}
	d.Start, d.Stop, d.Resend = hex(a), hex(r), hex(c)
	// the dictionary is copied into C memory: no Go pointer to Go memory crosses the call (cgo rule)
	nt := len(dictOff) - 1
	if nt < 0 {
		nt = 0
	}
	cOff := (*C.uint32_t)(C.malloc(C.size_t(4 * (nt + 1))))
	defer C.free(unsafe.Pointer(cOff))
	cBytes := (*C.uint8_t)(C.malloc(C.size_t(len(dictBytes) + 1)))
	defer C.free(unsafe.Pointer(cBytes))
	offs := unsafe.Slice((*uint32)(unsafe.Pointer(cOff)), nt+1)
	offs[0] = 0
	copy(offs, dictOff)
	copy(unsafe.Slice((*byte)(unsafe.Pointer(cBytes)), len(dictBytes)+1), dictBytes)
	types := C.kvg_type_dict{n_types: C.uint32_t(nt), off: cOff, bytes: cBytes}
	var mr *C.kvg_mdev_rescan
	var mp *C.kvg_mdev_rec
	if len(mdev) > 0 {
		mp = &mdev[0]
	}
	if rc := C.kvg_rescan_mdev(kvgCtx, mp, C.size_t(len(mdev)), &types, &mr); rc != C.KVG_OK {
		return d, false, fmt.Errorf("kvg_rescan_mdev: %s", C.GoString(C.kvg_last_error(kvgCtx)))
	}
	defer C.kvg_result_free(unsafe.Pointer(mr))
	a, r, c = keys(mr._type)
	for _, v := range a {
		d.StartVgpu = append(d.StartVgpu, uint16(v))
	}
	for _, v := range r {
		d.StopVgpu = append(d.StopVgpu, uint16(v))
	}
	for _, v := range c {
		d.ResendVgpu = append(d.ResendVgpu, uint16(v))
	}
	return d, pr.had_baseline == 0 || mr.had_baseline == 0, nil
}
