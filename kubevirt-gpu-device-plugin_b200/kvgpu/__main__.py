"""python -m kvgpu — InitiateDevicePlugin() of the reference (device_plugin.go:89-96, cmd/main.go) on
top of the GPU scan: createIommuDeviceMap + createVgpuIDMap through libkvgpu.so, then one
DevicePlugin server per device id / vGPU type, registered with the kubelet.

  python -m kvgpu --once --dump            scan, print the canonical dump, exit (no servers)
  python -m kvgpu --once --plugins         scan, print what each plugin would advertise (JSON)
  python -m kvgpu                          scan, serve, watch the device nodes, run until SIGTERM
  python -m kvgpu --rediscover-period 5    the same, and rescan every 5 s: plugins start, stop and update
                                           as devices and vGPUs appear, disappear or change

There is no CPU fallback: without a usable CUDA device the scan fails and the process exits non-zero
(the reference would log the failed walk and start no plugin)."""
import argparse
import json
import signal
import sys
import threading


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="python -m kvgpu", description=__doc__.split("\n\n")[0])
    ap.add_argument("--pci-ids", default="/usr/pci.ids", help="pciIdsFilePath (device_plugin.go:44)")
    ap.add_argument("--base-path", default="/sys/bus/pci/devices", help="basePath (:42)")
    ap.add_argument("--vgpu-base-path", default="/sys/bus/mdev/devices", help="vGpuBasePath (:43)")
    ap.add_argument("--root-path", default="/", help="rootPath for /dev/iommu and EGM discovery")
    ap.add_argument("--socket-dir", default=None, help="kubelet device-plugin directory (pluginapi.DevicePluginPath)")
    ap.add_argument("--device", type=int, default=0, help="CUDA device running the scan")
    ap.add_argument("--once", action="store_true", help="scan and print, do not serve")
    ap.add_argument("--dump", action="store_true", help="print the canonical dump of the five maps")
    ap.add_argument("--plugins", action="store_true", help="print the plugin specs as JSON")
    ap.add_argument("--rediscover-period", type=float, default=0.0, metavar="SECONDS",
                    help="rescan the trees this often and start / stop / update plugins (0: scan once)")
    args = ap.parse_args(argv)

    from . import DiscoveryScan, KvgError, canonical_dump
    try:
        ds = DiscoveryScan(args.pci_ids, args.base_path, args.vgpu_base_path, args.device)
    except KvgError as e:
        print("kvgpu: cannot create the scan context (no CPU fallback): %s" % e, file=sys.stderr)
        return 2
    try:
        if args.rediscover_period > 0 and not args.once:
            ds.rediscover()               # the first rescan: maps + the baseline later rescans are diffed against
        else:
            ds.create_iommu_device_map()  # :91
            ds.create_vgpu_id_map()       # :93
        specs = ds.create_device_plugins()
        if args.dump:
            sys.stdout.write(canonical_dump(ds.maps).decode("latin-1"))
        if args.plugins:
            json.dump([{"key": s.key, "device_name": s.device_name, "resource_name": s.resource_name,
                        "socket_path": s.socket_path, "env_key": s.env_key, "vgpu": s.vgpu, "devs": s.devs}
                       for s in specs], sys.stdout, indent=1)
            sys.stdout.write("\n")
        if args.once:
            return 0
        from . import dpapi, serve
        sockdir = args.socket_dir or dpapi.DEVICE_PLUGIN_PATH
        reval = serve.BatchRevalidator(ds.ctx.scan_pci, args.base_path)
        plugins = serve.plugins_from_specs(specs, ds.maps, reval, socket_dir=sockdir, base_path=args.base_path,
                                           root_path=args.root_path, vgpu_base_path=args.vgpu_base_path)
        watchers, started = [], []
        for p in plugins:                 # createDevicePlugins :131-137, :158-165: a failed start is logged, the rest go on
            try:
                p.start()
                started.append(p)
                w = serve.DeviceNodeWatcher(p)   # device nodes (or mdev nodes) + the plugin socket
                w.start()
                watchers.append(w)
            except Exception as e:        # noqa: BLE001
                print("kvgpu: error starting the %s device plugin: %s" % (p.device_name, e), file=sys.stderr)
        feed = None
        if args.rediscover_period > 0:
            live = {(s.vgpu, s.key): p for s, p in zip(specs, plugins) if p in started}
            feed = serve.RediscoveryFeed(ds, live, args.rediscover_period, revalidate=reval, socket_dir=sockdir,
                                         base_path=args.base_path, root_path=args.root_path,
                                         vgpu_base_path=args.vgpu_base_path)
            feed.watchers = {k: w for k, w in zip(live, watchers)}
            feed.start()
        stop = threading.Event()
        for sig in (signal.SIGTERM, signal.SIGINT):
            signal.signal(sig, lambda *_: stop.set())
        stop.wait()                        # <-stop (:166)
        if feed is not None:
            feed.stop()                    # stops every watcher the feed holds
            started, watchers = list(feed.plugins.values()), []
        for w in watchers:
            w.stop()
        for p in started:
            p.stop()
        return 0
    finally:
        ds.close()


if __name__ == "__main__":
    sys.exit(main())
