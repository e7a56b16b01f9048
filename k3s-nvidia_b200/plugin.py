"""The device-plugin host: Register / ListAndWatch / Allocate / GetPreferredAllocation over a unix
socket, on top of the C ABI (libb200probe.so).

Mirrors the plugin that /root/reference/README.md:116 installs (`helm upgrade --install nvdp
nvdp/nvidia-device-plugin ... --values values.yaml`) as configured by /root/reference/values.yaml:
resource ``nvidia.com/gpu`` (:17), 4 time-sliced replicas per GPU (:18), no rename (:14), requests
for more than one replica allowed (:15), MIG off (:11).  Upstream behaviour is [RECALLED] (the chart
is un-pinned and un-vendored; SURVEY.md §3.1-3.3, §8a rows a6-a9):
  - advertised IDs ``<GPU-UUID>::<replica>``; Allocate strips the suffix, dedupes, and returns
    ``NVIDIA_VISIBLE_DEVICES=<uuid[,uuid…]>`` (envvar list strategy, uuid ID strategy);
  - ``Device.health`` is the PASSIVE verdict only (XID/ECC event loop), bit-exact with the oracle;
    active-probe outcomes go to NFD labels (labels.py) that gate scheduling — never into health,
    or parity would break the first time a probe fails on a GPU that threw no XID;
  - ListAndWatch re-sends the complete list on every change; there is no path back to Healthy;
  - kubelet restart (socket re-created) => re-serve and re-Register.

The Go/cgo host `north_star` asks for cannot be compiled here (no Go toolchain); its source is in
host/go/ for a maintainer, and this Python host is the one that runs and is tested.
"""
from __future__ import annotations

import logging
import os
import threading
import time
from concurrent import futures
from dataclasses import dataclass
from typing import Dict, Iterable, List, Optional

import grpc

from . import api
from .config import DEFAULT_RESOURCE, PluginConfig, annotate, has_replica, strip_replica

log = logging.getLogger("b200probe.plugin")

ENV_VISIBLE_DEVICES = "NVIDIA_VISIBLE_DEVICES"


@dataclass
class AdvertisedDevice:
    id: str            # annotated ID kubelet sees
    uuid: str          # physical GPU
    index: int         # NVML index
    numa_node: int
    health: str = api.HEALTHY


class AllocationError(Exception):
    pass


def build_devices(infos, cfg: PluginConfig, resource: str = DEFAULT_RESOURCE) -> List[AdvertisedDevice]:
    """Physical GPUs -> advertised devices (replica expansion of values.yaml:16-18)."""
    replicas = cfg.replicas(resource)
    out = []
    for d in infos:
        if cfg.mig_strategy == "none" or d.mig_enabled <= 0:
            ids = [d.uuid] if replicas <= 1 else [annotate(d.uuid, r) for r in range(replicas)]
            out.extend(AdvertisedDevice(i, d.uuid, d.index, d.numa_node) for i in ids)
        # MIG strategies single/mixed are outside this path (values.yaml:11 selects "none")
    return out


def distributed_alloc(all_ids: Iterable[str], available: List[str], required: List[str], size: int) -> List[str]:
    """Preferred allocation for replicated devices [RECALLED upstream distributedAlloc]: spread
    the request over the physical GPUs with the fewest replicas already handed out.  Upstream
    sorts with an unstable sort; ties here break by the order of ``available`` (deterministic)."""
    avail_set, req_set = set(available), set(required)
    known = set(all_ids)
    candidates = [i for i in available if i in known and i not in req_set]
    needed = size - len([r for r in required if r in known])
    if needed < 0:
        needed = 0
    if len(candidates) < needed:
        raise AllocationError("not enough available devices to satisfy allocation")
    total: Dict[str, int] = {}
    free: Dict[str, int] = {}
    for c in candidates:
        free[strip_replica(c)] = free.get(strip_replica(c), 0) + 1
    for d in known:
        u = strip_replica(d)
        if u in free:
            total[u] = total.get(u, 0) + 1
    picked: List[str] = []
    for _ in range(needed):
        candidates.sort(key=lambda c: total[strip_replica(c)] - free[strip_replica(c)])   # stable
        c = candidates.pop(0)
        free[strip_replica(c)] -= 1
        picked.append(c)
    del avail_set
    return list(required) + picked


class DevicePlugin:
    """One plugin instance == one extended resource (``nvidia.com/gpu``)."""

    def __init__(self, probe, cfg: PluginConfig, *, resource: str = DEFAULT_RESOURCE,
                 socket_dir: str = api.DEVICE_PLUGIN_PATH, kubelet_socket: Optional[str] = None,
                 health_timeout_ms: int = 5000, disable_healthchecks: Optional[str] = None):
        self.probe = probe
        self.cfg = cfg
        self.base_resource = resource
        self.resource = cfg.resource_name(resource)
        self.socket_dir = socket_dir
        self.endpoint = "nvidia-" + self.resource.split("/", 1)[1].replace(".", "-") + ".sock"
        self.socket_path = os.path.join(socket_dir, self.endpoint)
        self.kubelet_socket = kubelet_socket or os.path.join(socket_dir, "kubelet.sock")
        self.health_timeout_ms = health_timeout_ms
        self.disable_healthchecks = os.environ.get("DP_DISABLE_HEALTHCHECKS") if disable_healthchecks is None else disable_healthchecks
        self._cv = threading.Condition()
        self._generation = 0
        self._stop = threading.Event()
        self._server: Optional[grpc.Server] = None
        self._threads: List[threading.Thread] = []
        self.devices: List[AdvertisedDevice] = []
        self.registrations = 0
        self.refresh_devices()

    # ---- device list --------------------------------------------------------------------------
    def refresh_devices(self) -> None:
        infos = [self.probe.device_info(i) for i in range(self.probe.device_count())]
        with self._cv:
            self.devices = build_devices(infos, self.cfg, self.base_resource)
            self._generation += 1
            self._cv.notify_all()

    def api_devices(self) -> List["api.Device"]:
        out = []
        for d in self.devices:
            dev = api.Device(ID=d.id, health=d.health)
            if d.numa_node >= 0:
                dev.topology.nodes.add(ID=d.numa_node)
            out.append(dev)
        return out

    def mark_unhealthy_mask(self, mask: int) -> bool:
        """Bit i of mask = physical GPU with NVML index i.  Every replica of that GPU turns
        Unhealthy (health is a property of the physical device).  Returns True on a change."""
        changed = False
        with self._cv:
            for d in self.devices:
                if (mask >> d.index) & 1 and d.health != api.UNHEALTHY:
                    d.health = api.UNHEALTHY
                    changed = True
                    log.info("'%s' device marked unhealthy: %s", self.resource, d.id)
            if changed:
                self._generation += 1
                self._cv.notify_all()
        return changed

    # ---- gRPC: DevicePlugin service --------------------------------------------------------------
    def GetDevicePluginOptions(self, request, context):  # noqa: N802
        return api.DevicePluginOptions(pre_start_required=False, get_preferred_allocation_available=True)

    def ListAndWatch(self, request, context):  # noqa: N802
        with self._cv:
            gen = self._generation
            resp = api.ListAndWatchResponse(devices=self.api_devices())
        yield resp
        while not self._stop.is_set() and context.is_active():
            with self._cv:
                self._cv.wait_for(lambda: self._generation != gen or self._stop.is_set(), timeout=0.2)
                if self._generation == gen:
                    continue
                gen = self._generation
                resp = api.ListAndWatchResponse(devices=self.api_devices())
            yield resp

    def GetPreferredAllocation(self, request, context):  # noqa: N802
        resp = api.PreferredAllocationResponse()
        all_ids = [d.id for d in self.devices]
        for req in request.container_requests:
            try:
                if self.cfg.is_shared(self.base_resource):
                    ids = distributed_alloc(all_ids, list(req.available_deviceIDs), list(req.must_include_deviceIDs), req.allocation_size)
                else:
                    # Unshared: upstream packs by NVLink topology; behind NVSwitch every pair is
                    # equidistant, so required-first then availability order is an equivalent choice.
                    req_ids = list(req.must_include_deviceIDs)
                    rest = [i for i in req.available_deviceIDs if i not in set(req_ids)]
                    if len(req_ids) + len(rest) < req.allocation_size:
                        raise AllocationError("not enough available devices to satisfy allocation")
                    ids = (req_ids + rest)[: max(req.allocation_size, len(req_ids))]
            except AllocationError as e:
                context.abort(grpc.StatusCode.UNKNOWN, f"error getting list of preferred allocation devices: {e}")
            resp.container_responses.add(deviceIDs=ids)
        return resp

    def allocate_container(self, ids: List[str]) -> "api.ContainerAllocateResponse":
        known = {d.id for d in self.devices}
        if self.cfg.is_shared(self.base_resource) and self.cfg.time_slicing.fail_requests_greater_than_one and len(ids) > 1:
            raise AllocationError(f"request for '{self.resource}: {len(ids)}' too large: maximum request size for shared resources is 1")
        for i in ids:
            if i not in known:
                raise AllocationError(f"invalid allocation request for '{self.resource}': unknown device: {i}")
        uuids: List[str] = []
        for i in ids:
            u = strip_replica(i) if has_replica(i) else i
            if u not in uuids:
                uuids.append(u)
        if self.cfg.device_id_strategy == "index":
            by_uuid = {d.uuid: d.index for d in self.devices}
            visible = [str(by_uuid[u]) for u in uuids]
        else:
            visible = uuids
        resp = api.ContainerAllocateResponse()
        resp.envs[ENV_VISIBLE_DEVICES] = ",".join(visible)
        return resp

    def Allocate(self, request, context):  # noqa: N802
        resp = api.AllocateResponse()
        for req in request.container_requests:
            try:
                resp.container_responses.append(self.allocate_container(list(req.devices_ids)))
            except AllocationError as e:
                context.abort(grpc.StatusCode.UNKNOWN, str(e))
        return resp

    def PreStartContainer(self, request, context):  # noqa: N802
        return api.PreStartContainerResponse()

    # ---- lifecycle ---------------------------------------------------------------------------------
    def serve(self) -> None:
        os.makedirs(self.socket_dir, exist_ok=True)
        if os.path.exists(self.socket_path):
            os.unlink(self.socket_path)
        self._server = grpc.server(futures.ThreadPoolExecutor(max_workers=8))
        api.add_servicer(self._server, "DevicePlugin", self)
        self._server.add_insecure_port("unix://" + self.socket_path)
        self._server.start()

    def register(self, timeout: float = 5.0) -> None:
        with grpc.insecure_channel("unix://" + self.kubelet_socket) as ch:
            grpc.channel_ready_future(ch).result(timeout=timeout)
            stub = api.RegistrationStub(ch)
            stub.Register(api.RegisterRequest(
                version=api.VERSION, endpoint=self.endpoint, resource_name=self.resource,
                options=api.DevicePluginOptions(pre_start_required=False, get_preferred_allocation_available=True)),
                timeout=timeout)
        self.registrations += 1
        log.info("Registered device plugin for '%s' with Kubelet", self.resource)

    def _health_loop(self) -> None:
        at_open = self.probe.health_open(self.disable_healthchecks or "")
        if at_open:
            self.mark_unhealthy_mask(at_open)
        while not self._stop.is_set():
            ev = self.probe.health_wait(self.health_timeout_ms)
            if ev.newly_unhealthy:
                log.info("XidCriticalError: Xid=%d on device %d; marking device as unhealthy", ev.event_data, ev.device_index)
                self.mark_unhealthy_mask(ev.newly_unhealthy)
            if ev.rc_wait not in (0, 10):       # neither SUCCESS nor TIMEOUT: a wait that keeps failing returns at once — back off, do not spin
                self._stop.wait(2.0)

    def _kubelet_watch(self, period: float) -> None:
        """kubelet restart re-creates its socket: serve again and re-Register."""
        def ident():
            try:
                st = os.stat(self.kubelet_socket)
                return (st.st_ino, st.st_ctime_ns)
            except FileNotFoundError:
                return None
        last = ident()
        while not self._stop.wait(period):
            cur = ident()
            if cur is not None and cur != last:
                log.info("inotify: %s created, restarting.", self.kubelet_socket)
                try:
                    if self._server:
                        # gRPC unlinks the socket path when the old server's teardown completes, which can be after
                        # serve() has bound the new one: wait for it, or the re-registered endpoint may vanish
                        self._server.stop(0).wait()
                    self.serve()
                    self.register()
                except Exception as e:  # noqa: BLE001
                    log.error("restart after kubelet restart failed: %s", e)
                    cur = last
            if cur is not None:
                last = cur

    def start(self, *, watch_kubelet_period: float = 1.0, health: bool = True) -> None:
        self.serve()
        self.register()
        if health:
            t = threading.Thread(target=self._health_loop, name="b200probe-health", daemon=True)
            t.start()
            self._threads.append(t)
        if watch_kubelet_period > 0:
            t = threading.Thread(target=self._kubelet_watch, args=(watch_kubelet_period,), name="b200probe-kubelet-watch", daemon=True)
            t.start()
            self._threads.append(t)

    def stop(self) -> None:
        self._stop.set()
        with self._cv:
            self._cv.notify_all()
        if self._server:
            self._server.stop(0.5)
        for t in self._threads:
            t.join(timeout=max(2.0, self.health_timeout_ms / 1000.0 + 1.0))
        self.probe.health_close()
        if os.path.exists(self.socket_path):
            try:
                os.unlink(self.socket_path)
            except OSError:
                pass


def main(argv=None) -> int:
    """`python -m k3s_nvidia_b200.plugin --config-file /config/config.yaml` — the container entry
    point that replaces the upstream plugin binary inside the nvdp DaemonSet."""
    import argparse

    from .config import parse_plugin_config
    from .labels import ActiveProbeRunner
    from .probe import Probe

    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--config-file", default=os.environ.get("CONFIG_FILE", "/config/config.yaml"))
    ap.add_argument("--socket-dir", default=api.DEVICE_PLUGIN_PATH)
    ap.add_argument("--features-dir", default="/etc/kubernetes/node-feature-discovery/features.d")
    ap.add_argument("--probe-interval", type=float, default=float(os.environ.get("B200PROBE_INTERVAL_S", "600")))
    ap.add_argument("--no-active-probe", action="store_true")
    ap.add_argument("--kubelet-socket", default=None)
    ap.add_argument("--nvml-path", default=None)
    ap.add_argument("--watch-period", type=float, default=1.0)
    ap.add_argument("--health-timeout-ms", type=int, default=5000)
    ap.add_argument("--no-health", action="store_true")
    args = ap.parse_args(argv)
    logging.basicConfig(level=logging.INFO, format="%(asctime)s %(name)s %(message)s")
    with open(args.config_file) as f:
        cfg = parse_plugin_config(f.read())
    import signal

    probe = Probe(args.nvml_path)

    def make(c):
        dp = DevicePlugin(probe, c, socket_dir=args.socket_dir, kubelet_socket=args.kubelet_socket, health_timeout_ms=args.health_timeout_ms)
        dp.start(watch_kubelet_period=args.watch_period, health=not args.no_health)
        return dp

    plugin = make(cfg)
    log.info("serving '%s' on %s (%d devices)", plugin.resource, plugin.socket_path, len(plugin.devices))
    runner = None
    if not args.no_active_probe:
        runner = ActiveProbeRunner(probe, features_dir=args.features_dir, interval_s=args.probe_interval)
        runner.start()
    reload_requested = threading.Event()
    signal.signal(signal.SIGHUP, lambda *_: reload_requested.set())

    def _term(*_):
        raise KeyboardInterrupt

    signal.signal(signal.SIGTERM, _term)
    try:
        while True:
            if not reload_requested.wait(1.0):
                continue
            reload_requested.clear()
            # SIGHUP: the chart's config-manager sidecar rewrote the config file [RECALLED] (same rule as host/cpp/main.cpp)
            try:
                with open(args.config_file) as f:
                    fresh = parse_plugin_config(f.read())
            except (OSError, ValueError) as e:
                log.error("reload of %s rejected, keeping the running configuration: %s", args.config_file, e)
                continue
            plugin.stop()
            plugin = make(fresh)
            log.info("reloaded %s: serving '%s' (%d devices)", args.config_file, plugin.resource, len(plugin.devices))
    except KeyboardInterrupt:
        pass
    finally:
        if runner:
            runner.stop()
        plugin.stop()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
