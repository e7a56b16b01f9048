"""The device-plugin host against a fake kubelet over real unix-domain gRPC (SURVEY.md §4)."""
import ctypes as C
import json
import os
import threading
import time
from concurrent import futures

import grpc
import pytest

import _oracle
from k3s_nvidia_b200 import api
from k3s_nvidia_b200 import config as cfgmod
from k3s_nvidia_b200.plugin import DevicePlugin, distributed_alloc

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
CFG = cfgmod.parse_helm_values(G["reference_inputs"]["values.yaml"]["text"]).default


class FakeKubelet:
    """v1beta1.Registration server on <dir>/kubelet.sock; records RegisterRequests."""

    def __init__(self, d):
        self.dir = d
        self.sock = os.path.join(d, "kubelet.sock")
        self.requests = []
        self.event = threading.Event()
        self.server = None

    def Register(self, request, context):  # noqa: N802
        self.requests.append(request)
        self.event.set()
        return api.Empty()

    def start(self):
        if os.path.exists(self.sock):
            os.unlink(self.sock)
        self.server = grpc.server(futures.ThreadPoolExecutor(max_workers=2))
        api.add_servicer(self.server, "Registration", self)
        self.server.add_insecure_port("unix://" + self.sock)
        self.server.start()

    def stop(self):
        if self.server:
            self.server.stop(0).wait()         # teardown unlinks the socket path: finish it before a restart binds it again

    def plugin_channel(self):
        req = self.requests[-1]
        return grpc.insecure_channel("unix://" + os.path.join(self.dir, req.endpoint))


@pytest.fixture
def stack(sock_dir, monkeypatch):
    from k3s_nvidia_b200.probe import Probe

    monkeypatch.setenv("MOCK_NVML_DEVICES", "2")
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    probe = Probe(_oracle.MOCK_NVML)
    plugin = DevicePlugin(probe, CFG, socket_dir=d, health_timeout_ms=5, disable_healthchecks="")
    plugin.start(watch_kubelet_period=0.05)
    assert kubelet.event.wait(5)
    mock = C.CDLL(_oracle.MOCK_NVML)
    mock.mock_nvml_push.argtypes = [C.c_int, C.c_int, C.c_ulonglong]
    yield kubelet, plugin, mock
    plugin.stop()
    probe.close()
    kubelet.stop()


U0 = "GPU-b2000000-0000-4000-8000-000000000000"
U1 = "GPU-b2000000-0000-4000-8000-000000000001"


def test_register_request(stack):
    kubelet, plugin, _ = stack
    r = kubelet.requests[0]
    assert (r.version, r.resource_name, r.endpoint) == ("v1beta1", "nvidia.com/gpu", "nvidia-gpu.sock")
    assert r.options.get_preferred_allocation_available is True and r.options.pre_start_required is False


def test_options_and_list(stack):
    kubelet, plugin, _ = stack
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        opts = stub.GetDevicePluginOptions(api.Empty())
        assert opts.get_preferred_allocation_available and not opts.pre_start_required
        stream = stub.ListAndWatch(api.Empty())
        first = next(stream)
        ids = [d.ID for d in first.devices]
        assert ids == [f"{U0}::{r}" for r in range(4)] + [f"{U1}::{r}" for r in range(4)]     # 2 GPUs x replicas 4
        assert {d.health for d in first.devices} == {"Healthy"}
        stream.cancel()


def test_xid_turns_every_replica_of_that_gpu_unhealthy_and_resends_full_list(stack):
    kubelet, plugin, mock = stack
    with kubelet.plugin_channel() as ch:
        stream = api.DevicePluginStub(ch).ListAndWatch(api.Empty())
        next(stream)
        mock.mock_nvml_push(0, 1, 79)            # critical XID on GPU 1
        upd = next(stream)
        assert len(upd.devices) == 8             # the COMPLETE list, not a delta
        health = {d.ID: d.health for d in upd.devices}
        assert all(health[f"{U1}::{r}"] == "Unhealthy" for r in range(4))
        assert all(health[f"{U0}::{r}"] == "Healthy" for r in range(4))
        mock.mock_nvml_push(0, 0, 13)            # application XID: skipped, no update
        mock.mock_nvml_push(0, 0, 48)            # then a critical one on GPU 0
        upd = next(stream)
        assert {d.health for d in upd.devices} == {"Unhealthy"}
        stream.cancel()


def test_allocate_strips_replicas_and_dedupes(stack):
    kubelet, plugin, _ = stack
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        # nvidia-smi.yaml / jellyfin.yaml: one unit of nvidia.com/gpu
        resp = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::2"])]))
        assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
        # failRequestsGreaterThanOne: false (values.yaml:15) -> two replicas allowed; same GPU collapses
        resp = stub.Allocate(api.AllocateRequest(container_requests=[
            api.ContainerAllocateRequest(devices_ids=[f"{U0}::0", f"{U0}::3"]),
            api.ContainerAllocateRequest(devices_ids=[f"{U1}::1", f"{U0}::1"])]))
        assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
        assert dict(resp.container_responses[1].envs) == {"NVIDIA_VISIBLE_DEVICES": f"{U1},{U0}"}
        assert len(resp.container_responses[0].mounts) == 0 and len(resp.container_responses[0].devices) == 0
        with pytest.raises(grpc.RpcError) as e:
            stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=["GPU-nope::0"])]))
        assert "unknown device" in e.value.details()
        assert stub.PreStartContainer(api.PreStartContainerRequest(devices_ids=[f"{U0}::0"])) is not None


def test_fail_requests_greater_than_one(stack, tmp_path):
    kubelet, plugin, _ = stack
    strict = cfgmod.parse_plugin_config(
        "version: v1\nsharing:\n  timeSlicing:\n    failRequestsGreaterThanOne: true\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 4\n")
    plugin.cfg = strict
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        with pytest.raises(grpc.RpcError) as e:
            stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::0", f"{U1}::0"])]))
        assert "maximum request size for shared resources is 1" in e.value.details()
        ok = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U1}::0"])]))
        assert dict(ok.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U1}
    plugin.cfg = CFG


def test_preferred_allocation_spreads_replicas_across_gpus(stack):
    kubelet, plugin, _ = stack
    all_ids = [d.id for d in plugin.devices]
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
            api.ContainerPreferredAllocationRequest(available_deviceIDs=all_ids, allocation_size=2)]))
        got = list(resp.container_responses[0].deviceIDs)
        assert {cfgmod.strip_replica(i) for i in got} == {U0, U1}
        # GPU0 already has 3 replicas out: the next one must come from GPU1
        avail = [f"{U0}::3"] + [f"{U1}::{r}" for r in range(4)]
        resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
            api.ContainerPreferredAllocationRequest(available_deviceIDs=avail, allocation_size=1)]))
        assert cfgmod.strip_replica(resp.container_responses[0].deviceIDs[0]) == U1
        with pytest.raises(grpc.RpcError):
            stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                api.ContainerPreferredAllocationRequest(available_deviceIDs=all_ids[:1], allocation_size=3)]))


def test_distributed_alloc_unit():
    ids = [f"A::{r}" for r in range(4)] + [f"B::{r}" for r in range(4)]
    got = distributed_alloc(ids, ids, [], 4)
    assert sorted(cfgmod.strip_replica(i) for i in got) == ["A", "A", "B", "B"]
    got = distributed_alloc(ids, ids, ["A::0"], 3)
    assert got[0] == "A::0" and len(got) == 3
    assert sorted(cfgmod.strip_replica(i) for i in got) == ["A", "A", "B"] or sorted(cfgmod.strip_replica(i) for i in got) == ["A", "B", "B"]


def test_kubelet_restart_triggers_reregistration(stack):
    kubelet, plugin, _ = stack
    n0 = len(kubelet.requests)
    kubelet.stop()
    time.sleep(0.2)
    kubelet.event.clear()
    kubelet.start()                              # socket re-created
    assert kubelet.event.wait(5), "plugin did not re-register after kubelet restart"
    assert len(kubelet.requests) == n0 + 1
    with kubelet.plugin_channel() as ch:
        first = next(api.DevicePluginStub(ch).ListAndWatch(api.Empty()))
        assert len(first.devices) == 8


def test_wire_format_field_numbers():
    """Spot-check the hand-built descriptor against the v1beta1 wire layout [RECALLED]."""
    d = api.Device(ID="x", health="Healthy")
    assert d.SerializeToString() == b"\x0a\x01x\x12\x07Healthy"
    r = api.RegisterRequest(version="v1beta1", endpoint="e", resource_name="nvidia.com/gpu")
    assert r.SerializeToString() == b"\x0a\x07v1beta1\x12\x01e\x1a\x0envidia.com/gpu"
    a = api.ContainerAllocateResponse()
    a.envs["K"] = "V"
    assert a.SerializeToString() == b"\x0a\x06\x0a\x01K\x12\x01V"
    c = api.ContainerPreferredAllocationRequest(available_deviceIDs=["a"], must_include_deviceIDs=["b"], allocation_size=3)
    assert c.SerializeToString() == b"\x0a\x01a\x12\x01b\x18\x03"
