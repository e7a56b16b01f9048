"""The NATIVE device-plugin host (host/cpp/b200-device-plugin: hand-written HTTP/2 + HPACK + gRPC framing +
protobuf wire format above the C ABI) against a fake kubelet over real unix-domain gRPC.  Same cases as
tests/test_plugin.py runs against the Python host: the two hosts must be indistinguishable to kubelet.
The peer here is grpcio (gRPC C-core), which Huffman-codes and indexes its headers and is strict about
HTTP/2 framing, so these tests also cover the transport."""
import json
import os
import signal
import subprocess
import sys
import time

import grpc
import pytest

import _oracle
from k3s_nvidia_b200 import api
from k3s_nvidia_b200 import config as cfgmod
from test_plugin import FakeKubelet, U0, U1

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.environ.get("B200_NATIVE_BIN") or os.path.join(ROOT, "host", "cpp", "build", "b200-device-plugin")
G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
VALUES = cfgmod.parse_helm_values(G["reference_inputs"]["values.yaml"]["text"])


@pytest.fixture(scope="module", autouse=True)
def _binary():
    if not os.path.exists(BIN):
        subprocess.run(["make", "-C", os.path.join(ROOT, "host", "cpp")], check=True, capture_output=True)


class Daemon:
    CMD = None          # None = the native binary; PyDaemon runs the Python twin with the same flags

    def __init__(self, d, config_text, extra_env=None, args=()):
        self.dir = d
        self.events = os.path.join(d, "events.txt")
        open(self.events, "w").close()
        cfg = os.path.join(d, "config.yaml")
        with open(cfg, "w") as f:
            f.write(config_text)
        env = dict(os.environ, MOCK_NVML_DEVICES="2", MOCK_NVML_EVENT_FILE=self.events)
        env.update(extra_env or {})
        self.log = open(os.path.join(d, "daemon.log"), "w")
        self.proc = subprocess.Popen([*(self.CMD or [BIN]), "--config-file", cfg, "--socket-dir", d, "--nvml-path", _oracle.MOCK_NVML, "--no-active-probe",
                                      "--watch-period", "0.05", "--health-timeout-ms", "5", *args], env=env, stderr=self.log)

    def wait_serving(self, timeout=10.0):
        """Registered AND past start(): the fake kubelet's handler sets its event before the response is on the
        wire, so a test that stops the kubelet right away would cut the daemon's initial Register short."""
        t_end = time.time() + timeout
        while time.time() < t_end:
            if " serving '" in self.logtext():
                return True
            if self.proc.poll() is not None:
                return False
            time.sleep(0.02)
        return False

    def push(self, kind, dev, data):
        with open(self.events, "a") as f:
            f.write(f"{kind} {dev} {data}\n")

    def stop(self):
        if self.proc.poll() is None:
            self.proc.send_signal(signal.SIGTERM)
            try:
                self.proc.wait(10)
            except subprocess.TimeoutExpired:
                self.proc.kill()
        self.log.close()
        text = self.logtext()                # sanitizer builds (make -C host/cpp asan tsan) report on stderr
        assert "Sanitizer" not in text and "runtime error" not in text, text[-4000:]

    def logtext(self):
        return open(os.path.join(self.dir, "daemon.log")).read()


class PyDaemon(Daemon):
    import sys as _sys
    CMD = [_sys.executable, "-m", "k3s_nvidia_b200.plugin"]


@pytest.fixture(params=["native", "python"])
def both_hosts(request, sock_dir, monkeypatch):
    """The same CLI contract for both hosts: flags, log lines the tests key on, signals."""
    monkeypatch.setenv("PYTHONPATH", ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    daemon = (Daemon if request.param == "native" else PyDaemon)(d, VALUES.raw_configs["default"])
    try:
        assert kubelet.event.wait(30) and daemon.wait_serving(30), "host did not register: " + daemon.logtext()
        yield kubelet, daemon
    finally:
        daemon.stop()
        kubelet.stop()


@pytest.fixture
def stack(sock_dir):
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    daemon = Daemon(d, VALUES.raw_configs["default"])          # the config document exactly as the chart mounts it
    try:
        assert kubelet.event.wait(10) and daemon.wait_serving(), "native plugin did not register: " + daemon.logtext()
        yield kubelet, daemon
    finally:
        daemon.stop()
        kubelet.stop()


def test_register_request(stack):
    kubelet, daemon = stack
    r = kubelet.requests[0]
    assert (r.version, r.resource_name, r.endpoint) == ("v1beta1", "nvidia.com/gpu", "nvidia-gpu.sock")
    assert r.options.get_preferred_allocation_available is True and r.options.pre_start_required is False


def test_options_and_list(stack):
    kubelet, daemon = stack
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        opts = stub.GetDevicePluginOptions(api.Empty())
        assert opts.get_preferred_allocation_available and not opts.pre_start_required
        stream = stub.ListAndWatch(api.Empty())
        first = next(stream)
        assert [d.ID for d in first.devices] == [f"{U0}::{r}" for r in range(4)] + [f"{U1}::{r}" for r in range(4)]
        assert {d.health for d in first.devices} == {"Healthy"}
        stream.cancel()


def test_native_list_is_byte_identical_to_the_python_host(stack, monkeypatch):
    """Same NVML state, same config -> the serialized ListAndWatchResponse of both hosts is the same bytes."""
    from k3s_nvidia_b200.plugin import DevicePlugin
    from k3s_nvidia_b200.probe import Probe

    kubelet, daemon = stack
    with kubelet.plugin_channel() as ch:
        raw = ch.unary_stream("/v1beta1.DevicePlugin/ListAndWatch", request_serializer=lambda m: m.SerializeToString(), response_deserializer=lambda b: b)
        stream = raw(api.Empty())
        native = next(stream)
        stream.cancel()
    monkeypatch.setenv("MOCK_NVML_DEVICES", "2")
    probe = Probe(_oracle.MOCK_NVML)
    try:
        py = DevicePlugin(probe, VALUES.default, socket_dir=str(daemon.dir) + "/py")
        want = api.ListAndWatchResponse(devices=py.api_devices()).SerializeToString()
    finally:
        probe.close()
    assert native == want


def test_xid_turns_every_replica_of_that_gpu_unhealthy_and_resends_full_list(stack):
    kubelet, daemon = stack
    with kubelet.plugin_channel() as ch:
        stream = api.DevicePluginStub(ch).ListAndWatch(api.Empty())
        next(stream)
        daemon.push(0, 1, 79)                    # critical XID on GPU 1
        upd = next(stream)
        assert len(upd.devices) == 8             # the COMPLETE list, not a delta
        health = {d.ID: d.health for d in upd.devices}
        assert all(health[f"{U1}::{r}"] == "Unhealthy" for r in range(4))
        assert all(health[f"{U0}::{r}"] == "Healthy" for r in range(4))
        daemon.push(0, 0, 13)                    # application XID: skipped, no update
        daemon.push(0, 0, 48)                    # then a critical one on GPU 0
        upd = next(stream)
        assert {d.health for d in upd.devices} == {"Unhealthy"}
        stream.cancel()


def test_allocate_strips_replicas_and_dedupes(stack):
    kubelet, daemon = stack
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        resp = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::2"])]))
        assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
        resp = stub.Allocate(api.AllocateRequest(container_requests=[
            api.ContainerAllocateRequest(devices_ids=[f"{U0}::0", f"{U0}::3"]),
            api.ContainerAllocateRequest(devices_ids=[f"{U1}::1", f"{U0}::1"])]))
        assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
        assert dict(resp.container_responses[1].envs) == {"NVIDIA_VISIBLE_DEVICES": f"{U1},{U0}"}
        assert len(resp.container_responses[0].mounts) == 0 and len(resp.container_responses[0].devices) == 0
        with pytest.raises(grpc.RpcError) as e:
            stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=["GPU-nope::0"])]))
        assert e.value.code() == grpc.StatusCode.UNKNOWN
        assert e.value.details() == "invalid allocation request for 'nvidia.com/gpu': unknown device: GPU-nope::0"
        assert stub.PreStartContainer(api.PreStartContainerRequest(devices_ids=[f"{U0}::0"])) is not None
        with pytest.raises(grpc.RpcError) as e:
            ch.unary_unary("/v1beta1.DevicePlugin/NoSuchMethod", request_serializer=lambda m: m.SerializeToString(), response_deserializer=lambda b: b)(api.Empty())
        assert e.value.code() == grpc.StatusCode.UNIMPLEMENTED


def test_fail_requests_greater_than_one(sock_dir):
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    daemon = Daemon(d, "version: v1\nsharing:\n  timeSlicing:\n    failRequestsGreaterThanOne: true\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 4\n")
    try:
        assert kubelet.event.wait(10) and daemon.wait_serving(), daemon.logtext()
        with kubelet.plugin_channel() as ch:
            stub = api.DevicePluginStub(ch)
            with pytest.raises(grpc.RpcError) as e:
                stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::0", f"{U1}::0"])]))
            assert "maximum request size for shared resources is 1" in e.value.details()
            ok = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U1}::0"])]))
            assert dict(ok.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U1}
    finally:
        daemon.stop()
        kubelet.stop()


def test_preferred_allocation_spreads_replicas_across_gpus(stack):
    kubelet, daemon = stack
    all_ids = [f"{U0}::{r}" for r in range(4)] + [f"{U1}::{r}" for r in range(4)]
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
            api.ContainerPreferredAllocationRequest(available_deviceIDs=all_ids, allocation_size=2)]))
        got = list(resp.container_responses[0].deviceIDs)
        assert {cfgmod.strip_replica(i) for i in got} == {U0, U1}
        avail = [f"{U0}::3"] + [f"{U1}::{r}" for r in range(4)]
        resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
            api.ContainerPreferredAllocationRequest(available_deviceIDs=avail, allocation_size=1)]))
        assert cfgmod.strip_replica(resp.container_responses[0].deviceIDs[0]) == U1
        with pytest.raises(grpc.RpcError) as e:
            stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                api.ContainerPreferredAllocationRequest(available_deviceIDs=all_ids[:1], allocation_size=3)]))
        assert "not enough available devices" in e.value.details()


def test_preferred_allocation_matches_python_host_exactly(stack):
    """distributed_alloc is deterministic in both hosts (ties by availability order): same picks."""
    import random

    from k3s_nvidia_b200.plugin import distributed_alloc

    kubelet, daemon = stack
    all_ids = [f"{U0}::{r}" for r in range(4)] + [f"{U1}::{r}" for r in range(4)]
    rng = random.Random(11)
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        for _ in range(40):
            avail = rng.sample(all_ids, rng.randint(1, 8))
            must = rng.sample(avail, rng.randint(0, min(2, len(avail))))
            size = rng.randint(len(must), len(avail))
            resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                api.ContainerPreferredAllocationRequest(available_deviceIDs=avail, must_include_deviceIDs=must, allocation_size=size)]))
            assert list(resp.container_responses[0].deviceIDs) == distributed_alloc(all_ids, avail, must, size)


def test_kubelet_restart_triggers_reregistration(stack):
    kubelet, daemon = stack
    n0 = len(kubelet.requests)
    kubelet.stop()
    time.sleep(0.2)
    kubelet.event.clear()
    kubelet.start()                              # socket re-created
    assert kubelet.event.wait(10), "native plugin did not re-register after kubelet restart: " + daemon.logtext()
    assert len(kubelet.requests) == n0 + 1
    with kubelet.plugin_channel() as ch:
        first = next(api.DevicePluginStub(ch).ListAndWatch(api.Empty()))
        assert len(first.devices) == 8


def test_many_calls_and_concurrent_streams_on_one_connection(stack):
    """HPACK dynamic-table state and flow-control accounting must survive a long-lived connection."""
    kubelet, daemon = stack
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        streams = [stub.ListAndWatch(api.Empty()) for _ in range(3)]
        for s in streams:
            assert len(next(s).devices) == 8
        for i in range(300):
            r = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::{i % 4}"])]))
            assert dict(r.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
        daemon.push(1, 0, 0)                     # double-bit ECC on GPU 0: not an XID event -> skipped, no update
        daemon.push(0, 1, 79)
        for s in streams:
            upd = next(s)
            assert [d.health for d in upd.devices] == ["Healthy"] * 4 + ["Unhealthy"] * 4
            s.cancel()


CONFIG_CASES = [
    "version: v1\n",
    "version: v2\n",
    "",
    "version: v1\nflags:\n  migStrategy: mixed\n",
    "version: v1\nflags:\n  migStrategy: sideways\n",
    "version: v1\nflags:\n  plugin:\n    deviceIDStrategy: index\n    passDeviceSpecs: true\n",
    "version: v1\nsharing:\n  timeSlicing:\n    renameByDefault: true\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 2\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n      - name: gpu\n        replicas: 3\n        rename: gpu-shared\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 0\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: four\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: true\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - replicas: 2\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: amd.com/gpu\n      replicas: 2\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 2\n    - name: gpu\n      replicas: 3\n",
    "version: v1\nsharing:\n  timeSlicing:\n    renameByDefault: maybe\n",
    "version: v1\nsharing:\n  timeSlicing:\n    resources: 7\n",
    "# comment first\nversion: 'v1'   # quoted\nflags: {}\nsharing:\n  timeSlicing:\n    resources: []\n",
    "version: v1\nsharing:\n  timeSlicing:\n    failRequestsGreaterThanOne: yes\n    resources:\n    - {name: nvidia.com/gpu, replicas: 2}\n",
    "---\nversion: v1\nflags:\n    migStrategy: \"single\"\nsharing:\n    timeSlicing:\n        resources:\n        -   name: nvidia.com/gpu\n            replicas: 0x10\n",
]


@pytest.mark.parametrize("i", range(len(CONFIG_CASES)))
def test_config_document_parses_like_the_python_host(i, tmp_path):
    """The native YAML subset + config rules against config.py (PyYAML) on the reference document, variants
    of it and malformed documents: same fields, or an error where Python raises one."""
    text = CONFIG_CASES[i]
    path = tmp_path / "c.yaml"
    path.write_text(text)
    out = json.loads(subprocess.run([BIN, "--check-config", str(path)], capture_output=True, text=True, check=True).stdout)
    try:
        c = cfgmod.parse_plugin_config(text)
    except Exception as e:  # noqa: BLE001 (ConfigError, or what a malformed document provokes)
        assert out["ok"] is False, (text, out, e)
        return
    if not out["ok"]:
        # the native reader refuses non-empty flow collections by design: that is the only allowed asymmetry
        assert "flow collections" in out["error"], (text, out)
        return
    assert out["version"] == c.version and out["mig_strategy"] == c.mig_strategy
    assert out["device_id_strategy"] == c.device_id_strategy and out["pass_device_specs"] == c.pass_device_specs
    assert out["rename_by_default"] == c.time_slicing.rename_by_default
    assert out["fail_requests_greater_than_one"] == c.time_slicing.fail_requests_greater_than_one
    assert out["resources"] == [{"name": r.name, "replicas": r.replicas, "rename": r.rename} for r in c.time_slicing.resources]
    assert (out["resource_name"], out["replicas"], out["is_shared"]) == (c.resource_name(), c.replicas(), c.is_shared())


def test_reference_values_yaml_config_document(tmp_path):
    """/root/reference/values.yaml:9-18 exactly as shipped (committed golden copy, sha256-pinned elsewhere)."""
    path = tmp_path / "c.yaml"
    path.write_text(VALUES.raw_configs["default"])
    out = json.loads(subprocess.run([BIN, "--check-config", str(path)], capture_output=True, text=True, check=True).stdout)
    assert out == {"ok": True, "version": "v1", "mig_strategy": "none", "device_list_strategy": "envvar", "device_id_strategy": "uuid",
                   "pass_device_specs": False, "rename_by_default": False, "fail_requests_greater_than_one": False,
                   "resources": [{"name": "nvidia.com/gpu", "replicas": 4, "rename": None}], "resource_name": "nvidia.com/gpu", "replicas": 4,
                   "is_shared": True}


def test_hpack_decoder_against_libnghttp2_deflater():
    """The native HPACK decoder (static + dynamic table, Huffman) fed with header blocks produced by the
    system libnghttp2's deflater (indexing + Huffman on), one decoder across all blocks."""
    import ctypes as C
    import ctypes.util
    import random

    name = ctypes.util.find_library("nghttp2")
    if not name:
        pytest.skip("libnghttp2 not on this box")
    lib = C.CDLL(name)

    class NV(C.Structure):
        _fields_ = [("name", C.c_char_p), ("value", C.c_char_p), ("namelen", C.c_size_t), ("valuelen", C.c_size_t), ("flags", C.c_uint8)]

    lib.nghttp2_hd_deflate_new.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    lib.nghttp2_hd_deflate_hd.restype = C.c_ssize_t
    lib.nghttp2_hd_deflate_hd.argtypes = [C.c_void_p, C.c_char_p, C.c_size_t, C.POINTER(NV), C.c_size_t]
    lib.nghttp2_hd_deflate_bound.restype = C.c_size_t
    lib.nghttp2_hd_deflate_bound.argtypes = [C.c_void_p, C.POINTER(NV), C.c_size_t]
    lib.nghttp2_hd_deflate_del.argtypes = [C.c_void_p]
    defl = C.c_void_p()
    assert lib.nghttp2_hd_deflate_new(C.byref(defl), 4096) == 0
    rng = random.Random(7541)
    names = [b":method", b":path", b":scheme", b":authority", b"content-type", b"te", b"user-agent", b"grpc-timeout", b"grpc-accept-encoding",
             b"x-custom-" + bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz-") for _ in range(12)), b"accept-encoding", b"cookie"]
    values = [b"POST", b"/v1beta1.DevicePlugin/Allocate", b"/v1beta1.DevicePlugin/ListAndWatch", b"http", b"localhost", b"application/grpc",
              b"trailers", b"grpc-python/1.80.0 grpc-c/48.0.0 (linux; chttp2)", b"4999997u", b"identity, deflate, gzip", b""]
    blocks, want = [], []
    try:
        for _ in range(300):
            hs = []
            for _ in range(rng.randint(1, 9)):
                n = rng.choice(names)
                v = rng.choice(values) if rng.random() < 0.7 else bytes(rng.randrange(32, 127) for _ in range(rng.randint(0, 80)))
                hs.append((n, v))
            if rng.random() < 0.1:
                hs.append((b"x-big", bytes(rng.randrange(32, 127) for _ in range(3000))))      # forces evictions
            arr = (NV * len(hs))(*[NV(n, v, len(n), len(v), 0) for n, v in hs])
            buf = C.create_string_buffer(lib.nghttp2_hd_deflate_bound(defl, arr, len(hs)))
            n = lib.nghttp2_hd_deflate_hd(defl, buf, len(buf), arr, len(hs))
            assert n > 0
            blocks.append(buf.raw[:n].hex())
            want.append([[a.decode(), b.decode()] for a, b in hs])
    finally:
        lib.nghttp2_hd_deflate_del(defl)
    out = subprocess.run([BIN, "--hpack-decode"], input="\n".join(blocks) + "\n", capture_output=True, text=True, check=True).stdout
    got = [json.loads(line) for line in out.splitlines()]
    assert got == want
    # malformed blocks are rejected, not mis-decoded: index 0, index past the tables, truncated string, EOS inside Huffman data
    bad = ["80", "ff7f", "0005616263", "0084ffffffff"]
    out = subprocess.run([BIN, "--hpack-decode"], input="\n".join(bad) + "\n", capture_output=True, text=True, check=True).stdout
    assert [json.loads(line) for line in out.splitlines()] == [{"error": "decode failed"}] * len(bad)


def test_flow_control_large_device_list_and_large_unary_response(sock_dir):
    """16 GPUs x 128 replicas = 2048 advertised devices: the ListAndWatch message (~110 KB) and a preferred
    allocation of 1500 IDs both exceed the 65,535-byte initial HTTP/2 windows, so DATA has to be cut into
    frames and wait for the peer's WINDOW_UPDATEs."""
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    daemon = Daemon(d, "version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 128\n",
                    extra_env={"MOCK_NVML_DEVICES": "16"})
    try:
        assert kubelet.event.wait(10) and daemon.wait_serving(), daemon.logtext()
        with kubelet.plugin_channel() as ch:
            stub = api.DevicePluginStub(ch)
            first = next(stub.ListAndWatch(api.Empty()))
            ids = [x.ID for x in first.devices]
            assert len(ids) == 2048 and len(set(ids)) == 2048 and first.ByteSize() > 100_000
            assert ids[:2] == ["GPU-b2000000-0000-4000-8000-000000000000::0", "GPU-b2000000-0000-4000-8000-000000000000::1"]
            resp = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                api.ContainerPreferredAllocationRequest(available_deviceIDs=ids, allocation_size=1500)]))
            got = list(resp.container_responses[0].deviceIDs)
            assert len(got) == 1500 and len(set(got)) == 1500 and set(got) <= set(ids)
            per_gpu = {}
            for i in got:
                per_gpu[cfgmod.strip_replica(i)] = per_gpu.get(cfgmod.strip_replica(i), 0) + 1
            assert max(per_gpu.values()) - min(per_gpu.values()) <= 1          # spread evenly over the 16 GPUs
            daemon.push(0, 3, 79)
            stream = stub.ListAndWatch(api.Empty())
            seen = next(stream)
            if all(x.health == "Healthy" for x in seen.devices):
                seen = next(stream)
            assert sum(x.health == "Unhealthy" for x in seen.devices) == 128
            stream.cancel()
    finally:
        daemon.stop()
        kubelet.stop()


def test_garbage_on_the_socket_does_not_take_the_daemon_down(stack):
    import socket

    kubelet, daemon = stack
    path = os.path.join(daemon.dir, "nvidia-gpu.sock")
    payloads = [b"GET / HTTP/1.1\r\nHost: x\r\n\r\n", b"\x00" * 64, os.urandom(4096),
                b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + b"\x00\x00\x05\x01\x04\x00\x00\x00\x01" + b"\xff\xff\xff\xff\xff",      # HEADERS with a bad HPACK block
                b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + b"\xff\xff\xff\x00\x00\x00\x00\x00\x01",                                   # 16 MiB frame announced, nothing sent
                b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + b"\x00\x00\x04\x08\x00\x00\x00\x00\x00" + b"\x00\x00\x00\x00" * 1]
    for p in payloads:
        s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        s.settimeout(2)
        s.connect(path)
        try:
            s.sendall(p)
            try:
                s.recv(65536)
            except (socket.timeout, ConnectionError):
                pass
        except (BrokenPipeError, ConnectionError):
            pass
        finally:
            s.close()
    assert daemon.proc.poll() is None, daemon.logtext()
    with kubelet.plugin_channel() as ch:
        assert len(next(api.DevicePluginStub(ch).ListAndWatch(api.Empty())).devices) == 8


def test_yaml_subset_differential_against_pyyaml(tmp_path):
    """Randomly generated plugin-config documents (block style, varied indentation, quoting, comments, booleans
    in YAML 1.1 spellings, list items at the parent's indentation or deeper): the native reader must accept and
    reject exactly what config.py over PyYAML does, with the same resulting fields."""
    import random

    rng = random.Random(20260921)

    def scalar(v):
        if isinstance(v, bool):
            return rng.choice(["true", "True", "yes", "on"] if v else ["false", "False", "no", "off"])
        if isinstance(v, int):
            return rng.choice([str(v), str(v), hex(v)]) if v >= 0 else str(v)
        q = rng.random()
        return f'"{v}"' if q < 0.25 else f"'{v}'" if q < 0.5 else v

    def comment():
        return rng.choice(["", "", "", "  # note", " #x"])

    docs = []
    for _ in range(250):
        ind = rng.choice([1, 2, 4])
        sp = " " * ind
        lines = []
        if rng.random() < 0.2:
            lines.append("# plugin configuration")
        if rng.random() < 0.15:
            lines.append("---")
        version = rng.choice(["v1"] * 8 + ["v2", "1"])
        lines.append(f"version: {scalar(version)}{comment()}")
        if rng.random() < 0.6:
            lines.append("flags:" + comment())
            if rng.random() < 0.8:
                lines.append(f"{sp}migStrategy: {scalar(rng.choice(['none', 'none', 'single', 'mixed', 'both']))}")
            if rng.random() < 0.4:
                lines.append(f"{sp}plugin:")
                lines.append(f"{sp}{sp}deviceIDStrategy: {scalar(rng.choice(['uuid', 'index', 'serial']))}")
                if rng.random() < 0.5:
                    lines.append(f"{sp}{sp}passDeviceSpecs: {scalar(rng.random() < 0.5)}")
        if rng.random() < 0.85:
            lines.append("sharing:")
            lines.append(f"{sp}timeSlicing:")
            if rng.random() < 0.5:
                lines.append(f"{sp}{sp}renameByDefault: {scalar(rng.random() < 0.5) if rng.random() < 0.9 else 'perhaps'}")
            if rng.random() < 0.5:
                lines.append(f"{sp}{sp}failRequestsGreaterThanOne: {scalar(rng.random() < 0.5)}")
            if rng.random() < 0.9:
                lines.append(f"{sp}{sp}resources:" + comment())
                item_ind = sp * 2 + (sp if rng.random() < 0.5 else "")
                for _ in range(rng.randint(0, 3)):
                    name = rng.choice(["nvidia.com/gpu", "gpu", "nvidia.com/mig-1g.10gb", "amd.com/gpu", "nvidia.com/" + "x" * 60])
                    reps = rng.choice([1, 2, 4, 8, 0, -1, "four", True])
                    dash_gap = " " * rng.choice([1, 1, 3])
                    fields = [("name", scalar(name)), ("replicas", scalar(reps))]
                    if rng.random() < 0.3:
                        fields.append(("rename", scalar(rng.choice(["gpu-shared", "nvidia.com/gpu.shared"]))))
                    if rng.random() < 0.2:
                        fields = fields[1:]            # missing name
                    rng.shuffle(fields)
                    lines.append(f"{item_ind}-{dash_gap}{fields[0][0]}: {fields[0][1]}{comment()}")
                    for k, v in fields[1:]:
                        lines.append(f"{item_ind} {dash_gap}{k}: {v}")
        docs.append("\n".join(lines) + ("\n" if rng.random() < 0.9 else ""))

    agree_ok = agree_err = 0
    for i, text in enumerate(docs):
        path = tmp_path / f"c{i}.yaml"
        path.write_text(text)
        out = json.loads(subprocess.run([BIN, "--check-config", str(path)], capture_output=True, text=True, check=True).stdout)
        try:
            c = cfgmod.parse_plugin_config(text)
        except Exception:  # noqa: BLE001
            assert out["ok"] is False, (text, out)
            agree_err += 1
            continue
        assert out["ok"] is True, (text, out)
        assert (out["version"], out["mig_strategy"], out["device_id_strategy"], out["pass_device_specs"]) == \
            (c.version, c.mig_strategy, c.device_id_strategy, c.pass_device_specs), text
        assert out["rename_by_default"] == c.time_slicing.rename_by_default and out["fail_requests_greater_than_one"] == c.time_slicing.fail_requests_greater_than_one
        assert out["resources"] == [{"name": r.name, "replicas": r.replicas, "rename": r.rename} for r in c.time_slicing.resources], text
        agree_ok += 1
    assert agree_ok > 30 and agree_err > 30, (agree_ok, agree_err)       # the generator exercises both outcomes


def _kube_schedule_and_allocate(pod_spec, node_labels, stub, advertised, in_use):
    """What scheduler + kubelet do with a pod on one node, reduced to the device-plugin path: nodeSelector
    against the node's labels, count of free units of the extended resource, GetPreferredAllocation, Allocate."""
    for k, v in (pod_spec.get("nodeSelector") or {}).items():
        if node_labels.get(k) != v:
            return None, f"node(s) didn't match Pod's node affinity/selector ({k}={node_labels.get(k)!r}, wants {v!r})"
    want = int(pod_spec["containers"][0]["resources"]["limits"]["nvidia.com/gpu"])
    free = [d.ID for d in advertised if d.health == "Healthy" and d.ID not in in_use]
    if len(free) < want:
        return None, "Insufficient nvidia.com/gpu"
    pref = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
        api.ContainerPreferredAllocationRequest(available_deviceIDs=free, allocation_size=want)]))
    ids = list(pref.container_responses[0].deviceIDs)
    resp = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=ids)]))
    in_use.update(ids)
    return (ids, dict(resp.container_responses[0].envs)), None


def test_config5_jellyfin_is_scheduled_onto_a_probe_healthy_node_via_allocate(stack, tmp_path):
    """BASELINE config 5: the reference's jellyfin Deployment (/root/reference/jellyfin.yaml, golden copy) with
    deploy/jellyfin-gated.patch.yaml merged in lands on the node only while the probe's gate label is true, and
    its container gets NVIDIA_VISIBLE_DEVICES=<uuid> from Allocate; four replicas fit one GPU (values.yaml:18)."""
    import yaml

    from k3s_nvidia_b200 import labels as L

    kubelet, daemon = stack
    docs = list(yaml.safe_load_all(G["reference_inputs"]["jellyfin.yaml"]["text"]))
    deployment = next(d for d in docs if d["kind"] == "Deployment")
    patch = yaml.safe_load(open(os.path.join(ROOT, "deploy", "jellyfin-gated.patch.yaml")))
    pod = dict(deployment["spec"]["template"]["spec"])
    pod.update(patch["spec"]["template"]["spec"])                     # strategic merge of the one added key
    assert pod["runtimeClassName"] == "nvidia" and pod["nodeSelector"] == {"nvidia.com/b200probe.healthy": "true"}

    def node_labels(healthy):
        lab = {"nvidia.com/b200probe.hbm-healthy": "true" if healthy else "false", "nvidia.com/b200probe.gemm-healthy": "true"}
        lab.update(L.gate_label(lab))
        path = L.write_feature_file(lab, str(tmp_path / "features.d"))
        return {**L.parse_feature_file(open(path).read()), "nvidia.com/gpu.present": "true"}     # what NFD turns the file into

    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        stream = stub.ListAndWatch(api.Empty())
        advertised = list(next(stream).devices)
        in_use = set()
        got, why = _kube_schedule_and_allocate(pod, node_labels(False), stub, advertised, in_use)
        assert got is None and "didn't match" in why                  # probe failed: the pod stays Pending
        got, why = _kube_schedule_and_allocate(pod, node_labels(True), stub, advertised, in_use)
        assert why is None
        ids, envs = got
        assert len(ids) == 1 and ids[0].split("::")[0] in (U0, U1) and envs == {"NVIDIA_VISIBLE_DEVICES": ids[0].split("::")[0]}
        # 2 GPUs x 4 replicas: seven more single-GPU pods fit, spread 4 + 4 over the two GPUs; the ninth is refused
        for _ in range(7):
            got, why = _kube_schedule_and_allocate(pod, node_labels(True), stub, advertised, in_use)
            assert why is None
        per_gpu = {}
        for i in in_use:
            per_gpu[i.split("::")[0]] = per_gpu.get(i.split("::")[0], 0) + 1
        assert per_gpu == {U0: 4, U1: 4}
        assert _kube_schedule_and_allocate(pod, node_labels(True), stub, advertised, in_use) == (None, "Insufficient nvidia.com/gpu")
        # an XID on GPU 1 takes its four units out of the schedulable pool (ListAndWatch update)
        daemon.push(0, 1, 79)
        advertised = list(next(stream).devices)
        assert sum(d.health == "Healthy" for d in advertised) == 4
        stream.cancel()


def test_limits_are_enforced_without_hurting_well_behaved_clients(stack):
    """A header block that never ends and a client that opens more streams than SETTINGS allows are cut off
    (GOAWAY), and the daemon keeps serving others."""
    import socket
    import struct

    kubelet, daemon = stack
    path = os.path.join(daemon.dir, "nvidia-gpu.sock")

    def frame(t, flags, stream, payload=b""):
        return struct.pack(">I", len(payload))[1:] + bytes([t, flags]) + struct.pack(">I", stream) + payload

    def talk(data):
        s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        s.settimeout(3)
        s.connect(path)
        got, cut = b"", False
        try:
            s.sendall(data)
        except (ConnectionError, BrokenPipeError):
            cut = True                               # the server hung up mid-send: its GOAWAY may still be in our receive queue
        try:
            while True:
                chunk = s.recv(65536)
                if not chunk:
                    cut = True
                    break
                got += chunk
        except ConnectionError:
            cut = True                               # a unix socket closed with our bytes unread resets us; the queue is dropped with it
        except socket.timeout:
            pass
        finally:
            s.close()
        # the connection was ended by the server, with a GOAWAY frame (type 7, stream 0) whenever we got to read it
        return cut and (b"\x07\x00\x00\x00\x00\x00" in got or not got or len(got) < 64)

    pre = b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + frame(4, 0, 0)
    # HEADERS without END_HEADERS followed by 10 x 16 KiB CONTINUATION frames of literal headers
    lit = b"\x00\x01a" + b"\x7f\xf1\x7e" + b"b" * 16368          # name "a", value of 16368 bytes (7-bit prefix integer 127 + 16241)
    flood = pre + frame(1, 0, 1, lit[:16000]) + b"".join(frame(9, 0, 1, lit[:16000]) for _ in range(10))
    assert talk(flood)
    # 150 streams opened and left half-open (no END_STREAM): refused once 100 are in flight
    hdr = (b"\x83\x86\x44\x1e/v1beta1.DevicePlugin/Allocate" + b"\x41\x09localhost" + b"\x5f\x10application/grpc" + b"\x40\x02te\x08trailers")
    many = pre + b"".join(frame(1, 4, 1 + 2 * i, hdr) for i in range(150))
    assert talk(many)
    assert daemon.proc.poll() is None
    with kubelet.plugin_channel() as ch:
        assert len(next(api.DevicePluginStub(ch).ListAndWatch(api.Empty())).devices) == 8


@pytest.mark.parametrize("variant", ["reference", "two-configs-keep", "no-gfd"])
def test_values_yaml_parses_like_the_python_host(variant, tmp_path):
    """/root/reference/values.yaml exactly as shipped (golden copy), plus variants of the chart values: gfd.enabled,
    runtimeClassName and every config.map.<name> block scalar must come out as config.py reads them."""
    text = G["reference_inputs"]["values.yaml"]["text"]
    if variant == "two-configs-keep":
        text = ("gfd:\n  enabled: false\nruntimeClassName: nvidia\nconfig:\n  map:\n    default: |\n      version: v1\n      flags:\n        migStrategy: none\n"
                "    shared8: |-\n      version: v1\n      sharing:\n        timeSlicing:\n          renameByDefault: true\n          resources:\n"
                "          - name: nvidia.com/gpu\n            replicas: 8\n")
    elif variant == "no-gfd":
        text = "runtimeClassName: nvidia   # nothing else\n"
    path = tmp_path / "values.yaml"
    path.write_text(text)
    out = json.loads(subprocess.run([BIN, "--check-values", str(path)], capture_output=True, text=True, check=True).stdout)
    want = cfgmod.parse_helm_values(text)
    assert out["ok"] and out["gfd_enabled"] == want.gfd_enabled and out["runtime_class_name"] == want.runtime_class_name
    assert out["raw_configs"] == want.raw_configs                     # block scalars byte for byte (|- strips, | keeps the newline)
    assert list(out["configs"]) == list(want.configs)
    for name, c in want.configs.items():
        o = out["configs"][name]
        assert (o["version"], o["mig_strategy"], o["rename_by_default"], o["resource_name"], o["replicas"], o["is_shared"]) == \
            (c.version, c.mig_strategy, c.time_slicing.rename_by_default, c.resource_name(), c.replicas(), c.is_shared())
    d = want.default
    assert (out["default"]["resource_name"], out["default"]["replicas"]) == (d.resource_name(), d.replicas())


def test_label_rules_match_the_python_host_on_synthetic_probe_results():
    """labels.hpp against labels.py on random probe outcomes: same keys, same rounding (half-to-even), same
    verdict sizes, same thresholds, same gate — compared as rendered feature files."""
    import random
    from types import SimpleNamespace as NS

    from k3s_nvidia_b200 import labels as L

    rng = random.Random(4242)
    mode_name = {1: "read", 2: "write", 4: "copy"}
    for trial in range(60):
        lines, hbm, gemm, passive = [], {}, {}, {}
        ngpu = rng.randint(1, 8)
        for gpu in range(ngpu):
            if rng.random() < 0.9:
                pts = []
                for lg in rng.sample(range(20, 31), rng.randint(1, 6)):
                    for mode in rng.sample([1, 2, 4], rng.randint(1, 3)):
                        gbs = rng.choice([rng.uniform(5000, 7300), rng.uniform(100, 6000), float(rng.randint(5000, 7000)) + 0.5])
                        ver = rng.choice([1, 1, 1, 0, -1])
                        resident = int((2 if mode == 4 else 1) * (1 << lg) <= 126 << 20)
                        lines.append(f"hbm {gpu} {1 << lg} {mode} {gbs!r} {ver} {resident}")
                        pts.append(NS(bytes=1 << lg, mode=mode_name[mode], gbs_median=gbs, verified=ver, cache_resident=bool(resident)))
                hbm[gpu] = pts
            if rng.random() < 0.8:
                tf, ver = rng.choice([rng.uniform(900, 1700), 1169.14, 1250.5]), rng.choice([1, 1, 0])
                lines.append(f"gemm {gpu} {tf!r} {ver}")
                gemm[gpu] = NS(tflops_median=tf, verified=ver)
            if rng.random() < 0.8:
                total = rng.choice([18, 18, 0, 12])
                st = dict(links_total=total, links_active=rng.choice([total, total, max(0, total - 2)]), fabric_state=rng.choice([3, 3, -1, 2]),
                          fabric_status=rng.choice([0, 0, 9]), fabric_health_mask=rng.choice([0, 0, 1, 2, 0x10]))
                lines.append(f"passive {gpu} {st['links_total']} {st['links_active']} {st['fabric_state']} {st['fabric_status']} {st['fabric_health_mask']}")
                passive[gpu] = st
        want = {}
        th = L.Thresholds()
        if hbm:
            want.update(L.hbm_labels(hbm, th))
        if gemm:
            want.update(L.gemm_labels(gemm, th))
        want.update(L.nvlink_passive_labels(passive))
        if ngpu >= 2 and rng.random() < 0.8:
            g = ngpu
            egress = [rng.choice([rng.uniform(600, 710), 671.5, 672.0]) for _ in range(g)]
            ingress = [rng.uniform(600, 710) for _ in range(g)]
            pair = [[0.0 if i == j else rng.choice([rng.uniform(80, 110), 0.0]) for j in range(g)] for i in range(g)]
            ver, mn = rng.choice([1, 1, 0]), rng.uniform(80, 100)
            lines.append(f"a2a {g} {ver} {mn!r} " + " ".join(repr(x) for x in egress + ingress + [v for row in pair for v in row]))
            want.update(L.nvlink_labels(NS(g=g, verified=ver, egress_gbs=egress, ingress_gbs=ingress, pair_gbs=pair, min_pair_gbs=mn), th))
        want.update(L.gate_label(want))
        out = subprocess.run([BIN, "--labels-from-stdin"], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
        assert out == L.render(want), (trial, lines)


def test_link_localisation_is_the_same_function_in_both_hosts():
    """SURVEY.md §8f.3 twin check: random pair matrices (healthy, one cold endpoint, cold rows / columns, single cold pairs, ties)
    joined with random passive link states give byte-identical label sets from labels.hpp and labels.py, for exchanges over a
    SUBSET of the node's GPUs (positions != NVML indices)."""
    import random
    from types import SimpleNamespace as NS

    from k3s_nvidia_b200 import _lib
    from k3s_nvidia_b200 import labels as L

    rng = random.Random(8763)
    for trial in range(120):
        n_node = rng.randint(2, 8)
        ids = sorted(rng.sample(range(n_node), rng.randint(2, n_node)))          # the idle GPUs that took part, by NVML index
        g = len(ids)
        base = rng.choice([700.0, 705.5, 692.0])
        pair = [[0.0 if i == j else base + rng.uniform(-4, 4) for j in range(g)] for i in range(g)]
        kind = rng.random()
        bad = rng.randrange(g)
        if kind < 0.25:                                                          # one endpoint cold in both directions
            for q in range(g):
                if q != bad:
                    pair[bad][q] = base * rng.uniform(0.5, 0.88)
                    pair[q][bad] = base * rng.uniform(0.5, 0.88)
        elif kind < 0.45:                                                        # cold row (egress) or column (ingress)
            for q in range(g):
                if q != bad:
                    if kind < 0.35:
                        pair[bad][q] = base * 0.8
                    else:
                        pair[q][bad] = base * 0.8
        elif kind < 0.6:                                                         # a single cold pair, or two with equal values (tie-breaks)
            i, j = rng.sample(range(g), 2)
            pair[i][j] = 500.0
            if rng.random() < 0.5:
                pair[j][i] = 500.0
        source = rng.choice([_lib.PAIR_STEPPED, _lib.PAIR_STEPPED, _lib.PAIR_ISOLATED, _lib.PAIR_SHARE])
        passive, lines = {}, []
        for idx in range(n_node):
            total = 18
            down = 0
            if rng.random() < 0.25:
                for link in rng.sample(range(18), rng.randint(1, 3)):
                    down |= 1 << link
            st = dict(links_total=total, links_active=total - bin(down).count("1"), active_mask=((1 << total) - 1) & ~down, fabric_state=3, fabric_status=0,
                      fabric_health_mask=0)
            passive[idx] = st
            lines.append(f"passive {idx} {total} {st['links_active']} 3 0 0 {st['active_mask']}")
        flat = [v for row in pair for v in row if v > 0]
        egress = [sum(pair[i]) / (g - 1) for i in range(g)]
        lines.append(f"a2a {g} 1 {min(flat)!r} " + " ".join(repr(x) for x in egress + egress + [v for row in pair for v in row]))
        lines.append(f"a2ax {source} " + " ".join(str(i) for i in ids))
        rep = NS(g=g, verified=1, egress_gbs=egress, ingress_gbs=egress, pair_gbs=pair, min_pair_gbs=min(flat), max_pair_gbs=max(flat), pair_source=source)
        th = L.Thresholds()
        want = {}
        want.update(L.nvlink_passive_labels(passive))
        want.update(L.nvlink_labels(rep, th, ids))
        want.update(L.nvlink_localise(rep, ids, passive))
        want.update(L.gate_label(want))
        out = subprocess.run([BIN, "--labels-from-stdin"], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
        assert out == L.render(want), (trial, kind, source, ids, lines[-2:], out, L.render(want))


@pytest.mark.parametrize("host", ["native", "python"])
def test_daemon_publishes_an_expiring_file_and_withdraws_it_on_sigterm(host, sock_dir, monkeypatch):
    """The active-probe runner inside the daemon (both hosts): first round at start-up writes features.d/b200probe with the
    expiry directive; SIGTERM wakes the runner out of its 600 s sleep at once (ADVICE r1: the native stop() could lose the
    wake-up and block for the whole interval), the verdicts are withdrawn and the process exits."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present: the round would run the real probes")
    monkeypatch.setenv("PYTHONPATH", ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    cfg = os.path.join(d, "config.yaml")
    open(cfg, "w").write(VALUES.raw_configs["default"])
    feat = os.path.join(d, "features.d")
    cmd = [BIN] if host == "native" else [sys.executable, "-m", "k3s_nvidia_b200.plugin"]
    env = dict(os.environ, MOCK_NVML_DEVICES="2")
    log = open(os.path.join(d, "daemon.log"), "w")
    proc = subprocess.Popen([*cmd, "--config-file", cfg, "--socket-dir", d, "--nvml-path", _oracle.MOCK_NVML, "--features-dir", feat,
                             "--probe-interval", "600", "--watch-period", "0.05", "--health-timeout-ms", "5"], env=env, stderr=log)
    try:
        path = os.path.join(feat, "b200probe")
        t_end = time.time() + 30
        while not os.path.exists(path) and time.time() < t_end and proc.poll() is None:
            time.sleep(0.05)
        assert os.path.exists(path), open(os.path.join(d, "daemon.log")).read()[-2000:]
        text = open(path).read()
        assert text.startswith("# +expiry-time=") and "nvidia.com/b200probe.healthy=false" in text       # no CUDA here: probes fail, gate false
        assert "nvidia.com/b200probe.gpu0.probe-state=probed" in text and "timestamp" not in text
        assert kubelet.event.wait(30)
        t0 = time.time()
        proc.send_signal(signal.SIGTERM)
        proc.wait(10)
        assert time.time() - t0 < 5.0, "the runner did not wake up from its interval sleep"
        assert not os.path.exists(path), "the feature file must be withdrawn on a clean stop"
        log.flush()
        text = open(os.path.join(d, "daemon.log")).read()
        assert "Sanitizer" not in text and "runtime error" not in text, text[-4000:]      # asan / tsan builds report on stderr
    finally:
        if proc.poll() is None:
            proc.kill()
        log.close()
        kubelet.stop()


def test_scripted_probe_rounds_give_the_same_labels_in_both_hosts(tmp_path, monkeypatch):
    """The whole policy of the active-probe runner, round by round, native host against Python host on the SAME script:
    calibration on the first healthy round (and the stricter gate it implies afterwards), a busy GPU skipped with its last idle
    verdict carried over and the exchange run over the idle subset, out-of-memory treated as inconclusive, cold cells named,
    everything busy -> verdicts stand.  The native runner sees the script through an LD_PRELOAD interposer over the probe entry
    points (tests/fake_probe), the Python runner through the duck-typed FakeProbe of test_labels.py; enumeration and passive
    link state come from the mock NVML in both."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from k3s_nvidia_b200 import labels as L
    from test_labels import FakeProbe

    fake = os.path.join(ROOT, "tests", "fake_probe", "libfakeprobe.so")
    rounds = [
        dict(copy={0: 7000.0}),                                                        # gpu0's own figure is above the pool's: calibrated at 7000
        dict(busy={1}, copy={0: 6100.0}),                                              # 6100 clears 0.9 x pool but not 0.9 x 7000; gpu1 keeps its verdict
        dict(nomem={2}, pair={(3, 0): 600.0, (3, 1): 600.0}),                          # exchange over {0,1,3}: gpu3's egress row is cold
        dict(pair={(0, 3): 500.0}),                                                    # all idle again: a single cold pair
        dict(busy={0, 1, 2, 3}),                                                       # nothing measurable: every verdict stands
    ]
    preload = fake
    if "asan" in os.path.basename(BIN):           # the ASan runtime must come first in the preload list
        preload = subprocess.check_output(["/usr/bin/g++", "-print-file-name=libasan.so"], text=True).strip() + ":" + fake
    env = dict(os.environ, MOCK_NVML_DEVICES="4", LD_PRELOAD=preload)
    for r, sc in enumerate(rounds):
        if sc.get("busy"):
            env[f"FAKE_R{r}_BUSY"] = ",".join(str(i) for i in sorted(sc["busy"]))
        if sc.get("nomem"):
            env[f"FAKE_R{r}_NOMEM"] = ",".join(str(i) for i in sorted(sc["nomem"]))
        if sc.get("copy"):
            env[f"FAKE_R{r}_COPY"] = ",".join(f"{i}:{v}" for i, v in sc["copy"].items())
        if sc.get("pair"):
            env[f"FAKE_R{r}_PAIR"] = ",".join(f"{a}>{b}:{v}" for (a, b), v in sc["pair"].items())
    out = subprocess.run([BIN, "--probe-rounds", str(len(rounds)), "--features-dir", str(tmp_path / "native"), "--nvml-path", _oracle.MOCK_NVML],
                         env=env, capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    assert "Sanitizer" not in out.stderr and "runtime error" not in out.stderr, out.stderr[-3000:]
    native = [L.parse_feature_file(chunk.split("\n", 1)[1]) for chunk in out.stdout.split("== round ")[1:]]
    assert len(native) == len(rounds)

    fp = FakeProbe(n=4)
    runner = L.ActiveProbeRunner(fp, features_dir=str(tmp_path / "py"), interval_s=3600)
    for r, sc in enumerate(rounds):
        fp.busy, fp.nomem = set(sc.get("busy", ())), set(sc.get("nomem", ()))
        fp.copy_gbs = {i: 6600.0 for i in range(4)}
        fp.copy_gbs.update(sc.get("copy", {}))
        fp.pair_override = dict(sc.get("pair", {}))
        py = runner.run_once()
        assert native[r] == py, (r, sorted(set(native[r].items()) ^ set(py.items())))
    P = "nvidia.com/b200probe."
    assert native[0][P + "healthy"] == "true"
    assert native[1][P + "gpu0.hbm-healthy"] == "false" and native[1][P + "gpu1.probe-state"] == "busy" and native[1][P + "gpu1.hbm-copy-gbs"] == "6600"
    assert native[2][P + "gpu2.probe-state"] == "no-memory" and native[2][P + "nvlink-suspect"] == "gpu3" and native[2][P + "nvlink-suspect-evidence"] == "egress-cold"
    assert native[3][P + "nvlink-cold-cell"] == "gpu0-to-gpu3" and native[3][P + "nvlink-suspect-evidence"] == "pair-only"
    assert native[4] == {**native[3], **{P + f"gpu{i}.probe-state": "busy" for i in range(4)}}
    # the per-pair labels can be switched off in both hosts; summary and localisation stay
    env["B200PROBE_PAIR_LABELS"] = "0"
    monkeypatch.setenv("B200PROBE_PAIR_LABELS", "0")
    out = subprocess.run([BIN, "--probe-rounds", "1", "--features-dir", str(tmp_path / "native2"), "--nvml-path", _oracle.MOCK_NVML],
                         env=env, capture_output=True, text=True, timeout=60)
    lean = L.parse_feature_file(out.stdout)
    fp2 = FakeProbe(n=4)
    fp2.copy_gbs[0] = 7000.0
    assert lean == L.ActiveProbeRunner(fp2, features_dir=str(tmp_path / "py2"), interval_s=3600).run_once()
    assert not [k for k in lean if "nvlink-to-gpu" in k] and lean[P + "nvlink-cold-cell"] == "none" and len(native[0]) - len(lean) == 12


def test_sighup_reloads_the_config_document(both_hosts):
    """SURVEY.md §8f.2: a rewritten config file + SIGHUP (what the chart's config-manager does [RECALLED]) -> new
    replica count advertised after a fresh Register; a document that does not parse keeps the running one.
    Run against the native daemon and the Python twin started from its CLI."""
    kubelet, daemon = both_hosts
    cfg = os.path.join(daemon.dir, "config.yaml")
    n0 = len(kubelet.requests)
    open(cfg, "w").write("version: v1\nsharing:\n  timeSlicing:\n    renameByDefault: true\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 2\n")
    kubelet.event.clear()
    daemon.proc.send_signal(signal.SIGHUP)
    assert kubelet.event.wait(10), daemon.logtext()
    t_end = time.time() + 5
    while "reloaded" not in daemon.logtext() and time.time() < t_end:
        time.sleep(0.02)
    r = kubelet.requests[-1]
    assert len(kubelet.requests) == n0 + 1 and (r.resource_name, r.endpoint) == ("nvidia.com/gpu.shared", "nvidia-gpu-shared.sock")
    with kubelet.plugin_channel() as ch:
        first = next(api.DevicePluginStub(ch).ListAndWatch(api.Empty()))
        assert [d.ID for d in first.devices] == [f"{U0}::0", f"{U0}::1", f"{U1}::0", f"{U1}::1"]
    open(cfg, "w").write("version: v7\n")
    daemon.proc.send_signal(signal.SIGHUP)
    t_end = time.time() + 5
    while "rejected" not in daemon.logtext() and time.time() < t_end:
        time.sleep(0.02)
    assert "rejected, keeping the running configuration: unknown version: 'v7'" in daemon.logtext()
    daemon.push(0, 0, 79)                        # the reloaded instance still follows the passive health events
    with kubelet.plugin_channel() as ch:
        stream = api.DevicePluginStub(ch).ListAndWatch(api.Empty())
        seen = next(stream)
        if all(d.health == "Healthy" for d in seen.devices):
            seen = next(stream)
        assert [d.health for d in seen.devices] == ["Unhealthy", "Unhealthy", "Healthy", "Healthy"]
        stream.cancel()
    assert len(kubelet.requests) == n0 + 1 and daemon.proc.poll() is None
    with kubelet.plugin_channel() as ch:
        assert len(next(api.DevicePluginStub(ch).ListAndWatch(api.Empty())).devices) == 4


def test_random_frame_sequences_never_crash_the_transport(stack):
    """Structure-aware fuzz of the HTTP/2 layer: valid preface, then random frames (all types, random flags, stream
    ids, lengths, HPACK-ish payloads).  Whatever the answer (GOAWAY, RST, silence), the daemon survives and serves."""
    import random
    import socket
    import struct

    kubelet, daemon = stack
    path = os.path.join(daemon.dir, "nvidia-gpu.sock")
    rng = random.Random(9113)

    def frame(t, flags, stream, payload=b""):
        return struct.pack(">I", len(payload))[1:] + bytes([t, flags]) + struct.pack(">I", stream & 0x7FFFFFFF) + payload

    good_hdr = b"\x83\x86\x44\x1e/v1beta1.DevicePlugin/Allocate" + b"\x41\x09localhost" + b"\x5f\x10application/grpc" + b"\x40\x02te\x08trailers"
    for _ in range(150):
        data = b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + (frame(4, 0, 0) if rng.random() < 0.8 else b"")
        for _ in range(rng.randint(1, 12)):
            t = rng.choice([0, 0, 1, 1, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 0x42])
            flags = rng.choice([0, 1, 4, 5, 8, 0x20, 0x24, 0x2D, rng.randrange(256)])
            stream = rng.choice([0, 1, 1, 3, 5, 2, rng.randrange(1 << 31)])
            kind = rng.random()
            if kind < 0.3:
                payload = good_hdr
            elif kind < 0.5:
                payload = b"\x00" + struct.pack(">I", rng.choice([0, 2, 5, 1 << 20])) + os.urandom(rng.randint(0, 40))     # gRPC-framed-ish DATA
            elif kind < 0.7:
                payload = os.urandom(rng.choice([0, 1, 4, 5, 6, 8, 9, 64, 300]))
            else:
                payload = bytes(rng.choice([0x80, 0xFF, 0x40, 0x20, 0x3F, 0x00, 0x7F, 0x0F]) for _ in range(rng.randint(0, 24)))
            data += frame(t, flags, stream, payload)
        s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        s.settimeout(0.05)
        try:
            s.connect(path)
            s.sendall(data)
            try:
                s.recv(65536)
            except (socket.timeout, ConnectionError):
                pass
        except (BrokenPipeError, ConnectionError):
            pass
        finally:
            s.close()
    assert daemon.proc.poll() is None, daemon.logtext()
    with kubelet.plugin_channel() as ch:
        stub = api.DevicePluginStub(ch)
        assert len(next(stub.ListAndWatch(api.Empty())).devices) == 8
        r = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::0"])]))
        assert dict(r.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}


def test_frames_on_a_finished_stream_and_oversize_frames_are_refused(stack):
    """ADVICE r1: DATA after END_STREAM used to append to the request a worker was already reading and dispatch the call a
    second time; frames above SETTINGS_MAX_FRAME_SIZE (never raised: 16384) were read up to 16 MiB.  Now: RST_STREAM
    (STREAM_CLOSED) for the late DATA and exactly one response; GOAWAY(FRAME_SIZE_ERROR) without reading the oversize frame."""
    import socket
    import struct

    kubelet, daemon = stack
    path = os.path.join(daemon.dir, "nvidia-gpu.sock")

    def frame(t, flags, stream, payload=b""):
        return struct.pack(">I", len(payload))[1:] + bytes([t, flags]) + struct.pack(">I", stream & 0x7FFFFFFF) + payload

    def read_frames(sock, seconds=1.0):
        sock.settimeout(0.2)
        buf, t_end = b"", time.time() + seconds
        while time.time() < t_end:
            try:
                chunk = sock.recv(65536)
            except socket.timeout:
                continue
            except ConnectionError:
                break
            if not chunk:
                break
            buf += chunk
        out = []
        while len(buf) >= 9:
            n = int.from_bytes(buf[:3], "big")
            out.append((buf[3], buf[4], int.from_bytes(buf[5:9], "big") & 0x7FFFFFFF, buf[9:9 + n]))
            buf = buf[9 + n:]
        return out

    hdr = b"\x83\x86\x44\x1e/v1beta1.DevicePlugin/Allocate" + b"\x41\x09localhost" + b"\x5f\x10application/grpc" + b"\x40\x02te\x08trailers"
    req = api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{U0}::0"])]).SerializeToString()
    body = b"\x00" + struct.pack(">I", len(req)) + req
    s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
    s.connect(path)
    s.sendall(b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + frame(4, 0, 0) + frame(1, 4, 1, hdr) + frame(0, 1, 1, body)      # a complete unary call ...
              + frame(0, 1, 1, body))                                                                                     # ... and DATA + END_STREAM again
    got = read_frames(s)
    s.close()
    rst = [f for f in got if f[0] == 3 and f[2] == 1]
    assert rst and int.from_bytes(rst[0][3], "big") == 5, got                      # RST_STREAM(STREAM_CLOSED) for the late DATA
    data = [f for f in got if f[0] == 0 and f[2] == 1]
    assert len(data) == 1, "the call must be answered exactly once"
    resp = api.AllocateResponse.FromString(data[0][3][5:])
    assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": U0}
    # oversize frame: only the 9-byte header is sent; a reader that waited for the body would hang instead of answering
    s = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
    s.connect(path)
    s.sendall(b"PRI * HTTP/2.0\r\n\r\nSM\r\n\r\n" + frame(4, 0, 0) + struct.pack(">I", 16385)[1:] + bytes([0, 0]) + struct.pack(">I", 1))
    got = read_frames(s)
    s.close()
    goaway = [f for f in got if f[0] == 7]
    assert goaway and int.from_bytes(goaway[0][3][4:8], "big") == 6, got             # FRAME_SIZE_ERROR
    assert daemon.proc.poll() is None
    with kubelet.plugin_channel() as ch:
        assert len(next(api.DevicePluginStub(ch).ListAndWatch(api.Empty())).devices) == 8


def test_committed_huffman_table_is_what_libnghttp2_implements(tmp_path):
    """host/cpp/hpack_huffman.inc regenerated from the system libnghttp2 (tools/gen_hpack_huffman.py) is byte-identical
    to the committed file: the table is pinned to an independent implementation of RFC 7541 Appendix B."""
    import ctypes.util
    import sys

    if not ctypes.util.find_library("nghttp2"):
        pytest.skip("libnghttp2 not on this box")
    out = tmp_path / "huff.inc"
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_hpack_huffman.py"), str(out)], check=True, capture_output=True, timeout=300)
    assert out.read_text() == open(os.path.join(ROOT, "host", "cpp", "hpack_huffman.inc")).read()


def test_unshared_config_and_index_strategy(sock_dir):
    """No time-slicing: bare UUIDs are advertised and preferred allocation is required-first; deviceIDStrategy
    index makes Allocate answer with NVML indices (both as plugin.py does)."""
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    daemon = Daemon(d, "version: v1\nflags:\n  migStrategy: none\n  plugin:\n    deviceIDStrategy: index\n", extra_env={"MOCK_NVML_DEVICES": "4"})
    try:
        assert kubelet.event.wait(10) and daemon.wait_serving(), daemon.logtext()
        with kubelet.plugin_channel() as ch:
            stub = api.DevicePluginStub(ch)
            ids = [x.ID for x in next(stub.ListAndWatch(api.Empty())).devices]
            assert ids == [f"GPU-b2000000-0000-4000-8000-00000000000{i}" for i in range(4)]
            resp = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[ids[2], ids[0]])]))
            assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": "2,0"}
            pref = stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                api.ContainerPreferredAllocationRequest(available_deviceIDs=ids, must_include_deviceIDs=[ids[3]], allocation_size=2)]))
            assert list(pref.container_responses[0].deviceIDs) == [ids[3], ids[0]]
            with pytest.raises(grpc.RpcError) as e:
                stub.GetPreferredAllocation(api.PreferredAllocationRequest(container_requests=[
                    api.ContainerPreferredAllocationRequest(available_deviceIDs=ids[:1], allocation_size=2)]))
            assert "not enough available devices" in e.value.details()
    finally:
        daemon.stop()
        kubelet.stop()


def test_probe_round_without_a_gpu_publishes_unhealthy_like_the_python_runner(tmp_path, monkeypatch):
    """GPU-less box: every active probe fails with B200PROBE_ENOCUDA (no CPU fallback anywhere) and both hosts publish
    the same feature file — probes unhealthy, gate false, passive NVLink view (mock NVML) still reported."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from k3s_nvidia_b200 import labels as L
    from k3s_nvidia_b200.probe import Probe

    env = dict(os.environ, MOCK_NVML_DEVICES="2", MOCK_NVML_LINKS_DOWN="1:4")
    out = subprocess.run([BIN, "--probe-once", "--features-dir", str(tmp_path / "native"), "--nvml-path", _oracle.MOCK_NVML], env=env,
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    assert "no CPU fallback" in out.stderr
    native = L.parse_feature_file(out.stdout)
    assert native == L.parse_feature_file(open(tmp_path / "native" / "b200probe").read())
    monkeypatch.setenv("MOCK_NVML_DEVICES", "2")
    monkeypatch.setenv("MOCK_NVML_LINKS_DOWN", "1:4")
    p = Probe(_oracle.MOCK_NVML)
    try:
        py = L.ActiveProbeRunner(p, features_dir=str(tmp_path / "py"), interval_s=3600).run_once()
    finally:
        p.close()
    assert "nvidia.com/b200probe.timestamp" not in native        # no churning label: staleness is the file's expiry directive
    assert out.stdout.count("# +expiry-time=") == 0 and open(tmp_path / "native" / "b200probe").read().startswith("# +expiry-time=")
    assert native == py
    assert native["nvidia.com/b200probe.healthy"] == "false" and native["nvidia.com/b200probe.gpu1.nvlink-links-ok"] == "false"


def test_both_hosts_skip_a_busy_gpu_the_same_way(tmp_path, monkeypatch):
    """A GPU with a foreign compute process (mock NVML) is not probed by either host: probe-state=busy, no verdict label
    for it (nothing to carry over on a first round), while the idle GPU's probe is attempted (and fails here: no CUDA)."""
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from k3s_nvidia_b200 import labels as L
    from k3s_nvidia_b200.probe import Probe

    env = dict(os.environ, MOCK_NVML_DEVICES="2", MOCK_NVML_BUSY="1:1:0")
    out = subprocess.run([BIN, "--probe-once", "--features-dir", str(tmp_path / "native"), "--nvml-path", _oracle.MOCK_NVML], env=env,
                         capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    assert "Sanitizer" not in out.stderr and "runtime error" not in out.stderr, out.stderr[-4000:]
    native = L.parse_feature_file(out.stdout)
    monkeypatch.setenv("MOCK_NVML_DEVICES", "2")
    monkeypatch.setenv("MOCK_NVML_BUSY", "1:1:0")
    p = Probe(_oracle.MOCK_NVML)
    try:
        py = L.ActiveProbeRunner(p, features_dir=str(tmp_path / "py"), interval_s=3600).run_once()
    finally:
        p.close()
    assert native == py
    P = "nvidia.com/b200probe."
    assert native[P + "gpu1.probe-state"] == "busy" and native[P + "gpu0.probe-state"] == "probed"
    assert P + "gpu1.hbm-healthy" not in native and native[P + "gpu0.hbm-healthy"] == "false"
    assert P + "nvlink-healthy" not in native                   # fewer than two idle GPUs: no exchange, no NVLink verdict
