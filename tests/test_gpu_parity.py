"""On the GPU box: enumeration + passive-health verdicts from three independent implementations
must agree exactly — libb200probe.so (product), the C oracle twin, and a pynvml twin
(SURVEY.md §8c: "the strongest bit-exact statement available").  Also drives the plugin's
ListAndWatch/Allocate against the REAL NVML of the box."""
import os
import threading
from concurrent import futures

import grpc
import pytest

import _oracle

pytestmark = pytest.mark.gpu

APP_XIDS = {13, 31, 43, 45, 68, 109}


def pynvml_twin(polls=3, timeout_ms=1):
    """Third restatement of SURVEY.md §3.3 in Python on pynvml."""
    import pynvml as nv

    nv.nvmlInit()
    out, handles = [], []
    for i in range(nv.nvmlDeviceGetCount()):
        h = nv.nvmlDeviceGetHandleByIndex(i)
        handles.append(h)
        out.append([i, nv.nvmlDeviceGetUUID(h), nv.nvmlDeviceGetName(h), nv.nvmlDeviceGetMemoryInfo(h).total,
                    tuple(nv.nvmlDeviceGetCudaComputeCapability(h)), "Healthy"])
    es = nv.nvmlEventSetCreate()
    want = nv.nvmlEventTypeXidCriticalError | nv.nvmlEventTypeDoubleBitEccError | nv.nvmlEventTypeSingleBitEccError
    for rec, h in zip(out, handles):
        try:
            sup = nv.nvmlDeviceGetSupportedEventTypes(h)
            nv.nvmlDeviceRegisterEvents(h, want & sup, es)
        except nv.NVMLError:
            rec[5] = "Unhealthy"
    for _ in range(polls):
        try:
            e = nv.nvmlEventSetWait_v2(es, timeout_ms)
        except nv.NVMLError as err:
            if err.value == nv.NVML_ERROR_TIMEOUT:
                continue
            for rec in out:
                rec[5] = "Unhealthy"
            continue
        if e.eventType != nv.nvmlEventTypeXidCriticalError or e.eventData in APP_XIDS:
            continue
        uuid = nv.nvmlDeviceGetUUID(e.device)
        for rec in out:
            if rec[1] == uuid:
                rec[5] = "Unhealthy"
    nv.nvmlEventSetFree(es)
    return [tuple(r) for r in out]


def test_three_way_enumeration_and_verdict_parity():
    from k3s_nvidia_b200.probe import Probe

    p = Probe()
    try:
        infos = [p.device_info(i) for i in range(p.device_count())]
        p.health_open("")
        for _ in range(3):
            p.health_wait(1)
        mask = p.health_mask()
        product = [(d.index, d.uuid, d.name, d.mem_total, d.cc, "Unhealthy" if (mask >> d.index) & 1 else "Healthy") for d in infos]
    finally:
        p.health_close()
        p.close()
    o = _oracle.load()
    assert o.oracle_ph_open(None, None) == 0
    try:
        for _ in range(3):
            o.oracle_ph_poll(1)
        oracle = _oracle.verdicts(o)
    finally:
        o.oracle_ph_close()
    twin = pynvml_twin()
    assert product == oracle == twin
    assert len(product) >= 1 and all(r[1].startswith("GPU-") for r in product)
    assert all(r[4] == (10, 0) and "B200" in r[2] for r in product)


def test_cuda_ordinals_resolve_by_uuid():
    import torch

    from k3s_nvidia_b200.probe import Probe

    p = Probe()
    try:
        t = torch.zeros(16, dtype=torch.uint8, device="cuda:0")
        p.hbm_fill(0, t.data_ptr(), 16, 1)          # first probe call initialises CUDA inside the library
        torch.cuda.synchronize()
        ords = sorted(p.device_info(i).cuda_ordinal for i in range(p.device_count()))
        assert ords == list(range(torch.cuda.device_count()))
    finally:
        p.close()


def test_plugin_on_real_nvml(sock_dir):
    """BASELINE config 5 plumbing: Register -> ListAndWatch (replicas x4 of the real UUIDs) ->
    Allocate one replica -> NVIDIA_VISIBLE_DEVICES is the real GPU's UUID."""
    import json

    from k3s_nvidia_b200 import api
    from k3s_nvidia_b200 import config as cfgmod
    from k3s_nvidia_b200.plugin import DevicePlugin
    from k3s_nvidia_b200.probe import Probe

    G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
    cfg = cfgmod.parse_helm_values(G["reference_inputs"]["values.yaml"]["text"]).default
    got = threading.Event()
    reqs = []

    class Kubelet:
        def Register(self, request, context):  # noqa: N802
            reqs.append(request)
            got.set()
            return api.Empty()

    d = str(sock_dir)
    srv = grpc.server(futures.ThreadPoolExecutor(max_workers=2))
    api.add_servicer(srv, "Registration", Kubelet())
    srv.add_insecure_port("unix://" + os.path.join(d, "kubelet.sock"))
    srv.start()
    p = Probe()
    plugin = DevicePlugin(p, cfg, socket_dir=d, health_timeout_ms=20)
    try:
        plugin.start(watch_kubelet_period=0)
        assert got.wait(5) and reqs[0].resource_name == "nvidia.com/gpu"
        uuids = [p.device_info(i).uuid for i in range(p.device_count())]
        with grpc.insecure_channel("unix://" + os.path.join(d, reqs[0].endpoint)) as ch:
            stub = api.DevicePluginStub(ch)
            first = next(stub.ListAndWatch(api.Empty()))
            assert [x.ID for x in first.devices] == [f"{u}::{r}" for u in uuids for r in range(4)]
            assert {x.health for x in first.devices} == {"Healthy"}
            resp = stub.Allocate(api.AllocateRequest(container_requests=[api.ContainerAllocateRequest(devices_ids=[f"{uuids[0]}::1"])]))
            assert dict(resp.container_responses[0].envs) == {"NVIDIA_VISIBLE_DEVICES": uuids[0]}
    finally:
        plugin.stop()
        p.close()
        srv.stop(0)


def test_active_probe_round_publishes_gate_label(tmp_path, monkeypatch):
    """configs 3/5: probe results surfaced as NFD labels; the gate label is true on a healthy box."""
    from k3s_nvidia_b200 import labels as L
    from k3s_nvidia_b200.probe import Probe

    monkeypatch.setenv("B200PROBE_IGNORE_TENANTS", "1")      # the test suite itself has just loaded this GPU

    p = Probe()
    try:
        r = L.ActiveProbeRunner(p, features_dir=str(tmp_path), interval_s=3600,
                                hbm_kwargs=dict(min_bytes=1 << 28, max_bytes=1 << 29, warmup=1, reps=3, verify=1))
        lab = r.run_once()
        text = open(tmp_path / "b200probe").read()
        assert L.parse_feature_file(text) == lab
        assert lab["nvidia.com/b200probe.hbm-healthy"] == "true", lab
        assert lab["nvidia.com/b200probe.gemm-healthy"] == "true", lab
        assert int(lab["nvidia.com/b200probe.gpu0.hbm-copy-gbs"]) > 5000
        assert lab["nvidia.com/b200probe.healthy"] == "true"
    finally:
        p.lib.b200probe_hbm_release(0)
        p.close()
