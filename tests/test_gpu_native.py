"""The native host on a real B200 box: real NVML enumeration behind ListAndWatch, and one active-probe round
(--probe-once: HBM sweep, GEMM, NVLink when >= 2 GPUs) publishing the same label set as the Python runner."""
import os
import subprocess

import pytest

import _oracle  # noqa: F401  (path set-up)
from k3s_nvidia_b200 import api
from test_native_plugin import BIN, Daemon, FakeKubelet

pytestmark = pytest.mark.gpu


def test_native_list_and_watch_matches_nvml_enumeration(sock_dir):
    from k3s_nvidia_b200.probe import Probe

    p = Probe()
    uuids = [p.device_info(i).uuid for i in range(p.device_count())]
    p.close()
    d = str(sock_dir)
    kubelet = FakeKubelet(d)
    kubelet.start()
    env = {k: v for k, v in os.environ.items() if not k.startswith("MOCK_NVML")}
    cfg = os.path.join(d, "config.yaml")
    open(cfg, "w").write("version: v1\nflags:\n  migStrategy: none\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 4\n")
    log = open(os.path.join(d, "daemon.log"), "w")
    proc = subprocess.Popen([BIN, "--config-file", cfg, "--socket-dir", d, "--no-active-probe", "--watch-period", "0"], env=env, stderr=log)
    try:
        assert kubelet.event.wait(20), open(os.path.join(d, "daemon.log")).read()
        with kubelet.plugin_channel() as ch:
            first = next(api.DevicePluginStub(ch).ListAndWatch(api.Empty()))
        assert [x.ID for x in first.devices] == [f"{u}::{r}" for u in uuids for r in range(4)]
        assert {x.health for x in first.devices} == {"Healthy"}
    finally:
        proc.terminate()
        proc.wait(10)
        kubelet.stop()


def test_native_probe_round_publishes_the_python_runner_label_set(tmp_path, monkeypatch):
    import torch

    # this pytest process holds a CUDA context and has just loaded the GPU: to the daemon it IS a tenant, and the round would
    # (correctly) skip the device as busy.  The comparison needs both hosts to probe.
    monkeypatch.setenv("B200PROBE_IGNORE_TENANTS", "1")

    from k3s_nvidia_b200 import labels as L
    from k3s_nvidia_b200.probe import Probe

    out = subprocess.run([BIN, "--probe-once", "--features-dir", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    native = L.parse_feature_file(out.stdout)
    assert native == L.parse_feature_file(open(tmp_path / "b200probe").read())
    assert native["nvidia.com/b200probe.hbm-healthy"] == "true", native
    assert native["nvidia.com/b200probe.gemm-healthy"] == "true", native
    assert native["nvidia.com/b200probe.healthy"] == "true", native
    if torch.cuda.device_count() >= 2:
        assert native["nvidia.com/b200probe.nvlink-data-ok"] == "true"
    p = Probe()
    try:
        py = L.ActiveProbeRunner(p, features_dir=str(tmp_path / "py")).run_once()
    finally:
        p.close()
    assert set(native) == set(py)
    flags = [k for k in py if k.endswith(("-ok", "-healthy", ".healthy", "links-active", "links-total"))]
    assert {k: native[k] for k in flags} == {k: py[k] for k in flags}
    for k in py:                                   # measured figures: same quantity, run-to-run noise only
        if k.endswith(("-gbs", "-tflops")) and "nvlink-to" not in k:
            assert abs(int(native[k]) - int(py[k])) <= 0.05 * int(py[k]) + 1, (k, native[k], py[k])
