"""values.yaml / plugin config semantics (SURVEY.md §4 "Config tests", §8a rows a1, a7, a8)."""
import hashlib
import json
import os

import pytest

from k3s_nvidia_b200 import config as cfgmod

G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden.json")))
VALUES = G["reference_inputs"]["values.yaml"]["text"]
# sha256 of the files as UntouchedWagons/K3S-NVidia ships them, read from the original when the golden copies were made
REFERENCE_SHA256 = {
    "values.yaml": "91df8e3127981db3178d7fef23b7c91d2ddab62051d8264c44742852a8ee0d3b",
    "nvidia-smi.yaml": "7f10e7f0ec783ef7ac1622abee2621d46d48adb937f002b5c2d29fda851853bc",
    "jellyfin.yaml": "558fde9ce57e282d4cf5a1c23f1497c0fa0cc0cc1b4b5a82b61efa2bf61d0e8f",
}


def test_fixture_is_byte_identical_to_the_reference_when_present():
    assert sorted(G["reference_inputs"]) == sorted(REFERENCE_SHA256)
    for name, want in REFERENCE_SHA256.items():
        doc = G["reference_inputs"][name]
        assert hashlib.sha256(doc["text"].encode()).hexdigest() == doc["sha256"] == want, name


def test_reference_values_parse_exactly():
    hv = cfgmod.parse_helm_values(VALUES)
    assert hv.gfd_enabled is True                      # values.yaml:1-2
    assert hv.runtime_class_name == "nvidia"           # values.yaml:4
    assert list(hv.configs) == ["default"]             # values.yaml:8
    c = hv.default
    assert c.version == "v1" and c.mig_strategy == "none"          # :9-11
    ts = c.time_slicing
    assert ts.rename_by_default is False and ts.fail_requests_greater_than_one is False   # :14-15
    assert [(r.name, r.replicas, r.rename) for r in ts.resources] == [("nvidia.com/gpu", 4, None)]   # :16-18
    assert c.resource_name() == "nvidia.com/gpu"       # renameByDefault:false -> name unchanged
    assert c.replicas() == 4 and c.is_shared()
    assert hv.raw_configs["default"].startswith("version: v1\nflags:\n  migStrategy: none\n")


def test_replica_expansion_one_gpu_is_four():
    """/root/reference/README.md:112 — "treat that one GPU as if it were actually four GPUs"."""
    u = "GPU-f524787b-e135-6b26-77fd-95e109aac3c0"
    ids = cfgmod.expand_replicas([u], 4)
    assert ids == [f"{u}::0", f"{u}::1", f"{u}::2", f"{u}::3"]
    assert all(cfgmod.strip_replica(i) == u and cfgmod.has_replica(i) for i in ids)
    assert cfgmod.expand_replicas([u], 1) == [u]
    eight = [f"GPU-{i:08x}" for i in range(8)]
    assert len(cfgmod.expand_replicas(eight, 4)) == 32           # 8 B200 -> 32 advertised devices
    assert cfgmod.strip_replica(u) == u


def test_rename_variants():
    doc = VALUES_DOC.replace("renameByDefault: false", "renameByDefault: true")
    assert cfgmod.parse_plugin_config(doc).resource_name() == "nvidia.com/gpu.shared"
    doc = VALUES_DOC.replace("replicas: 4", "replicas: 4\n        rename: gpu-ts")
    assert cfgmod.parse_plugin_config(doc).resource_name() == "nvidia.com/gpu-ts"
    plain = cfgmod.parse_plugin_config("version: v1\n")
    assert plain.resource_name() == "nvidia.com/gpu" and plain.replicas() == 1 and not plain.is_shared()


VALUES_DOC = cfgmod.parse_helm_values(VALUES).raw_configs["default"]


@pytest.mark.parametrize("bad,msg", [
    ("version: v2\n", "unknown version"),
    ("flags: {}\n", "unknown version"),
    ("version: v1\nflags:\n  migStrategy: sometimes\n", "migStrategy"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n", "missing a 'replicas'"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - replicas: 2\n", "missing a 'name'"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: 0\n", ">= 1"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: nvidia.com/gpu\n      replicas: four\n", "integer"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - name: amd.com/gpu\n      replicas: 2\n", "must start with"),
    ("version: v1\nsharing:\n  timeSlicing:\n    renameByDefault: maybe\n", "boolean"),
    ("version: v1\nsharing:\n  timeSlicing:\n    resources:\n    - {name: gpu, replicas: 2}\n    - {name: nvidia.com/gpu, replicas: 3}\n", "duplicate"),
])
def test_invalid_configs_are_rejected(bad, msg):
    with pytest.raises(cfgmod.ConfigError) as e:
        cfgmod.parse_plugin_config(bad)
    assert msg in str(e.value)


def test_manifests_request_one_unit_of_the_unrenamed_resource():
    """nvidia-smi.yaml:14-16 and jellyfin.yaml:27-29 request nvidia.com/gpu: "1" with
    runtimeClassName nvidia (:8 / :23) — the name the config above keeps advertising."""
    import yaml

    pod = yaml.safe_load(G["reference_inputs"]["nvidia-smi.yaml"]["text"])
    assert pod["spec"]["runtimeClassName"] == "nvidia"
    assert pod["spec"]["containers"][0]["resources"]["limits"] == {"nvidia.com/gpu": "1"}
    docs = list(yaml.safe_load_all(G["reference_inputs"]["jellyfin.yaml"]["text"]))
    dep = docs[0]["spec"]["template"]["spec"]
    assert dep["runtimeClassName"] == "nvidia"
    assert dep["containers"][0]["resources"]["limits"] == {"nvidia.com/gpu": "1"}
    assert cfgmod.parse_helm_values(VALUES).default.resource_name() in pod["spec"]["containers"][0]["resources"]["limits"]
