import os
import pathlib
import shutil
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Make sure the in-tree artefacts exist (build() normally runs before the tests; this
    covers a bare `pytest`).  Never rebuilds what is already there."""
    need = [
        os.path.join(ROOT, "k3s-nvidia_b200", "libb200probe.so"),
        os.path.join(ROOT, "oracle", "liboracle.so"),
        os.path.join(ROOT, "tests", "mock_nvml", "libnvidia-ml-mock.so"),
        os.path.join(ROOT, "tests", "fake_probe", "libfakeprobe.so"),
        os.path.join(ROOT, "host", "cpp", "build", "b200-device-plugin"),
    ]
    if not all(os.path.exists(p) for p in need):
        import __graft_entry__ as g

        g.build()
    yield


# A unix socket path holds at most 107 bytes.  The deepest one the tests bind is <dir>/py/nvidia-gpu-shared.sock.
_SOCK_DIR_MAX = 107 - len("/py/nvidia-gpu-shared.sock")


@pytest.fixture
def sock_dir(tmp_path):
    """Directory for the kubelet and plugin sockets: tmp_path, unless a long TMPDIR makes it too deep for a
    unix socket path, then a fresh short directory under /tmp that is removed afterwards."""
    if len(str(tmp_path)) <= _SOCK_DIR_MAX:
        yield tmp_path
        return
    d = tempfile.mkdtemp(prefix="b200probe-", dir="/tmp")
    try:
        yield pathlib.Path(d)
    finally:
        shutil.rmtree(d, ignore_errors=True)
