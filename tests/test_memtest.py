"""The HBM integrity probe without a GPU: ABI mirrors, the passive ECC / row-remap query against a scripted mock NVML, the
element oracle, the label rules and the runner policy of both hosts (compared with each other), the feature switched off,
no CPU fallback, and the SASS of the march kernel."""
import ctypes as C
import os
import random
import shutil
import subprocess
from types import SimpleNamespace as NS

import numpy as np
import pytest

import _oracle
from k3s_nvidia_b200 import labels as L

ROOT = _oracle.ROOT
MT = os.path.join(ROOT, "tests", "memtest")
MOCK_ECC = os.path.join(MT, "libnvidia-ml-mock-ecc.so")
FAKE_MEMTEST = os.path.join(MT, "libfakememtest.so")
ORACLE = os.path.join(MT, "libmemtest_oracle.so")
BIN = os.environ.get("B200_NATIVE_BIN") or os.path.join(ROOT, "host", "cpp", "build", "b200-device-plugin")
P = L.PREFIX


@pytest.fixture(scope="module", autouse=True)
def _libs():
    if not all(os.path.exists(p) for p in (MOCK_ECC, FAKE_MEMTEST, ORACLE)):
        subprocess.run(["make", "-C", MT], check=True, capture_output=True)


def _no_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")


# ---- ABI -----------------------------------------------------------------------------------------------------------
def test_struct_sizes_match_the_c_compiler(tmp_path):
    from k3s_nvidia_b200 import _lib

    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "b200probe.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                   "sizeof(b200probe_ecc_status_t),sizeof(b200probe_memtest_cfg_t),sizeof(b200probe_memtest_result_t),"
                   "offsetof(b200probe_memtest_result_t,ecc_after),offsetof(b200probe_memtest_result_t,first_bad_element));return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_lib.EccStatus), C.sizeof(_lib.MemtestCfg), C.sizeof(_lib.MemtestResult), _lib.MemtestResult.ecc_after.offset,
            _lib.MemtestResult.first_bad_element.offset]
    assert got == want


# ---- passive side: ECC mode, volatile totals, row remapper --------------------------------------------------------------
def test_hbm_ecc_reads_the_scripted_nvml_and_reports_minus_one_when_not_supported(monkeypatch):
    from k3s_nvidia_b200 import _lib
    from k3s_nvidia_b200.probe import Probe, ProbeError

    _lib.load().b200probe_shutdown()
    monkeypatch.setenv("MOCK_NVML_DEVICES", "3")
    monkeypatch.setenv("MOCK_NVML_ECC", "0:1:17:2,2:1:5:-1")
    monkeypatch.setenv("MOCK_NVML_REMAP", "0:3:1:1:0")
    p = Probe(MOCK_ECC)
    try:
        assert p.hbm_ecc(0) == dict(ecc_mode=1, corrected_volatile=17, uncorrected_volatile=2, remap_corrected_rows=3, remap_uncorrected_rows=1,
                                    remap_pending=1, remap_failure=0)
        none = dict(ecc_mode=-1, corrected_volatile=-1, uncorrected_volatile=-1, remap_corrected_rows=-1, remap_uncorrected_rows=-1, remap_pending=-1,
                    remap_failure=-1)
        assert p.hbm_ecc(1) == none                                        # not listed: every query NOT_SUPPORTED
        assert p.hbm_ecc(2) == dict(none, ecc_mode=1, corrected_volatile=5)   # one counter unsupported, the other read
        monkeypatch.setenv("MOCK_NVML_ECC", "0:1:20:2")                    # read at every query
        monkeypatch.setenv("MOCK_NVML_REMAP", "0:3:2:0:1")
        e = p.hbm_ecc(0)
        assert (e["corrected_volatile"], e["remap_pending"], e["remap_failure"]) == (20, 0, 1)
        with pytest.raises(ProbeError) as err:
            p.hbm_ecc(3)
        assert err.value.rc == -5
    finally:
        p.close()


def test_the_plain_mock_nvml_has_no_ecc_queries(monkeypatch):
    """The library treats the three queries as optional symbols: an NVML without them reads as NOT_SUPPORTED."""
    from k3s_nvidia_b200 import _lib
    from k3s_nvidia_b200.probe import Probe

    _lib.load().b200probe_shutdown()
    monkeypatch.setenv("MOCK_NVML_DEVICES", "1")
    p = Probe(_oracle.MOCK_NVML)
    try:
        assert set(p.hbm_ecc(0).values()) == {-1}
    finally:
        p.close()


def test_memtest_entry_and_element_return_enocuda_without_a_gpu(monkeypatch):
    _no_gpu()
    from k3s_nvidia_b200 import _lib
    from k3s_nvidia_b200.probe import Probe, ProbeError

    _lib.load().b200probe_shutdown()
    monkeypatch.setenv("MOCK_NVML_DEVICES", "1")
    p = Probe(MOCK_ECC)
    try:
        with pytest.raises(ProbeError) as e:
            p.hbm_memtest(0, fraction=0.5)
        assert e.value.rc == -4
        with pytest.raises(ProbeError) as e:
            p.memtest_element(0, 1 << 20, 4096, 0, _lib.MEMTEST_VERIFY, 1, 2)
        assert e.value.rc == -4
        with pytest.raises(ProbeError) as e:                               # arguments are checked before CUDA is touched
            p.hbm_memtest(0, fraction=1.5)
        assert e.value.rc == -1
        with pytest.raises(ProbeError) as e:
            p.memtest_element(0, 1 << 20, 4098, 0, _lib.MEMTEST_VERIFY, 1, 2)
        assert e.value.rc == -1
    finally:
        p.close()


# ---- the element oracle against a numpy restatement ---------------------------------------------------------------------
def test_element_oracle_against_numpy():
    o = C.CDLL(ORACLE)
    u64p = C.POINTER(C.c_uint64)
    o.oracle_memtest_verify.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, u64p, u64p, C.POINTER(C.c_uint32)]
    o.oracle_memtest_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
    rng = np.random.default_rng(7)
    for base, n, seed in [(0, 4096, 0xB200), ((1 << 32) - 100, 300, 0xFFFF4DFF), (5 << 33, 1000, 0x5A5AE85A)]:
        idx = np.arange(base, base + n, dtype=np.uint64)
        want = ((idx & 0xFFFFFFFF) * np.uint64(2654435761) & np.uint64(0xFFFFFFFF)).astype(np.uint32) ^ np.uint32(seed) ^ (idx >> np.uint64(32)).astype(np.uint32)
        got = np.empty(n, dtype=np.uint32)
        o.oracle_memtest_fill(got.ctypes.data, n, base, seed)
        assert np.array_equal(got, want)
        pos = np.sort(rng.choice(n, 3, replace=False))
        masks = [1 << 3, 0x80000000, 0x00FF0000]
        for i, m in zip(pos, masks):
            got[i] ^= m
        bad, first, bits = C.c_uint64(), C.c_uint64(), C.c_uint32()
        o.oracle_memtest_verify(got.ctypes.data, n, base, seed, C.byref(bad), C.byref(first), C.byref(bits))
        assert (bad.value, first.value, bits.value) == (3, base + int(pos[0]), masks[0] | masks[1] | masks[2])


# ---- label rules: Python and native on the same synthetic results -------------------------------------------------------
def _report(bytes_tested, bad, corr, unc, pending, failure):
    return NS(bytes_tested=bytes_tested, bad_words=bad, ecc_corrected_delta=corr, ecc_uncorrected_delta=unc, remap_pending=pending, remap_failure=failure)


def test_memtest_verdict_rules():
    gib = 1 << 30
    ok = L.memtest_labels(2, _report(161 * gib + (gib >> 1), 0, 12, 0, 1, 0))
    assert ok == {P + "gpu2.hbm-memtest-gib": "162", P + "gpu2.hbm-memtest-bad-words": "0", P + "gpu2.hbm-ecc-corrected-delta": "12",
                  P + "gpu2.hbm-ecc-uncorrected-delta": "0", P + "gpu2.hbm-row-remap-pending": "true", P + "gpu2.hbm-row-remap-failed": "false",
                  P + "gpu2.hbm-memtest-healthy": "true"}                  # corrected errors and a pending remap do not fail it
    assert L.memtest_labels(0, _report(gib, 1, 0, 0, 0, 0))[P + "gpu0.hbm-memtest-healthy"] == "false"
    assert L.memtest_labels(0, _report(gib, 0, 0, 3, 0, 0))[P + "gpu0.hbm-memtest-healthy"] == "false"
    assert L.memtest_labels(0, _report(gib, 0, 0, 0, 0, 1))[P + "gpu0.hbm-memtest-healthy"] == "false"
    unread = L.memtest_labels(0, _report(gib, 0, -1, -1, -1, -1))           # nothing readable from NVML: only the march decides
    assert unread == {P + "gpu0.hbm-memtest-gib": "1", P + "gpu0.hbm-memtest-bad-words": "0", P + "gpu0.hbm-memtest-healthy": "true"}
    assert L.gate_label({P + "hbm-healthy": "true", P + "hbm-memtest-healthy": "false"}) == {P + "healthy": "false"}
    assert L.gate_label({P + "hbm-memtest-healthy": "true"}) == {P + "healthy": "true"}


def test_label_rules_match_between_the_hosts():
    rng = random.Random(1807)
    for trial in range(80):
        lines, want = [], {}
        for gpu in range(rng.randint(1, 8)):
            r = _report(rng.choice([0, 1 << 29, 3 << 29, rng.randrange(1 << 38)]), rng.choice([0, 0, 0, 1, 977]), rng.choice([-1, 0, 0, 5]),
                        rng.choice([-1, 0, 0, 0, 2]), rng.choice([-1, 0, 1]), rng.choice([-1, 0, 0, 1]))
            lines.append(f"memtest {gpu} {r.bytes_tested} {r.bad_words} {r.ecc_corrected_delta} {r.ecc_uncorrected_delta} {r.remap_pending} {r.remap_failure}")
            want.update(L.memtest_labels(gpu, r))
        if rng.random() < 0.5:
            lines.append(f"gemm 0 {rng.uniform(900, 1700)!r} 1")
            want.update(L.gemm_labels({0: NS(tflops_median=float(lines[-1].split()[2]), verified=1)}, L.Thresholds()))
        L.ActiveProbeRunner._aggregate(want, "hbm-memtest-healthy")
        want.update(L.gate_label(want))
        out = subprocess.run([BIN, "--labels-from-stdin"], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
        assert out == L.render(want), (trial, lines)


# ---- runner policy, round by round, in both hosts ------------------------------------------------------------------------
class MemtestFakeProbe:
    """FakeProbe of test_labels.py plus a scripted hbm_memtest (the Python twin of tests/memtest/fake_memtest.c)."""

    def __new__(cls, n):
        from test_labels import FakeProbe

        class _P(FakeProbe):
            script = {}

            def hbm_memtest(self, idx, **kw):
                from k3s_nvidia_b200.probe import ProbeError

                self.calls.append(("memtest", idx, kw.get("fraction")))
                v = self.script.get(idx, (0, 0, 0, 0, 0))
                if v == "enomem":
                    raise ProbeError(L.ENOMEM, "hbm_memtest", "out of device memory")
                if v == "cuda":
                    raise ProbeError(1700, "hbm_memtest", "an illegal memory access was encountered")
                return _report(160 << 30, *v)

        return _P(n=n)


def _script_env(rounds):
    env = {}
    for r, sc in enumerate(rounds):
        if sc.get("busy"):
            env[f"FAKE_R{r}_BUSY"] = ",".join(str(i) for i in sorted(sc["busy"]))
        if sc.get("memtest"):
            env[f"FAKE_R{r}_MEMTEST"] = ",".join(f"{i}:{v}" if isinstance(v, str) else f"{i}:" + ":".join(map(str, v)) for i, v in sc["memtest"].items())
    return env


def _native_rounds(tmp_path, rounds, preload, extra_env):
    env = dict(os.environ, MOCK_NVML_DEVICES="4", LD_PRELOAD=preload, **_script_env(rounds), **extra_env)
    if "asan" in os.path.basename(BIN):
        env["LD_PRELOAD"] = subprocess.check_output(["/usr/bin/g++", "-print-file-name=libasan.so"], text=True).strip() + ":" + preload
    out = subprocess.run([BIN, "--probe-rounds", str(len(rounds)), "--features-dir", str(tmp_path), "--nvml-path", _oracle.MOCK_NVML],
                         env=env, capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr
    chunks = out.stdout.split("== round ")[1:] if len(rounds) > 1 else ["0\n" + out.stdout]
    return [L.parse_feature_file(c.split("\n", 1)[1]) for c in chunks], out.stderr


def _python_rounds(tmp_path, rounds, fp):
    runner = L.ActiveProbeRunner(fp, features_dir=str(tmp_path), interval_s=3600)
    got = []
    for sc in rounds:
        fp.busy = set(sc.get("busy", ()))
        type(fp).script = dict(sc.get("memtest", {}))
        got.append(runner.run_once())
    return got


ROUNDS = [
    dict(),                                                                       # all clean
    dict(memtest={1: (3, 0, 0, 0, 0)}),                                           # gpu1: mismatching words
    dict(busy={1}, memtest={0: (0, 4, 2, 0, 0)}),                                  # gpu1 busy keeps its failed verdict; gpu0 uncorrected ECC
    dict(memtest={2: (0, 0, 0, 1, 1), 3: (0, 9, 0, 1, 0)}),                        # gpu2 remap failed; gpu3 corrected + pending: healthy
    dict(memtest={0: "enomem", 3: "cuda"}),                                       # ENOMEM is inconclusive; a CUDA error fails, not retried
    dict(busy={0, 1, 2, 3}),                                                      # nothing measurable: every verdict stands
]


def test_scripted_rounds_with_the_memtest_on_give_the_same_labels_in_both_hosts(tmp_path, monkeypatch):
    _no_gpu()
    monkeypatch.setenv("B200PROBE_MEMTEST_FRACTION", "0.8")
    native, err = _native_rounds(tmp_path / "native", ROUNDS, FAKE_MEMTEST, {"B200PROBE_MEMTEST_FRACTION": "0.8"})
    assert "Sanitizer" not in err and "runtime error" not in err, err[-3000:]
    fp = MemtestFakeProbe(4)
    py = _python_rounds(tmp_path / "py", ROUNDS, fp)
    for r in range(len(ROUNDS)):
        assert native[r] == py[r], (r, sorted(set(native[r].items()) ^ set(py[r].items())))
    assert {c[2] for c in fp.calls if c[0] == "memtest"} == {0.8}
    n = native
    assert n[0][P + "hbm-memtest-healthy"] == "true" and n[0][P + "healthy"] == "true" and n[0][P + "gpu0.hbm-memtest-gib"] == "160"
    assert n[1][P + "gpu1.hbm-memtest-bad-words"] == "3" and n[1][P + "gpu1.hbm-memtest-healthy"] == "false" and n[1][P + "healthy"] == "false"
    assert n[1][P + "hbm-healthy"] == "true"                                      # the sweep's verdict is its own
    assert n[2][P + "gpu1.probe-state"] == "busy" and n[2][P + "gpu1.hbm-memtest-bad-words"] == "3"      # carried with the other hbm- labels
    assert n[2][P + "gpu0.hbm-ecc-uncorrected-delta"] == "2" and n[2][P + "gpu0.hbm-memtest-healthy"] == "false"
    assert n[3][P + "gpu2.hbm-row-remap-failed"] == "true" and n[3][P + "gpu2.hbm-memtest-healthy"] == "false"
    assert n[3][P + "gpu3.hbm-row-remap-pending"] == "true" and n[3][P + "gpu3.hbm-ecc-corrected-delta"] == "9"
    assert n[3][P + "gpu3.hbm-memtest-healthy"] == "true"
    assert n[4][P + "gpu0.probe-state"] == "no-memory" and n[4][P + "gpu0.hbm-memtest-healthy"] == "true"   # last verdict stands
    assert n[4][P + "gpu3.hbm-memtest-healthy"] == "false" and P + "gpu3.hbm-memtest-gib" not in n[4]
    assert n[5] == {**n[4], **{P + f"gpu{i}.probe-state": "busy" for i in range(4)}}


def test_feature_unset_gives_exactly_todays_labels(tmp_path, monkeypatch):
    """B200PROBE_MEMTEST_FRACTION unset or 0: the label set of the interposer without a memtest, in both hosts."""
    _no_gpu()
    monkeypatch.delenv("B200PROBE_MEMTEST_FRACTION", raising=False)
    plain = os.path.join(ROOT, "tests", "fake_probe", "libfakeprobe.so")
    before, _ = _native_rounds(tmp_path / "a", ROUNDS, plain, {})
    unset, _ = _native_rounds(tmp_path / "b", ROUNDS, FAKE_MEMTEST, {})
    zero, _ = _native_rounds(tmp_path / "c", ROUNDS, FAKE_MEMTEST, {"B200PROBE_MEMTEST_FRACTION": "0"})
    assert before == unset == zero
    assert not [k for r in before for k in r if "memtest" in k or "ecc-" in k or "remap" in k]
    from test_labels import FakeProbe

    fp = FakeProbe(n=4)                                                           # no hbm_memtest at all: it must not be called
    assert _python_rounds(tmp_path / "py", ROUNDS, fp) == before
    monkeypatch.setenv("B200PROBE_MEMTEST_FRACTION", "0")
    assert _python_rounds(tmp_path / "py0", ROUNDS, FakeProbe(n=4)) == before


# ---- SASS --------------------------------------------------------------------------------------------------------------
def test_memtest_kernel_moves_data_with_bulk_tma():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", "-fun", "hbm_memtest_kernel", os.path.join(ROOT, "k3s-nvidia_b200", "libb200probe.so")],
                         capture_output=True, text=True, timeout=300).stdout
    if "Function :" not in out:      # older cuobjdump: match by mangled-name substring over the whole dump
        full = subprocess.run([cuobjdump, "-sass", os.path.join(ROOT, "k3s-nvidia_b200", "libb200probe.so")], capture_output=True, text=True, timeout=300).stdout
        parts = full.split("Function : ")
        out = "\n".join(p for p in parts if p.split("\n", 1)[0].find("hbm_memtest_kernel") >= 0)
    assert "hbm_memtest_kernel" in out
    assert "UBLKCP.S.G" in out and "UBLKCP.G.S" in out                          # cp.async.bulk global->shared and shared->global
    assert "SYNCS.ARRIVE.TRANS64" in out and "TRYWAIT" in out                  # mbarrier expect_tx / try_wait
    assert "STL" not in out and "LDL" not in out
