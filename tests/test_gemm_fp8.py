"""The FP8 tensor-core probe without a GPU: the E4M3 operand classes against an independent oracle and torch's float8_e4m3fn,
no CPU fallback, the label rules and the runner policy of both hosts (compared with each other), the switch off, and the
SASS of the E4M3 kernel."""
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
FP8 = os.path.join(ROOT, "tests", "gemm_fp8")
ORACLE = os.path.join(FP8, "libfp8_oracle.so")
FAKE_FP8 = os.path.join(FP8, "libfakegemmfp8.so")
BIN = os.environ.get("B200_NATIVE_BIN") or os.path.join(ROOT, "host", "cpp", "build", "b200-device-plugin")
P = L.PREFIX
SEED = 0xB200


@pytest.fixture(scope="module", autouse=True)
def _libs():
    if not all(os.path.exists(p) for p in (ORACLE, FAKE_FP8)):
        subprocess.run(["make", "-C", FP8], check=True, capture_output=True)


def _no_gpu():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")


def _oracle_lib():
    o = C.CDLL(ORACLE)
    o.oracle_e4m3_value.restype = C.c_double
    o.oracle_e4m3_value.argtypes = [C.c_uint8]
    o.oracle_e4m3_round.restype = C.c_uint8
    o.oracle_e4m3_round.argtypes = [C.c_double]
    o.oracle_fp8_operand.restype = C.c_uint8
    o.oracle_fp8_operand.argtypes = [C.c_uint64, C.c_uint32, C.c_int]
    o.oracle_fp8_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]
    o.oracle_fp8_uniform_f32_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]
    o.oracle_fp8_dot.restype = C.c_double
    o.oracle_fp8_dot.argtypes = [C.c_int, C.c_uint32, C.c_int, C.c_int, C.c_int]
    return o


# ---- E4M3 encoding: the oracle against torch.float8_e4m3fn ----------------------------------------------------------------
def test_oracle_decodes_every_e4m3_byte_like_torch():
    import torch

    o = _oracle_lib()
    want = torch.arange(256, dtype=torch.int32).to(torch.uint8).view(torch.float8_e4m3fn).to(torch.float64).numpy()
    got = np.array([o.oracle_e4m3_value(v) for v in range(256)])
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.isnan(got).sum() == 2            # 0x7F and 0xFF
    assert np.array_equal(got[~np.isnan(got)], want[~np.isnan(want)])
    assert got[0x7E] == 448.0 and got[0x01] == 2.0**-9 and got[0x08] == 2.0**-6


def test_oracle_rounds_like_torch():
    """Nearest E4M3 value, ties to even, over random values and every midpoint between neighbours."""
    import torch

    o = _oracle_lib()
    vals = sorted({o.oracle_e4m3_value(v) for v in range(0x7F)})
    mids = [(a + b) / 2 for a, b in zip(vals, vals[1:])]
    rng = np.random.default_rng(5)
    xs = np.concatenate([mids, -np.array(mids), rng.uniform(-1, 1, 4000), rng.uniform(-448, 448, 2000), rng.uniform(-2**-5, 2**-5, 2000)]).astype(np.float32)
    want = torch.from_numpy(xs).to(torch.float8_e4m3fn).view(torch.uint8).numpy()
    got = np.array([o.oracle_e4m3_round(float(x)) for x in xs], dtype=np.uint8)
    assert np.array_equal(got, want)


# ---- the library's E4M3 operand generator --------------------------------------------------------------------------------
RANGES = [(0, 50_000), ((1 << 33) + 12_345, 50_001)]          # >= 10^5 elements per class and matrix, one range past 2^32


@pytest.mark.parametrize("cls", [0, 1], ids=["exact", "uniform"])
@pytest.mark.parametrize("mat", [0, 1], ids=["A", "B"])
def test_operand_bits_match_the_oracle(cls, mat):
    import torch

    from k3s_nvidia_b200 import _lib

    lib, o = _lib.load(), _oracle_lib()
    which = _lib.GEMM_FILL_E4M3 | (cls << 1) | mat
    for e0, n in RANGES:
        got = np.array([lib.b200probe_gemm_operand_bits(e0 + i, SEED, which) for i in range(n)], dtype=np.uint16)
        assert got.max() <= 0xFF                                               # the byte, in the low 8 bits
        want = np.empty(n, dtype=np.uint8)
        o.oracle_fp8_fill(want.ctypes.data, e0, n, SEED, (cls << 1) | mat)
        assert np.array_equal(got.astype(np.uint8), want)
        vals = torch.from_numpy(want.copy()).view(torch.float8_e4m3fn).to(torch.float64).numpy()
        if cls == 0:
            assert np.array_equal(vals, np.round(vals)) and vals.min() == -8 and vals.max() == 7
        else:                                                                  # the rounding pinned by torch, from the same fp32 values
            x = np.empty(n, dtype=np.float32)
            o.oracle_fp8_uniform_f32_fill(x.ctypes.data, e0, n, SEED, mat)
            assert np.array_equal(torch.from_numpy(x).to(torch.float8_e4m3fn).view(torch.uint8).numpy(), want)
            assert np.all(np.abs(vals) <= 1.0) and len(np.unique(want)) > 100


def test_bf16_operand_classes_are_unchanged():
    """which 0-3 keep returning the bf16 classes the CPU oracle restates."""
    from k3s_nvidia_b200 import _lib

    lib = _lib.load()
    o = C.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
    o.oracle_gemm_elem_bits.restype = o.oracle_gemm_uniform_bits.restype = C.c_uint16
    o.oracle_gemm_elem_bits.argtypes = o.oracle_gemm_uniform_bits.argtypes = [C.c_uint64, C.c_uint32, C.c_int]
    for e in list(range(2000)) + [(1 << 34) + 7 * i for i in range(2000)]:
        for mat in (0, 1):
            assert lib.b200probe_gemm_operand_bits(e, SEED, mat) == o.oracle_gemm_elem_bits(e, SEED, mat)
            assert lib.b200probe_gemm_operand_bits(e, SEED, 2 | mat) == o.oracle_gemm_uniform_bits(e, SEED, mat)


def test_exact_class_sums_stay_exact_in_fp32():
    """The EXACT class's premise: |products| <= 64, so partial sums up to K = 2^18 stay below 2^24."""
    o = _oracle_lib()
    vals = {o.oracle_e4m3_value(o.oracle_fp8_operand(e, SEED, m)) for e in range(4096) for m in (0, 1)}
    assert vals == set(float(v) for v in range(-8, 8))
    assert 64 * 2**18 <= 2**24


def test_fp8_entry_and_launch_return_enocuda_without_a_gpu(monkeypatch):
    _no_gpu()
    from k3s_nvidia_b200 import _lib
    from k3s_nvidia_b200.probe import Probe, ProbeError

    _lib.load().b200probe_shutdown()
    monkeypatch.setenv("MOCK_NVML_DEVICES", "1")
    p = Probe(_oracle.MOCK_NVML)
    try:
        for cls in (_lib.GEMM_EXACT, _lib.GEMM_UNIFORM):
            with pytest.raises(ProbeError) as e:
                p.gemm_fp8(0, m=256, n=256, k=128, operands=cls)
            assert e.value.rc == -4
        with pytest.raises(ProbeError) as e:
            p.gemm_fp8_launch(0, 1 << 20, 2 << 20, 3 << 20, 256, 256, 128)
        assert e.value.rc == -4
        assert p.lib.b200probe_gemm_fill(0, 1 << 20, 4096, SEED, _lib.GEMM_FILL_E4M3, None) == -4
    finally:
        p.close()


# ---- label rules: Python and native on the same synthetic results -------------------------------------------------------
def test_fp8_verdict_rules(monkeypatch):
    monkeypatch.delenv("B200PROBE_GEMM_FP8_MIN_TFLOPS", raising=False)
    th = L.Thresholds()
    assert th.gemm_fp8_min_tflops == pytest.approx(0.70 * L.GEMM_FP8_MEASURED_TFLOPS)
    fast, slow = L.GEMM_FP8_MEASURED_TFLOPS, 0.69 * L.GEMM_FP8_MEASURED_TFLOPS
    got = L.gemm_fp8_labels({0: NS(tflops_median=fast, verified=1), 3: NS(tflops_median=slow, verified=1)}, th)
    assert got == {P + "gpu0.gemm-fp8-tflops": str(int(round(fast))), P + "gpu0.gemm-fp8-data-ok": "true", P + "gpu0.gemm-fp8-healthy": "true",
                   P + "gpu3.gemm-fp8-tflops": str(int(round(slow))), P + "gpu3.gemm-fp8-data-ok": "true", P + "gpu3.gemm-fp8-healthy": "false",
                   P + "gemm-fp8-healthy": "false"}
    bad = L.gemm_fp8_labels({1: NS(tflops_median=fast, verified=0)}, th)
    assert bad[P + "gpu1.gemm-fp8-data-ok"] == "false" and bad[P + "gemm-fp8-healthy"] == "false"
    assert L.gate_label({P + "gemm-healthy": "true", P + "gemm-fp8-healthy": "false"}) == {P + "healthy": "false"}
    assert L.gate_label({P + "gemm-fp8-healthy": "true"}) == {P + "healthy": "true"}
    monkeypatch.setenv("B200PROBE_GEMM_FP8_MIN_TFLOPS", "100")
    assert L.Thresholds().gemm_fp8_min_tflops == 100.0
    for v, on in (("1", True), ("0", False), ("", False)):
        monkeypatch.setenv("B200PROBE_GEMM_FP8", v)
        assert L.gemm_fp8_enabled() is on
    monkeypatch.delenv("B200PROBE_GEMM_FP8")
    assert not L.gemm_fp8_enabled()


def test_label_rules_match_between_the_hosts(monkeypatch):
    monkeypatch.delenv("B200PROBE_GEMM_FP8_MIN_TFLOPS", raising=False)
    monkeypatch.delenv("B200PROBE_GEMM_MIN_TFLOPS", raising=False)
    rng = random.Random(2031)
    pool = L.GEMM_FP8_MEASURED_TFLOPS
    for trial in range(60):
        lines, per = [], {}
        for gpu in range(rng.randint(1, 8)):
            r = NS(tflops_median=rng.choice([rng.uniform(0.5 * pool, 1.2 * pool), 0.7 * pool, 0.0]), verified=rng.choice([1, 1, 1, 0, -1]))
            lines.append(f"gemm_fp8 {gpu} {r.tflops_median!r} {r.verified}")
            per[gpu] = r
        want = L.gemm_fp8_labels(per, L.Thresholds())
        if rng.random() < 0.5:
            lines.append(f"gemm 0 {rng.uniform(900, 1700)!r} 1")
            want.update(L.gemm_labels({0: NS(tflops_median=float(lines[-1].split()[2]), verified=1)}, L.Thresholds()))
        want.update(L.gate_label(want))
        out = subprocess.run([BIN, "--labels-from-stdin"], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout
        assert out == L.render(want), (trial, lines)


# ---- runner policy, round by round, in both hosts ------------------------------------------------------------------------
def _fp8_fake_probe(n):
    """FakeProbe of test_labels.py plus a scripted gemm_fp8 (the Python twin of tests/gemm_fp8/fake_gemm_fp8.c)."""
    from test_labels import FakeProbe

    class _P(FakeProbe):
        script = {}

        def gemm_fp8(self, idx, **kw):
            from k3s_nvidia_b200.probe import GemmReport, ProbeError

            self.calls.append(("gemm_fp8", idx, kw.get("warmup"), kw.get("reps")))
            v = self.script.get(idx, 3000.0)
            if v == "mismatch":
                raise ProbeError(-6, "gemm_fp8", "3 of 1024 sampled outputs differ")
            if v == "enomem":
                raise ProbeError(L.ENOMEM, "gemm_fp8", "out of device memory")
            if v == "cuda":
                raise ProbeError(1700, "gemm_fp8", "an illegal memory access was encountered")
            return GemmReport(8192, 8192, 8192, 0.4, 0.4, float(v), float(v) * 1.01, 0.0, 0.0, 0.0, 1024, 0, 1, 2, 1)

    return _P(n=n)


def _script_env(rounds):
    env = {}
    for r, sc in enumerate(rounds):
        if sc.get("busy"):
            env[f"FAKE_R{r}_BUSY"] = ",".join(str(i) for i in sorted(sc["busy"]))
        if sc.get("fp8"):
            env[f"FAKE_R{r}_FP8"] = ",".join(f"{i}:{v}" for i, v in sc["fp8"].items())
    return env


def _native_rounds(tmp_path, rounds, preload, extra_env):
    env = {k: v for k, v in os.environ.items() if not k.startswith("B200PROBE_GEMM_FP8")}
    env.update(MOCK_NVML_DEVICES="4", LD_PRELOAD=preload, **_script_env(rounds), **extra_env)
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
        type(fp).script = dict(sc.get("fp8", {}))
        got.append(runner.run_once())
    return got


SLOW = round(0.5 * 3000.0)
ROUNDS = [
    dict(),                                                        # all healthy at the interposer's 3000 TFLOP/s: calibrates every GPU
    dict(fp8={1: SLOW}),                                           # gpu1 slow: below 0.70 x its calibrated figure
    dict(busy={1}, fp8={0: "mismatch"}),                           # gpu1 busy carries its slow verdict; gpu0 a data mismatch
    dict(fp8={2: "enomem", 3: "cuda"}),                            # ENOMEM is inconclusive; a CUDA error fails
    dict(busy={0, 1, 2, 3}),                                       # nothing measurable: every verdict stands
]


def test_scripted_rounds_with_fp8_on_give_the_same_labels_in_both_hosts(tmp_path, monkeypatch):
    _no_gpu()
    monkeypatch.delenv("B200PROBE_GEMM_FP8_MIN_TFLOPS", raising=False)
    monkeypatch.setenv("B200PROBE_GEMM_FP8", "1")
    native, err = _native_rounds(tmp_path / "native", ROUNDS, FAKE_FP8, {"B200PROBE_GEMM_FP8": "1"})
    assert "Sanitizer" not in err and "runtime error" not in err, err[-3000:]
    fp = _fp8_fake_probe(4)
    py = _python_rounds(tmp_path / "py", ROUNDS, fp)
    for r in range(len(ROUNDS)):
        assert native[r] == py[r], (r, sorted(set(native[r].items()) ^ set(py[r].items())))
    assert {c[2:] for c in fp.calls if c[0] == "gemm_fp8"} == {(2, 5)}
    n = native
    assert n[0][P + "gpu0.gemm-fp8-tflops"] == "3000" and n[0][P + "gpu3.gemm-fp8-data-ok"] == "true"
    assert n[0][P + "gemm-fp8-healthy"] == "true" and n[0][P + "healthy"] == "true"
    assert n[1][P + "gpu1.gemm-fp8-tflops"] == str(SLOW) and n[1][P + "gpu1.gemm-fp8-healthy"] == "false"
    assert n[1][P + "gemm-fp8-healthy"] == "false" and n[1][P + "healthy"] == "false" and n[1][P + "gemm-healthy"] == "true"
    assert n[2][P + "gpu1.probe-state"] == "busy" and n[2][P + "gpu1.gemm-fp8-tflops"] == str(SLOW)        # carried by the "gemm-" prefix
    assert n[2][P + "gpu1.gemm-fp8-healthy"] == "false"
    assert n[2][P + "gpu0.gemm-fp8-healthy"] == "false" and P + "gpu0.gemm-fp8-tflops" not in n[2]
    assert n[3][P + "gpu2.probe-state"] == "no-memory" and n[3][P + "gpu2.gemm-fp8-healthy"] == "true"    # last verdict stands
    assert n[3][P + "gpu3.gemm-fp8-healthy"] == "false" and n[3][P + "gpu0.gemm-fp8-healthy"] == "true"
    assert n[4] == {**n[3], **{P + f"gpu{i}.probe-state": "busy" for i in range(4)}}


def test_switch_unset_or_zero_gives_exactly_todays_labels(tmp_path, monkeypatch):
    """B200PROBE_GEMM_FP8 unset or 0: the label set of the interposer without an FP8 probe, in both hosts."""
    _no_gpu()
    monkeypatch.delenv("B200PROBE_GEMM_FP8", raising=False)
    plain = os.path.join(ROOT, "tests", "fake_probe", "libfakeprobe.so")
    before, _ = _native_rounds(tmp_path / "a", ROUNDS, plain, {})
    unset, _ = _native_rounds(tmp_path / "b", ROUNDS, FAKE_FP8, {})
    zero, _ = _native_rounds(tmp_path / "c", ROUNDS, FAKE_FP8, {"B200PROBE_GEMM_FP8": "0"})
    assert before == unset == zero
    assert not [k for r in before for k in r if "fp8" in k]
    from test_labels import FakeProbe

    assert _python_rounds(tmp_path / "py", ROUNDS, FakeProbe(n=4)) == before        # no gemm_fp8 at all: it must not be called
    monkeypatch.setenv("B200PROBE_GEMM_FP8", "0")
    assert _python_rounds(tmp_path / "py0", ROUNDS, FakeProbe(n=4)) == before


# ---- SASS --------------------------------------------------------------------------------------------------------------
def test_e4m3_kernel_runs_on_the_fp8_tensor_core_path():
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    full = subprocess.run([cuobjdump, "-sass", os.path.join(ROOT, "k3s-nvidia_b200", "libb200probe.so")], capture_output=True, text=True,
                          timeout=300).stdout
    parts = [p for p in full.split("Function : ") if "gemm_e4m3_tn_2cta_512_kernel" in p.split("\n", 1)[0]]
    assert len(parts) == 1
    s = parts[0]
    assert "UTCQMMA.2CTA" in s                                                   # tcgen05.mma.cta_group::2.kind::f8f6f4
    assert "UTMALDG" in s and "UTCBAR.2CTA.MULTICAST" in s and "LDTM.x32" in s
    assert "UTCHMMA" not in s and "HMMA." not in s and "HGMMA" not in s
