"""GPU checks of the FP8 tensor-core probe (tcgen05.mma kind::f8f6f4, E4M3 operands, bf16 C).  EXACT: the whole C bit-exact
against the fp64 contraction rounded once to bf16 (tolerance 0, the operands make every fp32 partial sum exact); UNIFORM: the
whole C within 2^-8 |ref| + 2^-10 sqrt(K).  Device operands equal the independent oracle byte for byte."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import _oracle

pytestmark = pytest.mark.gpu
SEED = 0xB200
ROOT = _oracle.ROOT
PROFILE = os.path.join(ROOT, "profiles", "gemm_fp8_bench_r01.txt")


@pytest.fixture(scope="module")
def env():
    import torch

    from k3s_nvidia_b200.probe import Probe

    assert torch.cuda.is_available()
    subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "gemm_fp8")], check=True, capture_output=True)
    o = C.CDLL(os.path.join(ROOT, "tests", "gemm_fp8", "libfp8_oracle.so"))
    o.oracle_fp8_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int]
    p = Probe()
    yield torch, p, o
    p.close()                        # b200probe_init is a no-op while a handle is open: later tests load their own NVML


def operands(torch, p, o, m, n, k, cls, check_oracle=True):
    """A [m][k], B [n][k] E4M3 filled on the device by the library; with check_oracle, compared with the oracle byte for byte."""
    from k3s_nvidia_b200 import _lib as L

    st = torch.cuda.current_stream().cuda_stream
    out = []
    for mat, rows in ((0, m), (1, n)):
        t = torch.empty(rows * k, dtype=torch.uint8, device="cuda:0")
        p._check(p.lib.b200probe_gemm_fill(0, t.data_ptr(), rows * k, SEED, L.GEMM_FILL_E4M3 | (cls << 1) | mat, st), "gemm_fill")
        if check_oracle:
            want = np.empty(rows * k, dtype=np.uint8)
            o.oracle_fp8_fill(want.ctypes.data, 0, rows * k, SEED, (cls << 1) | mat)
            got = t.cpu().numpy()
            assert np.array_equal(got, want), f"matrix {mat}: {(got != want).sum()} bytes differ from the oracle"
        out.append(t)
    return out


def run(torch, p, a, b, m, n, k):
    c = torch.full((m, n), -1, dtype=torch.int16, device="cuda:0")          # poison: NaN in bf16
    p.gemm_fp8_launch(0, a.data_ptr(), b.data_ptr(), c.data_ptr(), m, n, k, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return c


def reference(torch, a, b, m, n, k):
    """A @ B^T in fp64 on the device: exact for the EXACT class (integers, |C| < 2^53)"""
    a64 = a.view(torch.float8_e4m3fn).to(torch.float64).view(m, k)
    b64 = b.view(torch.float8_e4m3fn).to(torch.float64).view(n, k)
    return a64 @ b64.t()


def bf16_once(torch, ref64):
    """one round-to-nearest-even to bf16 (fp64 -> fp32 is exact for the EXACT class: |C| <= 64 K < 2^24)"""
    return ref64.to(torch.float32).to(torch.bfloat16).view(torch.int16)


@pytest.mark.parametrize("m,n,k", [(256, 256, 128), (512, 256, 256), (768, 512, 384), (1280, 256, 128), (256, 768, 1024), (2048, 2048, 2048)])
def test_exact_class_whole_c_is_bit_exact(env, m, n, k):
    torch, p, o = env
    a, b = operands(torch, p, o, m, n, k, 0)
    c = run(torch, p, a, b, m, n, k)
    want = bf16_once(torch, reference(torch, a, b, m, n, k))
    bad = int((c != want).sum().item())
    assert bad == 0, f"{bad} of {m * n} outputs differ from the fp64 contraction rounded to bf16"


def test_exact_class_at_8192_accumulates_exactly(env):
    """Partial sums reach 2^19 here: an accumulator that kept fewer than 19 significant bits would show up as mismatches."""
    torch, p, o = env
    m = n = k = 8192
    a, b = operands(torch, p, o, m, n, k, 0, check_oracle=False)
    c = run(torch, p, a, b, m, n, k)
    ref = reference(torch, a, b, m, n, k)
    bad = int((c != bf16_once(torch, ref)).sum().item())
    assert bad == 0, f"{bad} of {m * n} outputs differ; max |C| = {ref.abs().max().item():.0f}"


def test_accumulator_keeps_large_partial_sums_exact(env):
    """Known answers whose running sums grow far past the final values: A = 7 everywhere, B rows of +7 (C = 49 K = 401408 at
    K = 8192), +7 then -7 (partial sums up to 200704, C = 0), and [-8, 7] integers sorted descending (the sum climbs, then
    falls).  Any addition into the fp32 accumulator that dropped a bit below 2^19 would leave a wrong C."""
    torch, p, o = env
    m, n, k = 256, 256, 8192
    a = torch.full((m, k), 7.0, device="cuda:0").to(torch.float8_e4m3fn)
    g = torch.Generator(device="cpu").manual_seed(11)
    rows = [torch.full((k,), 7.0), torch.cat([torch.full((k // 2,), 7.0), torch.full((k // 2,), -7.0)])]
    rows += [torch.randint(-8, 8, (k,), generator=g).float().sort(descending=True).values for _ in range(n - 2)]
    b = torch.stack(rows).to("cuda:0").to(torch.float8_e4m3fn)
    a, b = a.view(torch.uint8).reshape(-1), b.view(torch.uint8).reshape(-1)
    c = run(torch, p, a, b, m, n, k)
    ref = reference(torch, a, b, m, n, k)
    peak = (a.view(torch.float8_e4m3fn).view(m, k)[:1].to(torch.float64) * b.view(torch.float8_e4m3fn).view(n, k).to(torch.float64)).cumsum(1).abs().max()
    assert ref[0, 0].item() == 49 * k and ref[0, 1].item() == 0 and peak.item() >= 49 * k
    bad = int((c != bf16_once(torch, ref)).sum().item())
    assert bad == 0, f"{bad} of {m * n} outputs differ; running sums reach {peak.item():.0f}"


def test_uniform_class_whole_c_is_within_tolerance(env, record_property):
    torch, p, o = env
    m = n = k = 2048
    a, b = operands(torch, p, o, m, n, k, 1)
    c = run(torch, p, a, b, m, n, k)
    ref = reference(torch, a, b, m, n, k)
    got = c.view(torch.bfloat16).to(torch.float64)
    tol = ref.abs() * 2.0**-8 + 2.0**-10 * k**0.5
    ratio = ((got - ref).abs() / tol).max().item()
    assert ratio <= 1.0, f"max |err| / tol = {ratio:.3f}"
    one = torch.ones((), dtype=torch.float32, device="cuda:0")
    cub = torch._scaled_mm(a.view(torch.float8_e4m3fn).view(m, k), b.view(torch.float8_e4m3fn).view(n, k).t(), scale_a=one, scale_b=one,
                           out_dtype=torch.bfloat16)
    differ = int((cub.view(torch.int16) != c).sum().item())
    record_property("elements_differing_from_cublaslt_fp8", differ)
    print(f"UNIFORM 2048^3: max err/tol {ratio:.3f}; {differ} of {m * n} outputs differ from cuBLASLt FP8's C")


def test_device_fill_matches_the_oracle_at_an_odd_length(env):
    torch, p, o = env
    from k3s_nvidia_b200 import _lib as L

    for which in range(4):
        t = torch.zeros(4099 + 13, dtype=torch.uint8, device="cuda:0")
        p._check(p.lib.b200probe_gemm_fill(0, t.data_ptr(), 4099, SEED, L.GEMM_FILL_E4M3 | which, torch.cuda.current_stream().cuda_stream), "fill")
        want = np.empty(4099, dtype=np.uint8)
        o.oracle_fp8_fill(want.ctypes.data, 0, 4099, SEED, which)
        got = t.cpu().numpy()
        assert np.array_equal(got[:4099], want) and not got[4099:].any()        # nothing written past elems


@pytest.mark.parametrize("cls", [0, 1], ids=["exact", "uniform"])
def test_library_entry_at_8192_and_release(env, cls):
    torch, p, o = env
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(0)[0]
    r = p.gemm_fp8(0, operands=cls)
    assert (r.m, r.n, r.k, r.samples) == (8192, 8192, 8192, 1024)
    assert r.verified == 1 and r.bad == 0 and r.operands == cls             # EXACT: every sample equals the fp64 contraction rounded to bf16
    if cls == 1:
        assert r.max_err_over_tol <= 1.0
    p._check(p.lib.b200probe_gemm_release(0), "gemm_release")
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free1 >= free0 - (64 << 20), f"{(free0 - free1) >> 20} MiB still held after release"


def test_bad_shapes_and_pointers_are_einval(env):
    torch, p, o = env
    from k3s_nvidia_b200.probe import ProbeError

    buf = torch.empty(1 << 22, dtype=torch.uint8, device="cuda:0")
    base = buf.data_ptr()
    st = torch.cuda.current_stream().cuda_stream
    for args in ((base, base + (1 << 20), base + (2 << 20), 256, 256, 64),          # k not a multiple of 128
                 (base, base + (1 << 20), base + (2 << 20), 128, 256, 128),         # m not a multiple of 256
                 (base + 1, base + (1 << 20), base + (2 << 20), 256, 256, 128),     # misaligned A
                 (base, base + (1 << 20) + 8, base + (2 << 20), 256, 256, 128),     # misaligned B
                 (base, base + (1 << 20), base + (2 << 20) + 2, 256, 256, 128)):    # misaligned C
        assert p.lib.b200probe_gemm_fp8_launch(0, *args, st) == -1, args
    for shape in (dict(m=256, n=256, k=64), dict(m=128, n=256, k=128), dict(m=256, n=128, k=128)):
        with pytest.raises(ProbeError) as e:
            p.gemm_fp8(0, **shape)
        assert e.value.rc == -1


def test_rate_against_the_recorded_figure(env):
    torch, p, o = env
    with open(PROFILE) as f:
        rec = json.loads([ln for ln in f if ln.startswith("{")][0])
    want = rec["exact"]["probe_entry"]["tflops_median"]
    r = p.gemm_fp8(0, operands=0)
    p.lib.b200probe_gemm_release(0)
    assert r.verified == 1
    assert r.tflops_median <= 4500.0, "above the data sheet's dense FP8 rate: a timing error"
    assert r.tflops_median >= 0.9 * want, f"{r.tflops_median:.0f} TFLOP/s against {want:.0f} recorded in {os.path.basename(PROFILE)}"


def test_native_round_publishes_the_python_fp8_keys(tmp_path, monkeypatch, env):
    torch, p, o = env
    from k3s_nvidia_b200 import labels as L
    from test_native_plugin import BIN

    monkeypatch.setenv("B200PROBE_IGNORE_TENANTS", "1")          # this pytest process holds a context: to the daemon it is a tenant
    monkeypatch.setenv("B200PROBE_GEMM_FP8", "1")
    out = subprocess.run([BIN, "--probe-once", "--features-dir", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-3000:]
    native = L.parse_feature_file(out.stdout)
    py = L.ActiveProbeRunner(p, features_dir=str(tmp_path / "py")).run_once()
    fp8 = sorted(k for k in py if "gemm-fp8" in k)
    assert fp8 and fp8 == sorted(k for k in native if "gemm-fp8" in k)
    assert L.PREFIX + "gpu0.gemm-fp8-tflops" in fp8 and L.PREFIX + "gemm-fp8-healthy" in fp8
    for lab in (native, py):
        assert lab[L.PREFIX + "gpu0.gemm-fp8-data-ok"] == "true" and lab[L.PREFIX + "gpu0.gemm-fp8-healthy"] == "true", lab
        assert lab[L.PREFIX + "gemm-fp8-healthy"] == "true" and lab[L.PREFIX + "healthy"] == "true"
    for k in fp8:
        if k.endswith("-tflops"):
            assert abs(int(native[k]) - int(py[k])) <= 0.05 * int(py[k]) + 1, (k, native[k], py[k])
