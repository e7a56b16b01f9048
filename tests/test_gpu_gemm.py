"""GPU parity for the tcgen05 GEMM probe: bit-exact against the fp64 oracle contraction rounded
once to bf16 (operands k/128 make every fp32 partial sum exact; tolerance = 0 ulp, stated here)."""
import numpy as np
import pytest

import _oracle

pytestmark = pytest.mark.gpu
SEED = 0xB200


@pytest.fixture(scope="module")
def env():
    import torch

    from k3s_nvidia_b200.probe import Probe

    assert torch.cuda.is_available()
    p = Probe()
    yield torch, p, _oracle.load()
    p.close()                        # b200probe_init is a no-op while a handle is open: later tests load their own NVML


def oracle_operands(o, rows, k, which, seed=SEED):
    """integer numerators (value = n/128), from the oracle's element function"""
    out = np.empty((rows, k), dtype=np.int64)
    for r in range(rows):
        for c in range(k):
            out[r, c] = int(round(o.oracle_gemm_elem(r * k + c, seed, which) * 128))
    return out


def bf16_bits(f32):
    u = f32.astype(np.float32).view(np.uint32).astype(np.uint64)
    r = 0x7FFF + ((u >> 16) & 1)
    return ((u + r) >> 16).astype(np.uint16)


# every kernel the launcher can pick: 512 x 256 per CTA pair with 32-byte stores from registers (default) or staged tensor stores,
# 256 x 256 per CTA pair (double-buffered accumulators, tensor-store epilogue), single CTA
KERNELS = {"pair512-stg": {}, "pair512-tma": {"B200PROBE_GEMM_EPI": "1"}, "pair256": {"B200PROBE_GEMM_VARIANT": "2"}, "single": {"B200PROBE_GEMM_VARIANT": "1"}}


@pytest.mark.parametrize("kernel", sorted(KERNELS))
@pytest.mark.parametrize("m,n,k", [(128, 256, 64), (256, 512, 128), (384, 256, 320), (128, 768, 1024), (512, 256, 192), (768, 512, 256), (1280, 256, 64)])
def test_whole_matrix_bit_exact_vs_oracle(env, m, n, k, kernel, monkeypatch):
    torch, p, o = env
    for kk, vv in KERNELS[kernel].items():
        monkeypatch.setenv(kk, vv)          # read per launch by the library
    st = torch.cuda.current_stream().cuda_stream
    a = torch.empty(m * k, dtype=torch.int16, device="cuda:0")
    b = torch.empty(n * k, dtype=torch.int16, device="cuda:0")
    c = torch.full((m * n,), -1, dtype=torch.int16, device="cuda:0")
    p._check(p.lib.b200probe_gemm_fill(0, a.data_ptr(), m * k, SEED, 0, st), "fill A")
    p._check(p.lib.b200probe_gemm_fill(0, b.data_ptr(), n * k, SEED, 1, st), "fill B")
    p._check(p.lib.b200probe_gemm_launch(0, a.data_ptr(), b.data_ptr(), c.data_ptr(), m, n, k, st), "gemm")
    torch.cuda.synchronize()
    # operands: device generator == oracle generator, bit for bit
    A = oracle_operands(o, m, k, 0)
    B = oracle_operands(o, n, k, 1)
    got_a = a.cpu().numpy().view(np.uint16).reshape(m, k)
    assert np.array_equal(got_a, bf16_bits((A / 128.0).astype(np.float32)))
    assert got_a[0, 0] == o.oracle_gemm_elem_bits(0, SEED, 0)
    # contraction: exact integer arithmetic, one rounding
    want = bf16_bits(((A @ B.T).astype(np.float64) / 16384.0).astype(np.float32))
    got = c.cpu().numpy().view(np.uint16).reshape(m, n)
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} mismatches, first at {bad[:5].tolist()}"


@pytest.mark.parametrize("m,n,k", [(128, 256, 64), (256, 512, 128), (384, 256, 320), (256, 768, 1024)])
def test_uniform_class_whole_matrix_within_tolerance(env, m, n, k):
    """SURVEY.md §8d's operand class (bf16 U(-1,1) from Philox, seed 0xB200): operands bit-identical to the oracle's
    generator; every output within 2^-8 |ref| + 2^-10 sqrt(K) of the fp64 contraction of those operands (tolerance
    stated here and in oracle_gemm_uniform_tol: half a bf16 ulp for the final rounding + the fp32 accumulation allowance)."""
    torch, p, o = env
    st = torch.cuda.current_stream().cuda_stream
    a = torch.empty(m * k, dtype=torch.int16, device="cuda:0")
    b = torch.empty(n * k, dtype=torch.int16, device="cuda:0")
    c = torch.full((m * n,), -1, dtype=torch.int16, device="cuda:0")
    p._check(p.lib.b200probe_gemm_fill(0, a.data_ptr(), m * k, SEED, 2, st), "fill A uniform")
    p._check(p.lib.b200probe_gemm_fill(0, b.data_ptr(), n * k, SEED, 3, st), "fill B uniform")
    p._check(p.lib.b200probe_gemm_launch(0, a.data_ptr(), b.data_ptr(), c.data_ptr(), m, n, k, st), "gemm")
    torch.cuda.synchronize()

    def bits(rows, which):
        return np.array([o.oracle_gemm_uniform_bits(e, SEED, which) for e in range(rows * k)], dtype=np.uint16).reshape(rows, k)

    def f64(bits16):
        return (bits16.astype(np.uint32) << 16).view(np.float32).astype(np.float64)

    A, B = bits(m, 0), bits(n, 1)
    assert np.array_equal(a.cpu().numpy().view(np.uint16).reshape(m, k), A)
    assert np.array_equal(b.cpu().numpy().view(np.uint16).reshape(n, k), B)
    ref = f64(A) @ f64(B).T
    got = f64(c.cpu().numpy().view(np.uint16).reshape(m, n))
    tol = np.abs(ref) / 256.0 + np.sqrt(k) / 1024.0
    assert tol[0, 0] == o.oracle_gemm_uniform_tol(k, ref[0, 0])
    over = np.abs(got - ref) / tol
    assert over.max() <= 1.0, f"max err/tol {over.max():.3f} at {np.unravel_index(over.argmax(), over.shape)}"
    assert abs(ref[3, 5] - o.oracle_gemm_uniform_dot(k, SEED, 3, 5)) < 1e-9


def test_headline_size_sampled_and_stable(env):
    """BASELINE GEMM probe at M=N=K=8192, both operand classes: 1024 sampled outputs against fp64 (EXACT: bit for bit;
    UNIFORM: within the stated tolerance), checksum of C identical run to run (the kernel is deterministic), TFLOP/s
    stable within 1% (north_star's run-to-run bound) and not below 0.9 x the published figure."""
    torch, p, o = env
    from k3s_nvidia_b200 import _lib as L

    for cls, floor in ((L.GEMM_EXACT, 0.9 * 1667.0), (L.GEMM_UNIFORM, 0.9 * 1450.0)):
        p.gemm(0, warmup=3, reps=10, operands=cls)            # settle clocks and fill the resident operands
        r1 = p.gemm(0, warmup=3, reps=10, operands=cls)
        r2 = p.gemm(0, warmup=3, reps=10, operands=cls)
        assert r1.verified == 1 and r1.bad == 0 and r1.samples == 1024 and r1.operands == cls
        assert r1.max_abs_err < 0.5 and (cls == L.GEMM_EXACT or r1.max_err_over_tol <= 1.0)
        assert (r1.c_sum64, r1.c_xor32) == (r2.c_sum64, r2.c_xor32)
        assert abs(r1.tflops_median - r2.tflops_median) / r1.tflops_median < 0.01
        assert r1.tflops_median > floor
    p.lib.b200probe_gemm_release(0)


def test_bad_shapes_fail_loudly(env):
    torch, p, o = env
    from k3s_nvidia_b200.probe import ProbeError

    with pytest.raises(ProbeError):
        p.gemm(0, m=100, n=256, k=64)
    with pytest.raises(ProbeError):
        p.gemm(0, m=128, n=256, k=72)
    with pytest.raises(ProbeError):
        p.gemm(0, m=256, n=256, k=64, operands=7)
