"""GPU: the HBM integrity probe.  March elements against the CPU oracle (bit-exact), injected flips located exactly, the
full-memory entry on an idle B200 (clean, nothing left allocated), ENOMEM, and the element rate against the copy sweep."""
import ctypes as C
import os

import numpy as np
import pytest

import _oracle

pytestmark = pytest.mark.gpu

SEED = 0xB200
V, W = 1, 2
NONE = 2**64 - 1
ORACLE = os.path.join(_oracle.ROOT, "tests", "memtest", "libmemtest_oracle.so")
# ragged (not 16-byte multiples), below one 8 KiB stage, straddling stages and the worker stride
SIZES = [4, 12, 20, 8192 - 4, 8192 + 4, 3 * 8192 + 36, (1 << 20) + 12, 37 * 8192 * 4 + 16, 64 << 20]
BASES = [0, 12345, (1 << 32) - 1000]          # the last straddles a 2^32-word boundary of the pattern's index


@pytest.fixture(scope="module")
def env():
    import torch

    from k3s_nvidia_b200.probe import Probe

    assert torch.cuda.is_available()
    p = Probe()
    o = C.CDLL(ORACLE)
    u64p = C.POINTER(C.c_uint64)
    o.oracle_memtest_verify.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, u64p, u64p, C.POINTER(C.c_uint32)]
    o.oracle_memtest_fill.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32]
    yield torch, p, o
    p.close()


def _want(o, n, base, seed):
    out = np.empty(n, dtype=np.uint32)
    o.oracle_memtest_fill(out.ctypes.data, n, base, seed & 0xFFFFFFFF)
    return out


def _verify(o, words, base, seed):
    bad, first, bits = C.c_uint64(), C.c_uint64(), C.c_uint32()
    o.oracle_memtest_verify(words.ctypes.data, words.size, base, seed & 0xFFFFFFFF, C.byref(bad), C.byref(first), C.byref(bits))
    return bad.value, first.value, bits.value


@pytest.mark.parametrize("base", BASES)
@pytest.mark.parametrize("nbytes", SIZES)
def test_march_elements_are_bit_exact_against_the_oracle(env, nbytes, base):
    torch, p, o = env
    pad = 64
    buf = torch.full((nbytes + pad,), 0xAA, dtype=torch.uint8, device="cuda:0")
    n = nbytes // 4
    s1 = SEED ^ 0x5A5A5A5A
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, W, 0, SEED) == (0, NONE, 0)
    assert np.array_equal(buf[:nbytes].cpu().numpy().view(np.uint32), _want(o, n, base, SEED))
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V | W, SEED, ~SEED) == (0, NONE, 0)
    got = buf[:nbytes].cpu().numpy().view(np.uint32)
    assert np.array_equal(got, ~_want(o, n, base, SEED)) and _verify(o, got, base, ~SEED)[0] == 0
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V | W, ~SEED, s1) == (0, NONE, 0)
    assert np.array_equal(buf[:nbytes].cpu().numpy().view(np.uint32), _want(o, n, base, s1))
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V, s1, 0) == (0, NONE, 0)
    assert (buf[nbytes:].cpu().numpy() == 0xAA).all(), "wrote past the end"


@pytest.mark.parametrize("nbytes,base", [(64 << 20, 0), (3 * 8192 + 36, 7), ((1 << 20) + 12, (1 << 32) - 1000)])
def test_injected_flips_are_located_exactly(env, nbytes, base):
    """Flips written from the host: one lone bit, a word with several bits (the OR names the data lanes), and one in the
    ragged tail.  The flip made between E1 and E2 is seen against the complemented expectation."""
    torch, p, o = env
    buf = torch.zeros(nbytes, dtype=torch.uint8, device="cuda:0")
    words = buf.view(torch.int32)
    n = nbytes // 4
    p.memtest_element(0, buf.data_ptr(), nbytes, base, W, 0, SEED)
    flips = {n // 3: 1 << 9, n - 1: 1 << 30, 5: 0x0F0}
    for i, m in flips.items():
        words[i] ^= m
    want_bits = 0
    for m in flips.values():
        want_bits |= m
    # E1: the flips are seen; E1 writes ~P(s0) everywhere, the faults included
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V | W, SEED, ~SEED) == (3, base + min(flips), want_bits)
    assert _verify(o, words.cpu().numpy().view(np.uint32), base, ~SEED) == (0, NONE, 0)
    words[n // 2] ^= 1                                                        # between E1 and E2
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V | W, ~SEED, SEED ^ 1) == (1, base + n // 2, 1)
    assert p.memtest_element(0, buf.data_ptr(), nbytes, base, V, SEED ^ 1, 0) == (0, NONE, 0)


def test_memtest_entry_on_an_idle_gpu(env):
    torch, p, o = env
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0, total = torch.cuda.mem_get_info(0)
    r = p.hbm_memtest(0, fraction=0.9)
    free1, _ = torch.cuda.mem_get_info(0)
    assert r.bad_words == 0 and r.first_bad_word == NONE and r.bad_bits == 0 and r.first_bad_element == -1
    assert r.bytes_tested >= 0.9 * r.free_before - (1 << 30)
    assert r.chunks == -(-r.bytes_tested // (1 << 30)) and r.passes == 1 and r.total == total
    assert r.ecc_uncorrected_delta <= 0
    assert abs(free1 - free0) <= 64 << 20, "the memtest must not keep device memory"
    assert r.gbs > 0 and r.test_ms > 0 and r.alloc_ms > 0
    print(f"memtest: {r.bytes_tested / 2**30:.1f} GiB of {r.free_before / 2**30:.1f} GiB free, alloc {r.alloc_ms:.1f} ms, "
          f"test {r.test_ms:.1f} ms, {r.gbs:.0f} GB/s, ECC corrected delta {r.ecc_corrected_delta}, remap {r.remap_pending}/{r.remap_failure}")


def test_min_bytes_above_total_memory_is_enomem_with_nothing_left(env):
    torch, p, o = env
    from k3s_nvidia_b200.probe import ProbeError

    free0, total = torch.cuda.mem_get_info(0)
    with pytest.raises(ProbeError) as e:
        p.hbm_memtest(0, fraction=1.0, min_bytes=total + (1 << 30))
    assert e.value.rc == -10
    free1, _ = torch.cuda.mem_get_info(0)
    assert abs(free1 - free0) <= 64 << 20


def _kernel_ms(prof, name):
    """Mean device time of the kernels whose name contains `name` in a torch.profiler trace, in ms."""
    for ev in prof.key_averages():
        if name in ev.key and ev.count:
            total = getattr(ev, "device_time_total", None)
            if total is None:
                total = ev.cuda_time_total
            return total / ev.count / 1e3
    raise AssertionError(f"no {name} in the trace")


def test_element_rate_against_the_copy_sweep(env):
    """Verify+write moves 2N bytes, like a copy of N.  Kernel time of the element from torch.profiler over 1 GiB, against
    the library's copy sweep at 1 GiB in the same process.  Floor: 0.85 of the copy rate."""
    from torch.profiler import ProfilerActivity, profile

    torch, p, o = env
    from k3s_nvidia_b200 import _lib as L

    cp = p.hbm_sweep(0, min_bytes=1 << 30, max_bytes=1 << 30, modes=L.HBM_COPY, warmup=2, reps=10, verify=0)[0].gbs_median
    p.lib.b200probe_hbm_release(0)
    nbytes = 1 << 30
    b = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
    p.memtest_element(0, b.data_ptr(), nbytes, 0, W, 0, SEED)
    seed = SEED
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(10):
            assert p.memtest_element(0, b.data_ptr(), nbytes, 0, V | W, seed, ~seed)[0] == 0
            seed = ~seed & 0xFFFFFFFF
    elem = 2 * nbytes / (_kernel_ms(prof, "hbm_memtest_kernel") * 1e-3) / 1e9
    print(f"memtest element {elem:.0f} GB/s (kernel time), hbm copy sweep {cp:.0f} GB/s ({elem / cp:.2f})")
    assert elem >= 0.85 * cp
