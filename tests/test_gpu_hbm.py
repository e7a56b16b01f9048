"""GPU parity: the sm_100a HBM kernels (through the C ABI) against the CPU oracle.  Bit-exact."""
import numpy as np
import pytest

import _oracle

pytestmark = pytest.mark.gpu

SEED = 0xB200
TUNINGS = [
    dict(variant=0),                                                   # TMA ring, defaults
    dict(variant=0, stage_bytes=4096, stages=2, warps_per_cta=1),      # smallest ring
    dict(variant=0, stage_bytes=16384, stages=3, warps_per_cta=4),
    dict(variant=0, stage_bytes=8192, stages=8, warps_per_cta=2, ctas_per_sm=1),
    dict(variant=1),                                                   # direct LDG/STG
]
# ragged, tiny, empty, below/above one ring chunk, non-16-multiples (word tail)
SIZES = [0, 4, 12, 16, 20, 4096, 4100, 8192 + 8, 65536 - 4, 1 << 20, (1 << 20) + 4, 3 * (1 << 20) + 36, 37 * 8192 * 4 + 16]


@pytest.fixture(scope="module")
def env():
    import torch

    from k3s_nvidia_b200.probe import Probe

    assert torch.cuda.is_available()
    p = Probe()
    yield torch, p, _oracle.load()
    p.close()                        # b200probe_init is a no-op while a handle is open: later tests load their own NVML


def _dev_checksum(torch, p, t, nbytes, **tuning):
    part = torch.zeros(2, dtype=torch.int64, device="cuda:0")
    p.hbm_read(0, t.data_ptr(), nbytes, part.data_ptr(), torch.cuda.current_stream().cuda_stream, **tuning)
    torch.cuda.synchronize()
    return part[0].item() & 0xFFFFFFFFFFFFFFFF, part[1].item() & 0xFFFFFFFF


@pytest.mark.parametrize("tuning", TUNINGS, ids=lambda t: "-".join(f"{k}{v}" for k, v in t.items()))
@pytest.mark.parametrize("nbytes", SIZES)
def test_fill_copy_read_match_oracle(env, tuning, nbytes):
    torch, p, o = env
    st = torch.cuda.current_stream().cuda_stream
    pad = 64
    src = torch.full((nbytes + pad,), 0xAA, dtype=torch.uint8, device="cuda:0")
    dst = torch.full((nbytes + pad,), 0x55, dtype=torch.uint8, device="cuda:0")
    p.hbm_fill(0, src.data_ptr(), nbytes, SEED, st, **tuning)
    p.hbm_copy(0, src.data_ptr(), dst.data_ptr(), nbytes, st, **tuning)
    torch.cuda.synchronize()
    want = _oracle.pattern(o, 0, nbytes // 4, SEED)
    got_src = src.cpu().numpy()
    got_dst = dst.cpu().numpy()
    assert np.array_equal(got_src[:nbytes].view(np.uint32), want), "fill differs from oracle"
    assert np.array_equal(got_dst[:nbytes].view(np.uint32), want), "copy differs from oracle"
    assert (got_src[nbytes:] == 0xAA).all() and (got_dst[nbytes:] == 0x55).all(), "wrote past the end"
    assert _dev_checksum(torch, p, dst, nbytes, **tuning) == _oracle.pattern_checksum(o, nbytes // 4, SEED)


def test_read_checksum_of_arbitrary_data(env):
    torch, p, o = env
    g = torch.Generator(device="cpu").manual_seed(7)
    host = torch.randint(0, 256, (5 * (1 << 20) + 52,), dtype=torch.uint8, generator=g)
    dev = host.cuda()
    for tuning in TUNINGS:
        assert _dev_checksum(torch, p, dev, host.numel(), **tuning) == _oracle.checksum(o, host.numpy())


@pytest.mark.parametrize("direct", [False, True], ids=["tma-ring", "ldg"])
def test_verdict_pass_finds_injected_faults(env, direct, monkeypatch):
    """The probe's own verdict: flipped bits anywhere in the swept range are counted and located exactly
    as the oracle does (single bit, bursts, first/last word, ragged tail, fault in the non-16-byte tail)."""
    import subprocess, sys, json, os

    torch, p, o = env
    if direct:
        # the kernel choice is latched per process: run the same cases in a child with the LDG kernel selected
        code = ("import sys, json; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_gpu_hbm as t; print(json.dumps(t._fault_cases()))"
                % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__))))
        out = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, B200PROBE_VERIFY_DIRECT="1"), capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.strip().splitlines()[-1]) == "ok"
    else:
        assert _fault_cases() == "ok"


def _fault_cases():
    import torch

    from k3s_nvidia_b200.probe import Probe

    p, o = Probe(), _oracle.load()
    st = torch.cuda.current_stream().cuda_stream
    for nbytes in ((8 << 20), (5 << 20) + 8192 + 12, 52, 16):
        words = nbytes // 4
        buf = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
        p.hbm_fill(0, buf.data_ptr(), nbytes, SEED, st)
        torch.cuda.synchronize()
        clean = _oracle.pattern_checksum(o, words, SEED)
        assert p.hbm_verify(0, buf.data_ptr(), nbytes, SEED) == (clean[0], clean[1], 0, 2**64 - 1)
        assert p.hbm_verify(0, buf.data_ptr(), nbytes, SEED ^ 1)[2] == words          # wrong seed: every word differs
        w32 = buf.view(torch.int32)
        rng = np.random.default_rng(nbytes)
        cases = [[0], [words - 1], sorted(rng.choice(words, size=min(words, 7), replace=False).tolist()),
                 list(range(max(0, words // 2 - 3), min(words, words // 2 + 40)))]
        for idxs in cases:
            keep = w32[idxs].clone()
            w32[idxs] = w32[idxs] ^ torch.tensor([1 << (i % 31) for i in idxs], dtype=torch.int32, device="cuda:0")
            host = buf.cpu().numpy()
            want_bad, want_first = _oracle.verify(o, host.view(np.uint32), SEED)
            s, x, bad, first = p.hbm_verify(0, buf.data_ptr(), nbytes, SEED)
            assert (bad, first) == (want_bad, want_first) == (len(idxs), idxs[0]), (nbytes, idxs[:4], bad, first)
            assert (s, x) == _oracle.checksum(o, host.view(np.uint32))
            w32[idxs] = keep
        assert p.hbm_verify(0, buf.data_ptr(), nbytes, SEED)[2] == 0
    return "ok"


def test_verdict_pass_on_a_blank_buffer_and_bad_arguments(env):
    """A buffer that never received the pattern: every word that the pattern says is non-zero counts."""
    torch, p, o = env
    from k3s_nvidia_b200.probe import ProbeError

    nbytes = 1 << 20
    buf = torch.zeros(nbytes, dtype=torch.uint8, device="cuda:0")
    want = _oracle.pattern(o, 0, nbytes // 4, SEED)
    s, x, bad, first = p.hbm_verify(0, buf.data_ptr(), nbytes, SEED)
    assert (s, x) == (0, 0) and bad == int(np.count_nonzero(want)) and first == int(np.flatnonzero(want)[0])
    with pytest.raises(ProbeError):
        p.hbm_verify(0, buf.data_ptr() + 4, 1 << 10, SEED)          # misaligned pointer
    with pytest.raises(ProbeError):
        p.hbm_verify(0, buf.data_ptr(), 1022, SEED)                 # not a multiple of 4


def test_copy_host_roundtrip(env):
    torch, p, o = env
    rng = np.random.default_rng(3)
    src = rng.integers(0, 2**32, size=(1 << 22) + 3, dtype=np.uint32)
    dst = np.zeros_like(src)
    s, x = p.hbm_copy_host(0, src, dst)
    assert np.array_equal(src, dst)
    assert (s, x) == _oracle.checksum(o, src)


def test_copy_host_roundtrip_pinned_pipelined(env):
    """Pinned buffers through the three-stream chunk pipeline (ragged last chunk, several chunk sizes)."""
    import os

    torch, p, o = env
    nbytes = (40 << 20) + 20
    src = p.host_alloc(nbytes)
    dst = p.host_alloc(nbytes)
    try:
        rng = np.random.default_rng(5)
        src[:] = rng.integers(0, 256, size=nbytes, dtype=np.uint8)
        for chunk in (None, 1 << 20, (3 << 20) + 16):
            if chunk:
                os.environ["B200PROBE_HOST_CHUNK_BYTES"] = str(chunk)
            dst[:] = 0
            s, x = p.hbm_copy_host(0, src, dst)
            os.environ.pop("B200PROBE_HOST_CHUNK_BYTES", None)
            assert np.array_equal(src, dst)
            assert (s, x) == _oracle.checksum(o, src.view(np.uint32))
    finally:
        p.host_free(src)
        p.host_free(dst)


def test_full_size_properties(env):
    """BASELINE config 2 at its largest size (1 GiB): closed-form checksum of the pattern,
    copy == source (checksum of checksums), idempotence of a second copy."""
    torch, p, o = env
    nbytes = 1 << 30
    st = torch.cuda.current_stream().cuda_stream
    src = torch.empty(nbytes, dtype=torch.uint8, device="cuda:0")
    dst = torch.zeros(nbytes, dtype=torch.uint8, device="cuda:0")
    p.hbm_fill(0, src.data_ptr(), nbytes, SEED, st)
    want = _oracle.pattern_checksum(o, nbytes // 4, SEED)
    assert _dev_checksum(torch, p, src, nbytes) == want
    assert _dev_checksum(torch, p, src, nbytes, variant=1) == want
    p.hbm_copy(0, src.data_ptr(), dst.data_ptr(), nbytes, st)
    assert _dev_checksum(torch, p, dst, nbytes) == want
    p.hbm_copy(0, dst.data_ptr(), src.data_ptr(), nbytes, st, variant=1)
    assert _dev_checksum(torch, p, src, nbytes) == want
    # spot-check 1 MiB windows byte-for-byte against the oracle
    for off in (0, (1 << 29) - (1 << 19), nbytes - (1 << 20)):
        got = dst[off: off + (1 << 20)].cpu().numpy().view(np.uint32)
        assert np.array_equal(got, _oracle.pattern(o, off // 4, (1 << 20) // 4, SEED))


def test_sweep_default_config_verified(env):
    torch, p, o = env
    pts = p.hbm_sweep(0, min_bytes=1 << 20, max_bytes=1 << 28, warmup=1, reps=3, verify=1)
    assert len(pts) == 9 * 3
    for pt in pts:
        assert pt.verified == 1
        assert (pt.sum64, pt.xor32) == _oracle.pattern_checksum(o, pt.bytes // 4, SEED)
        assert pt.gbs_median > 0


def test_bad_arguments_fail_loudly(env):
    torch, p, o = env
    from k3s_nvidia_b200.probe import ProbeError

    t = torch.zeros(1024, dtype=torch.uint8, device="cuda:0")
    with pytest.raises(ProbeError):
        p.hbm_fill(0, t.data_ptr(), 6, SEED)            # not a multiple of 4
    with pytest.raises(ProbeError):
        p.hbm_fill(0, t.data_ptr() + 4, 16, SEED)       # misaligned
    with pytest.raises(ProbeError):
        p.hbm_fill(0, t.data_ptr(), 16, SEED, variant=0, stages=1)
    with pytest.raises(ProbeError):
        p.hbm_fill(99, t.data_ptr(), 16, SEED)
